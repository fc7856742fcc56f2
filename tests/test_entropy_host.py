"""CPU tests of the per-token policy entropy and the entropy bonus: the oracle's definition against the reference's own
helper (tests/golden/cfg1_entropy.npz, from BaseLearner.compute_entropy_bonus, distributed_actor.py:266-281), the CLI
flags and their way into the learner config, the trainer's entropy metric, and the argument checks of the new C entry
points (no GPU needed)."""
import ctypes
import os

import numpy as np
import pytest
import torch

from oracle import entropy_oracle as eo
from oracle import learner_oracle as lo

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def _cfg1():
    return lo.OracleConfig(vocab=512, hidden=128, inter=256, n_layers=2, n_q_heads=4, n_kv_heads=2, head_dim=32,
                           lora_r=16, lora_alpha=16)


def test_oracle_entropy_matches_reference_helper():
    z = np.load(os.path.join(GOLDEN, "cfg1_entropy.npz"))
    cfg = _cfg1()
    params, nf4 = lo.make_params(cfg, seed=int(z["param_seed"]))
    assert lo.params_digest(params, nf4) == str(z["param_sha256"])
    P, T, B = int(z["P"]), int(z["T"]), int(z["train_batch_size"])
    prompts, answers, _ = lo.make_batch(cfg, 4, P, T, seed=1, ragged=True)
    ids, am, ansm = lo.pad_batch(prompts, answers, P, T)
    assert np.array_equal(ansm.numpy(), z["answer_mask"])
    with torch.no_grad():
        H = eo.compute_current_policy_entropy(params, cfg, ids, am, P)
    ref = torch.from_numpy(z["entropy"])
    d = (H - ref).abs().max().item()
    print(f"oracle vs reference helper: max |dH| = {d:.3e} nats (H in [{ref.min():.3f}, {ref.max():.3f}])")
    assert d <= 1e-5
    assert 0 < ref.min() and ref.max() <= np.log(cfg.vocab) + 1e-5
    # the helper's own aggregate (alpha * unmasked mean over micro-batch 0): what the commented call at :377-378 computes
    alpha = float(z["bonus_mb0_alpha"])
    assert abs(alpha * H[:B].double().mean().item() - float(z["bonus_mb0"])) <= 1e-7


def test_oracle_loss_entropy_term():
    """compute_gradients(entropy_alpha=a) loss = compute_loss() - a * sum over micro-batches of mean_i(sum_t mask H / len_i),
    and its gradient = the plain gradient + the gradient of that term."""
    cfg = _cfg1()
    params, _ = lo.make_params(cfg, seed=1234)
    P, T, B = 16, 32, 2
    prompts, answers, _ = lo.make_batch(cfg, 4, P, T, seed=1, ragged=True)
    ids, am, ansm = lo.pad_batch(prompts, answers, P, T)
    r = [0.5, -0.25, 1.0, 0.3]
    g0, base = lo.compute_gradients(params, cfg, ids, am, ansm, r, P, B, "pg")
    alpha = 0.05
    g1, with_h = eo.compute_gradients(params, cfg, ids, am, ansm, r, P, B, "pg", entropy_alpha=alpha)
    g2, same = eo.compute_gradients(params, cfg, ids, am, ansm, r, P, B, "pg")
    assert same == base and all(torch.equal(g2[k], g0[k]) for k in g0)
    assert any(not torch.allclose(g1[k], g0[k]) for k in g0)
    with torch.no_grad():
        H = eo.compute_current_policy_entropy(params, cfg, ids, am, P).double()
    m = ansm.double()
    per = (H * m).sum(-1) / m.sum(-1)
    want = base - alpha * sum(per[i:i + B].mean().item() for i in range(0, 4, B))
    assert abs(with_h - want) <= 1e-6 * max(1.0, abs(want))


def test_cli_entropy_flags_default_and_forwarding():
    from distrl_llm_b200.train_distributed import build_parser, config_from_args
    ap = build_parser()
    cfg = config_from_args(ap.parse_args([]))
    assert cfg["entropy_alpha"] == 0.0 and cfg["log_entropy"] is False
    cfg = config_from_args(ap.parse_args(["--entropy_alpha", "0.01", "--log_entropy"]))
    assert cfg["entropy_alpha"] == 0.01 and cfg["log_entropy"] is True


class _HostPolicy:
    """Just what BaseLearner.__init__ reads from a Policy (no device work happens in the constructor)."""

    def __init__(self):
        from distrl_llm_b200.policy import LMConfig
        self.cfg = LMConfig(vocab=512, hidden=128, inter=256, n_layers=2, n_q_heads=4, n_kv_heads=2, head_dim=32)
        self.max_batch = 4
        self.device = torch.device("cpu")


@pytest.mark.parametrize("argv,alpha,logs", [([], 0.0, False), (["--log_entropy"], 0.0, True),
                                             (["--entropy_alpha", "-0.05"], -0.05, True)])
def test_learner_reads_the_entropy_config(argv, alpha, logs):
    from distrl_llm_b200.learner import GRPOLearner, IdTokenizer
    from distrl_llm_b200.train_distributed import build_parser, config_from_args
    cfg = config_from_args(build_parser().parse_args(["--train_batch_size", "2"] + argv))
    ln = GRPOLearner(_HostPolicy(), IdTokenizer(), cfg)
    assert ln.entropy_alpha == alpha and ln.log_entropy is logs
    assert ln.last_metrics() == {}


class _EntLearner:
    def __init__(self, metrics):
        self.metrics = metrics

    def generate(self, task, sampling_params=None):
        return dict(task, answers=[], token_lengths=[])

    def compute_gradients(self, chunk):
        return {}, 1.0

    def apply_merged_gradients(self, grads):
        pass

    def train(self, candidates):
        return 0.5

    def save_adapter(self):
        pass

    def last_metrics(self):
        return dict(self.metrics)


def _run_trainer(monkeypatch, learner_metrics, extra):
    from distrl_llm_b200 import local_rpc, trainer as tr
    from distrl_llm_b200.generator import StubGenerator, synthetic_reward_function
    from tests.test_trainer_host import _oracle_prep
    from distrl_llm_b200 import trainer_prep
    monkeypatch.setattr(trainer_prep, "apply_advantages_and_topk", _oracle_prep)
    actors = [local_rpc.ActorHandle(lambda i=i: StubGenerator(500, 4, 12, seed=i)) for i in range(2)]
    learners = [local_rpc.ActorHandle(lambda m=m: _EntLearner(m)) for m in learner_metrics]
    config = dict(episodes=1, batch_size=6, learner_chunk_size=0, num_candidates=4, save_every=100, eval_every=0, topk=3,
                  learner="grpo", run_name="t", number_of_actors=2, number_of_learners=len(learners), max_steps=1, **extra)
    t = tr.Trainer(tr.SyntheticDataset(12, 500, 10, seed=0), tr.SyntheticDataset(2, 500, 10, seed=1),
                   synthetic_reward_function, config, actors=actors, learners=learners)
    t.train()
    for h in actors + learners:
        h.shutdown()
    return t.history[0]


def test_trainer_logs_token_weighted_entropy(monkeypatch):
    m = _run_trainer(monkeypatch, [{"entropy": 2.0, "entropy_tokens": 30}, {"entropy": 4.0, "entropy_tokens": 10},
                                   {"entropy": float("nan"), "entropy_tokens": 0}], {"entropy_alpha": 0.01})
    assert m["entropy"] == pytest.approx((2.0 * 30 + 4.0 * 10) / 40)
    m = _run_trainer(monkeypatch, [{"entropy": 3.0, "entropy_tokens": 7}], {"log_entropy": True})
    assert m["entropy"] == pytest.approx(3.0)


def test_trainer_has_no_entropy_key_when_off(monkeypatch):
    m = _run_trainer(monkeypatch, [{}, {}], {})
    assert "entropy" not in m and "loss" in m


def test_entropy_entry_points_reject_bad_arguments_without_gpu():
    from distrl_llm_b200 import _capi
    lib = _capi.load_library()
    rc = lib.b200rl_logprob_entropy(None, 0, None, None, None, None, None, 0.0, None, 0, 0, 0, None, None, None, 0, 0, 0,
                                    0.0, None, None)
    assert rc < 0 and b"logprob_entropy" in lib.b200rl_last_error()
    dummy = ctypes.c_void_p(16)   # never dereferenced: the checks fail before any launch
    rc = lib.b200rl_logprob_entropy(dummy, 8, dummy, dummy, None, None, None, 0.0, dummy, 1, 8, 1, None, None, None, 1, 1,
                                    1, 0.0, None, None)   # ent_out missing
    assert rc < 0 and b"ent_out" in lib.b200rl_last_error()
    rc = lib.b200rl_loss_value_entropy(dummy, dummy, dummy, None, 0.0, None, 0.0, dummy, 1, 1, 0, None, 0.01, None, None)
    assert rc < 0 and b"loss_value_entropy" in lib.b200rl_last_error()
    ea = _capi.EntropyArgs(0.01, None, None)
    la = _capi.LossArgs(1, 0, 1, 0, None, 0.0, None, 0.0)
    assert lib.b200rl_model_pass_ent(None, None, None, None, None, None, None, 1, 1, 1, ctypes.byref(la), ctypes.byref(ea),
                                     None) < 0
    assert lib.b200rl_model_pass_packed_ent(None, None, None, None, None, ctypes.byref(la), ctypes.byref(ea), None) < 0
    with pytest.raises(RuntimeError):
        _capi.check(rc, "loss_value_entropy")
