"""ORACLE — TEST INFRASTRUCTURE ONLY.  Generates tests/golden/*.npz by executing the REFERENCE's own
learner code (BY571/DistRL-LLM, /root/reference) verbatim.

Runs only in the build container (the GPU box has no /root/reference); the fixtures it writes are
committed.  Recipe (SURVEY.md §8c, probe-verified):
  * stub the un-installable third-party modules in sys.modules: ray, unsloth, unsloth_zoo.vllm_utils,
    bitsandbytes (Adam8bit -> torch.optim.Adam), vllm — none of their arithmetic is used;
  * import the reference's distributed_actor.py unmodified; build Learner / GRPOLearner with
    cls.__new__ (their __init__ loads a 7B checkpoint through Unsloth) and set the attributes the hot
    path reads: tokenizer (FakeTok: token-id lists in, reference padding rules out), policy (stock HF
    Qwen2ForCausalLM, eager attention, + a torch LoRA wrapper with PEFT's formula on the 7 target
    modules of helper.py:29-37), max_prompt_tokens, max_new_tokens, update_batch_size, optimizer;
  * no GPU here: Tensor.to("cuda") is mapped to a no-op (the reference hard-codes .to("cuda")),
    torch.amp.autocast(device_type="cuda") degrades to fp32 on a CUDA-less host, which is the fp32
    golden; a second golden is taken with autocast redirected to CPU bf16.
The advantage / top-k block of Trainer.train (distributed_trainer.py:262-294) is inline code, so it is
executed by exec()-ing exactly those source lines with a fake `self`.

Usage: python oracle/make_golden.py   (writes tests/golden/)
"""
from __future__ import annotations

import os
import sys
import textwrap
import types

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = os.environ.get("B200RL_REFERENCE", "/root/reference")
sys.path.insert(0, ROOT)

from oracle import learner_oracle as lo  # noqa: E402


# ---------------------------------------------------------------------------------------------------
def install_stubs():
    def mod(name, **attrs):
        m = types.ModuleType(name)
        m.__dict__.update(attrs)
        sys.modules[name] = m
        return m

    def remote(*a, **k):
        if len(a) == 1 and callable(a[0]) and not k:
            return a[0]
        return lambda cls: cls

    mod("ray", remote=remote, get=lambda x, **k: x, init=lambda *a, **k: None, is_initialized=lambda: True)
    mod("ray.util")
    mod("ray.util.placement_group", placement_group=lambda *a, **k: None)
    mod("ray.util.scheduling_strategies", PlacementGroupSchedulingStrategy=object)

    class FastLanguageModel:
        @staticmethod
        def for_training(m):
            m.train()

        @staticmethod
        def for_inference(m):
            m.eval()

        @staticmethod
        def get_peft_model(*a, **k):
            raise RuntimeError("stub")

    mod("unsloth", FastLanguageModel=FastLanguageModel)
    mod("unsloth_zoo")
    mod("unsloth_zoo.vllm_utils", load_lora=lambda *a, **k: None, save_lora=lambda *a, **k: None)
    optim = types.SimpleNamespace(Adam8bit=torch.optim.Adam)
    mod("bitsandbytes", optim=optim)
    mod("vllm", SamplingParams=lambda **k: types.SimpleNamespace(**k))
    mod("wandb", init=lambda **k: None, log=lambda *a, **k: None)
    mod("datasets")
    # no CUDA in the build container: the reference hard-codes .to("cuda")
    if not torch.cuda.is_available():
        _orig_to = torch.Tensor.to

        def _to(self, *a, **k):
            if a and a[0] == "cuda":
                a = ("cpu",) + tuple(a[1:])
            if k.get("device") == "cuda":
                k["device"] = "cpu"
            return _orig_to(self, *a, **k)

        torch.Tensor.to = _to


class _Enc(dict):
    def to(self, device):
        return self


class FakeTok:
    """Token-id passthrough tokenizer emulating the reference's two batch_encode_plus calls
    (distributed_actor.py:217-229): padding='max_length', truncation=True, padding_side left/right."""

    def __init__(self, pad_id=0):
        self.pad_id = pad_id

    def batch_encode_plus(self, items, return_tensors="pt", padding="max_length", padding_side="right",
                          max_length=None, truncation=True):
        n = len(items)
        ids = torch.full((n, max_length), self.pad_id, dtype=torch.long)
        mask = torch.zeros((n, max_length), dtype=torch.long)
        for i, it in enumerate(items):
            it = list(it)[:max_length]
            if padding_side == "left":
                if it:
                    ids[i, max_length - len(it):] = torch.tensor(it)
                    mask[i, max_length - len(it):] = 1
            else:
                ids[i, :len(it)] = torch.tensor(it)
                mask[i, :len(it)] = 1
        return _Enc(input_ids=ids, attention_mask=mask)


class LoraLinear(torch.nn.Module):
    """PEFT lora.Linear forward restated: base(x) + lora_B(lora_A(x)) * scaling, adapter name 'default'."""

    def __init__(self, base, A, B, scaling):
        super().__init__()
        self.base_layer = base
        for p in base.parameters():
            p.requires_grad_(False)
        r = A.shape[0]
        self.lora_A = torch.nn.ModuleDict({"default": torch.nn.Linear(A.shape[1], r, bias=False)})
        self.lora_B = torch.nn.ModuleDict({"default": torch.nn.Linear(r, B.shape[0], bias=False)})
        self.lora_A["default"].weight.data.copy_(A)
        self.lora_B["default"].weight.data.copy_(B)
        self.scaling = scaling

    def forward(self, x):
        return self.base_layer(x) + self.lora_B["default"](self.lora_A["default"](x)) * self.scaling


def build_hf_policy(cfg: lo.OracleConfig, params: dict):
    from transformers import Qwen2Config, Qwen2ForCausalLM
    hc = Qwen2Config(vocab_size=cfg.vocab, hidden_size=cfg.hidden, intermediate_size=cfg.inter,
                     num_hidden_layers=cfg.n_layers, num_attention_heads=cfg.n_q_heads,
                     num_key_value_heads=cfg.n_kv_heads, rms_norm_eps=cfg.rms_eps,
                     rope_parameters={"rope_type": "default", "rope_theta": cfg.rope_theta},
                     max_position_embeddings=4096, tie_word_embeddings=False, attention_dropout=0.0)
    hc._attn_implementation = "eager"
    model = Qwen2ForCausalLM(hc).float()
    for p in model.parameters():
        p.requires_grad_(False)
    with torch.no_grad():
        model.model.embed_tokens.weight.copy_(params["embed"])
        model.lm_head.weight.copy_(params["lm_head"])
        model.model.norm.weight.copy_(params["final_norm"])
        for i, layer in enumerate(model.model.layers):
            at, mlp = layer.self_attn, layer.mlp
            at.q_proj.weight.copy_(params[f"l{i}.wq"]); at.q_proj.bias.copy_(params[f"l{i}.bq"])
            at.k_proj.weight.copy_(params[f"l{i}.wk"]); at.k_proj.bias.copy_(params[f"l{i}.bk"])
            at.v_proj.weight.copy_(params[f"l{i}.wv"]); at.v_proj.bias.copy_(params[f"l{i}.bv"])
            at.o_proj.weight.copy_(params[f"l{i}.wo"])
            mlp.gate_proj.weight.copy_(params[f"l{i}.wg"])
            mlp.up_proj.weight.copy_(params[f"l{i}.wu"])
            mlp.down_proj.weight.copy_(params[f"l{i}.wd"])
            layer.input_layernorm.weight.copy_(params[f"l{i}.ln1"])
            layer.post_attention_layernorm.weight.copy_(params[f"l{i}.ln2"])
    s = cfg.lora_scale
    for i, layer in enumerate(model.model.layers):
        at, mlp = layer.self_attn, layer.mlp
        for owner, attr, m in ((at, "q_proj", "q"), (at, "k_proj", "k"), (at, "v_proj", "v"), (at, "o_proj", "o"),
                               (mlp, "gate_proj", "gate"), (mlp, "up_proj", "up"), (mlp, "down_proj", "down")):
            setattr(owner, attr, LoraLinear(getattr(owner, attr), params[f"l{i}.{m}.A"].detach(),
                                            params[f"l{i}.{m}.B"].detach(), s))
    return model


HF_NAME = {"q": "self_attn.q_proj", "k": "self_attn.k_proj", "v": "self_attn.v_proj", "o": "self_attn.o_proj",
           "gate": "mlp.gate_proj", "up": "mlp.up_proj", "down": "mlp.down_proj"}


def hf_grad_name(i, m, ab):
    return f"model.layers.{i}.{HF_NAME[m]}.lora_{ab}.default.weight"


def make_reference_learner(kind, cfg, params, P, T, train_batch_size, lr=2e-5):
    import distributed_actor as da  # the reference module, unmodified
    cls = da.Learner if kind == "pg" else da.GRPOLearner
    ln = cls.__new__(cls)
    ln.tokenizer = FakeTok()
    ln.policy = build_hf_policy(cfg, params)
    ln.max_prompt_tokens = P
    ln.max_new_tokens = T
    ln.update_batch_size = train_batch_size
    ln.model_gpu_id = 0
    ln.optimizer = torch.optim.Adam([p for p in ln.policy.parameters() if p.requires_grad], lr=lr)
    return ln


def run_reference_trainer_block(rewards_per_problem, learner_type, topk, answers=None):
    """exec() the reference's own advantage + top-k source lines (distributed_trainer.py:262-294)."""
    src = open(os.path.join(REF, "distributed_trainer.py")).read().split("\n")
    block = textwrap.dedent("\n".join(src[261:294]))  # 1-based lines 262..294
    n_prob = len(rewards_per_problem)
    C = rewards_per_problem[0].shape[0]
    cand = {
        "rewards": [r.copy() for r in rewards_per_problem],
        "token_lengths": [[1] * C for _ in range(n_prob)],
        "answers": answers or [[f"a{j}_{c}" for c in range(C)] for j in range(n_prob)],
        "problem": [[f"p{j}"] * C for j in range(n_prob)],
    }
    ns = {"np": np, "candidates": [cand], "self": types.SimpleNamespace(learner_type=learner_type, topk=topk),
          "mean_task_acc_rewards": [], "mean_task_format_reward": [], "mean_task_token_length": [],
          "max_task_acc_rewards": [], "min_task_acc_rewards": []}
    exec(block, ns)
    return ns["candidates"][0]


def main():
    assert os.path.isdir(REF), f"{REF} not found: goldens can only be generated in the build container"
    install_stubs()
    sys.path.insert(0, REF)
    out_dir = os.path.join(ROOT, "tests", "golden")
    os.makedirs(out_dir, exist_ok=True)
    torch.manual_seed(0)

    # ---- BASELINE config 1: PG (and GRPO) learner, tiny 2-layer/128-dim model, 4 completions len 32 ----
    cfg = lo.OracleConfig(vocab=512, hidden=128, inter=256, n_layers=2, n_q_heads=4, n_kv_heads=2, head_dim=32,
                          lora_r=16, lora_alpha=16)
    P, T, B = 16, 32, 2
    seed = 1234
    params, nf4 = lo.make_params(cfg, seed=seed)
    prompts, answers, _ = lo.make_batch(cfg, 4, P, T, seed=1, ragged=True)
    rewards = np.array([1.1, 0.1, 0.2, 1.0])  # summed (format+accuracy) rewards of one group of 4
    baseline = rewards.mean()
    fixtures = {"P": P, "T": T, "train_batch_size": B, "rewards": rewards, "baseline": baseline,
                "cfg": np.array([cfg.vocab, cfg.hidden, cfg.inter, cfg.n_layers, cfg.n_q_heads, cfg.n_kv_heads,
                                 cfg.head_dim, cfg.lora_r, cfg.lora_alpha], dtype=np.float64)}
    for i, (p, a) in enumerate(zip(prompts, answers)):
        fixtures[f"prompt{i}"] = np.array(p)
        fixtures[f"answer{i}"] = np.array(a)
    # the parameters are not stored (they would more than double the file): the loader regenerates them from the seed
    # and checks them against this digest
    fixtures["param_seed"] = np.int64(seed)
    fixtures["param_sha256"] = np.array(lo.params_digest(params, nf4))

    for mode in ("fp32", "bf16"):
        ctx = None
        if mode == "bf16":
            real_autocast = torch.amp.autocast

            def cpu_autocast(device_type="cuda", dtype=None, **k):  # redirect the reference's cuda autocast
                return real_autocast(device_type="cpu", dtype=dtype, **k)

            torch.amp.autocast = cpu_autocast
            ctx = real_autocast
        for kind in ("pg", "grpo"):
            ln = make_reference_learner(kind, cfg, params, P, T, B)
            # PG subtracts the per-problem baseline in Learner.train (:403-406); GRPO gets normalised advantages
            if kind == "pg":
                r = list(rewards - baseline)
            else:
                adv, _ = lo.group_advantages(np.stack([rewards * 0.0, rewards], -1), "grpo")
                r = list(adv)
                fixtures["grpo_adv"] = np.asarray(adv)
            ln.policy.train()
            grads, loss = ln._compute_gradients(prompts, answers, r)  # REFERENCE CODE (distributed_actor.py:283-294)
            fixtures[f"{mode}.{kind}.loss"] = np.float64(loss)
            for i in range(cfg.n_layers):
                for m in lo.LORA_MODULES:
                    for ab in ("A", "B"):
                        fixtures[f"{mode}.{kind}.grad.l{i}.{m}.{ab}"] = grads[hf_grad_name(i, m, ab)].float().numpy()
            if mode == "fp32" and kind == "pg":
                # per-token log-probs from the reference's scoring function (:215-261)
                with torch.no_grad():
                    lp, am = ln.compute_current_policy_probs(ln.policy, prompts[:B], answers[:B])
                fixtures["fp32.logp_mb0"] = lp.float().numpy()
                fixtures["answer_mask_mb0"] = am.numpy()
                # multi-learner merge + step: two learners' grads through the reference's apply_merged_gradients
                g1, _ = ln._compute_gradients(prompts[:2], answers[:2], r[:2])
                g2, _ = ln._compute_gradients(prompts[2:], answers[2:], r[2:])
                ln.optimizer.zero_grad()
                ln.apply_merged_gradients([g1, g2])  # REFERENCE CODE (:302-333) with Adam8bit -> torch Adam
                # stored as the fp32 update (new - old), which compresses better and adds back to the new value exactly
                sd = dict(ln.policy.named_parameters())
                for i in range(cfg.n_layers):
                    for m in lo.LORA_MODULES:
                        for ab in ("A", "B"):
                            new = sd[hf_grad_name(i, m, ab)].detach().numpy()
                            old = params[f"l{i}.{m}.{ab}"].detach().numpy()
                            assert np.array_equal(old + (new - old), new)
                            fixtures[f"fp32.merged_update.l{i}.{m}.{ab}"] = new - old
            if mode == "fp32" and kind == "grpo":
                # quirk Q1: a micro-batch containing an exact-zero reward is skipped (:459)
                rq = [0.5, 0.0, -0.25, 1.0]
                gq, lq = ln._compute_gradients(prompts, answers, rq)
                fixtures["fp32.q1.rewards"] = np.array(rq)
                fixtures["fp32.q1.loss"] = np.float64(lq)
                fixtures["fp32.q1.grad.l0.q.B"] = gq[hf_grad_name(0, "q", "B")].numpy()
        if ctx is not None:
            torch.amp.autocast = ctx
    np.savez_compressed(os.path.join(out_dir, "cfg1_learner.npz"), **fixtures)

    # ---- Trainer advantage / top-k block, executed from the reference source ----
    rng = np.random.default_rng(7)
    adv_fix = {}
    for case, (n_prob, C, topk) in enumerate([(3, 8, 8), (2, 16, 4), (2, 256, 128), (2, 7, 16)]):
        rw = []
        for _ in range(n_prob):
            fmt = rng.choice([0.0, 0.1, 0.2, 0.35], size=C)
            acc = (rng.random(C) < 0.3).astype(np.float64) + rng.random(C) * 1e-3  # distinct sums: no argsort ties
            rw.append(np.stack([fmt, acc], -1))
        adv_fix[f"c{case}.rewards"] = np.stack(rw)
        adv_fix[f"c{case}.topk"] = np.int64(topk)
        for lt in ("grpo", "pg"):
            out = run_reference_trainer_block(rw, lt, topk)
            adv_fix[f"c{case}.{lt}.filtered_rewards"] = np.stack(out["rewards"])
            adv_fix[f"c{case}.{lt}.filtered_answers"] = np.array(out["answers"])
            if lt == "pg":
                adv_fix[f"c{case}.pg.baselines"] = np.array(out["baselines"])
    np.savez_compressed(os.path.join(out_dir, "trainer_advantages.npz"), **adv_fix)
    print("wrote", os.listdir(out_dir))


if __name__ == "__main__":
    main()
