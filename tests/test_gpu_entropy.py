"""GPU tests of the per-token policy entropy and the entropy bonus (reference: BaseLearner.compute_entropy_bonus,
distributed_actor.py:266-281, never called: :377-379 and :472-480 are commented out).  Definitions: DESIGN.md.

  * G7 entropy variant (b200rl_logprob_entropy) against float64 torch on the same bf16 logits, and against the plain
    kernel: log-probs bit-identical, bonus-free gradients bit-identical;
  * loss-value variant against a float64 host formula;
  * the learner (classic and packed layouts, compact rows, fused passes, KL + clip) against the fp32 oracle
    (oracle/entropy_oracle.py on top of oracle/learner_oracle.py), the reference-pinned config-1 fixture and one full-width layer;
  * entropy logging off vs on with alpha = 0: bit-identical; two learners on one GPU log the token-weighted mean."""
import math

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

from oracle import entropy_oracle as eo  # noqa: E402  (checker only)
from oracle import learner_oracle as lo  # noqa: E402  (checker only)


# ---------------------------------------------------------------------------------------------------
# kernel
# ---------------------------------------------------------------------------------------------------
def _logits(rows, V, device, seed):
    g = torch.Generator(device=device).manual_seed(seed)
    z = torch.randn(rows, V, generator=g, device=device) * 3
    z[0, 7] = 60.0                     # a very peaked row (p_max ~ 1 - 1e-19)
    z[1, :V // 2] -= 20.0              # half the vocabulary far below the rest
    return z.to(torch.bfloat16)


def _slots_plain(logits, targets, coef, klw, ref_lp, old_lp, clip_eps, slot, n, write_grad):
    from distrl_llm_b200._capi import check, lib, ptr, stream
    rows, V = logits.shape
    lp = torch.zeros(n, device=logits.device, dtype=torch.float32)
    check(lib().b200rl_logprob_slots(ptr(logits), logits.stride(0), ptr(targets), ptr(coef), ptr(klw), ptr(ref_lp),
                                     ptr(old_lp), float(clip_eps), ptr(lp), rows, V, 1 if write_grad else 0, ptr(slot),
                                     stream()), "logprob_slots")
    return lp


def _entropy_weights(mask, alpha, Bm, nb):
    lens = mask.sum(1)
    e = torch.where(lens[:, None] > 0, alpha * mask.double() / (lens[:, None].double().clamp(min=1) * Bm * nb), 0.0)
    return lens.to(torch.int32), e.reshape(-1)


@pytest.mark.parametrize("rows,V,Bm", [(9, 512, 3), (64, 152064, 4), (33, 8192, 3)])
def test_entropy_kernel_vs_fp64(cuda, rows, V, Bm):
    from distrl_llm_b200 import ops
    T, nb, alpha = rows // Bm, 2, 0.7
    z = _logits(rows, V, cuda, seed=rows)
    g = torch.Generator(device=cuda).manual_seed(1)
    targets = torch.randint(0, V, (rows,), generator=g, device=cuda, dtype=torch.int32)
    mask = (torch.rand(Bm, T, generator=g, device=cuda) < 0.8).to(torch.int32)
    mask[0, :] = 1
    mask[-1, :] = 0                    # a len = 0 row: no bonus
    coef = torch.randn(rows, generator=g, device=cuda) * 1e-2 * mask.reshape(-1).float()
    coef[:3] = 0.0                     # rows 0..2: coef = 0 with e != 0 (mask[0] = 1)
    lens, e = _entropy_weights(mask, alpha, Bm, nb)
    # fp64 reference on the same bf16 logits
    z64 = z.double().requires_grad_(True)
    logp = torch.log_softmax(z64, -1)
    H = -(logp.exp() * logp).sum(-1)
    lp64 = logp.gather(1, targets.long()[:, None]).squeeze(1)
    ((coef.double() * lp64).sum() - (e * H).sum()).backward()
    dz_ref = z64.grad
    # scoring only
    zs = z.clone()
    lp, ent = ops.logprob_entropy(zs, targets, T=T)
    assert torch.equal(zs, z)
    assert torch.equal(lp, ops.logprob(z.clone(), targets))
    dH = (ent.double() - H.detach()).abs() / H.detach().clamp(min=1.0)
    print(f"rows {rows} V {V}: max |dH| / max(1, H) = {dH.max().item():.3e} (H in [{H.min().item():.3e}, {H.max().item():.3f}])")
    # fp32 accumulation of (s, u) over up to 152064 terms: measured on B200 <= 2.5e-7 (all three shapes)
    assert dH.max().item() <= 5e-7
    # scoring + gradient, bonus on
    zg, zp = z.clone(), z.clone()
    lp_g, ent_g = ops.logprob_entropy(zg, targets, coef, True, mask=mask, lens=lens, T=T, Bm=Bm, nb=nb, alpha=alpha)
    lp_p = ops.logprob(zp, targets, coef, True)
    assert torch.equal(lp_g, lp_p) and torch.equal(ent_g, ent)
    rel = ((zg.double() - dz_ref).norm() / dz_ref.norm()).item()
    print(f"rows {rows} V {V}: dz rel-L2 vs fp64 autograd {rel:.3e}")
    assert rel < 6e-3
    both_zero = (coef == 0) & (e == 0)
    assert both_zero.any() and float(zg[both_zero].float().abs().max()) == 0.0
    only_e = (coef == 0) & (e != 0)
    assert only_e.any() and float(zg[only_e].float().abs().max()) > 0.0
    # alpha = 0: the gradient is bit-identical to the plain kernel's
    z0 = z.clone()
    ops.logprob_entropy(z0, targets, coef, True, mask=mask, lens=lens, T=T, Bm=Bm, nb=nb, alpha=0.0)
    assert torch.equal(z0, zp)


def test_entropy_kernel_with_kl_clip_and_slots(cuda):
    from distrl_llm_b200 import ops
    Bm, T, V, nb, alpha = 4, 12, 8192, 1, -0.3
    n = Bm * T
    g = torch.Generator(device=cuda).manual_seed(3)
    mask = (torch.rand(Bm, T, generator=g, device=cuda) < 0.7).to(torch.int32)
    slot = torch.nonzero(mask.reshape(-1)).squeeze(1).to(torch.int32)           # compact rows: the live positions
    R = slot.numel()
    z = _logits(R, V, cuda, seed=5)
    targets = torch.randint(0, V, (R,), generator=g, device=cuda, dtype=torch.int32)
    coef = torch.randn(n, generator=g, device=cuda) * 1e-2 * mask.reshape(-1).float()
    klw = 0.05 * mask.reshape(-1).float()
    # reference / old log-probs near the current ones, so that the KL weight stays O(klw) and clipping hits some rows
    lp0 = _slots_plain(z.clone(), targets, None, None, None, None, 0.0, slot, n, False)
    ref_lp = lp0 + 0.1 * torch.randn(n, generator=g, device=cuda)
    old_lp = lp0 + 0.3 * torch.randn(n, generator=g, device=cuda)
    lens, e = _entropy_weights(mask, alpha, Bm, nb)
    zp, zg, z0 = z.clone(), z.clone(), z.clone()
    lp_p = _slots_plain(zp, targets, coef, klw, ref_lp, old_lp, 0.2, slot, n, True)
    lp_g, ent = ops.logprob_entropy(zg, targets, coef, True, klw=klw, ref_lp=ref_lp, old_lp=old_lp, clip_eps=0.2, slot=slot,
                                    mask=mask, lens=lens, T=T, Bm=Bm, nb=nb, alpha=alpha, n_slots=n)
    assert torch.equal(lp_g, lp_p)
    live = torch.zeros(n, dtype=torch.bool, device=cuda)
    live[slot.long()] = True
    assert float(ent[~live].abs().max()) == 0.0 and float(lp_g[~live].abs().max()) == 0.0
    logp = torch.log_softmax(z.double(), -1)
    H = -(logp.exp() * logp).sum(-1)
    assert ((ent[slot.long()].double() - H).abs() / H.clamp(min=1)).max().item() <= 5e-7
    # bonus gradient = plain gradient (KL + clip) + e p (ln p + H)
    p = logp.exp()
    ref = zp.double() + e[slot.long()][:, None] * p * (logp + H[:, None])
    rel = ((zg.double() - ref).norm() / ref.norm()).item()
    print(f"KL + clip + slots: dz rel-L2 {rel:.3e}")
    bonus = ((ref - zp.double()).norm() / ref.norm()).item()
    print(f"KL + clip + slots: bonus share of dz {bonus:.3e}")
    assert rel < 6e-3 and bonus > 10 * rel   # the bonus term is far above the rounding error
    ops.logprob_entropy(z0, targets, coef, True, klw=klw, ref_lp=ref_lp, old_lp=old_lp, clip_eps=0.2, slot=slot,
                        mask=mask, lens=lens, T=T, Bm=Bm, nb=nb, alpha=0.0, n_slots=n)
    assert torch.equal(z0, zp)


@pytest.mark.parametrize("grpo", [False, True])
def test_entropy_loss_value_vs_host(cuda, grpo):
    from distrl_llm_b200 import ops
    Bm, T, alpha = 5, 37, 0.013
    rng = np.random.default_rng(4)
    mask = (rng.random((Bm, T)) < 0.6).astype(np.int32)
    mask[2] = 0                                    # len = 0: contributes nothing
    lp = (-rng.random((Bm, T)) * 5).astype(np.float32)
    ent = (rng.random((Bm, T)) * 6).astype(np.float32)
    adv = rng.normal(size=Bm)
    d = lambda a: torch.from_numpy(a).to(cuda)
    accum = torch.full((1,), 0.25, device=cuda, dtype=torch.float64)
    eacc = torch.tensor([1.5, 2.0], device=cuda, dtype=torch.float64)
    ops.loss_value_entropy(d(lp), d(mask), d(adv), d(ent), alpha, accum, grpo, eacc)
    total = 0.0
    for i in range(Bm):
        L = mask[i].sum()
        if L == 0:
            continue
        pol = adv[i] if grpo else adv[i] * (lp[i].astype(np.float64) * mask[i]).sum() / L
        total += pol + alpha * (ent[i].astype(np.float64) * mask[i]).sum() / L
    want = 0.25 - total / Bm
    got = accum.item()
    assert abs(got - want) <= 1e-9, (got, want)
    hs, hn = eacc.tolist()
    assert abs(hs - 1.5 - (ent.astype(np.float64) * mask).sum()) <= 1e-9 and hn == 2.0 + mask.sum()
    # alpha = 0: the plain loss value, bit for bit
    a0, a1 = torch.zeros(1, device=cuda, dtype=torch.float64), torch.zeros(1, device=cuda, dtype=torch.float64)
    ops.loss_value_entropy(d(lp), d(mask), d(adv), d(ent), 0.0, a0, grpo)
    ops.loss_value(d(lp), d(mask), d(adv), a1, grpo)
    assert torch.equal(a0, a1)


# ---------------------------------------------------------------------------------------------------
# learner vs oracle
# ---------------------------------------------------------------------------------------------------
def _mk_cfg(ocfg):
    from distrl_llm_b200.policy import LMConfig
    return LMConfig(vocab=ocfg.vocab, hidden=ocfg.hidden, inter=ocfg.inter, n_layers=ocfg.n_layers,
                    n_q_heads=ocfg.n_q_heads, n_kv_heads=ocfg.n_kv_heads, head_dim=ocfg.head_dim,
                    lora_r=ocfg.lora_r, lora_alpha=ocfg.lora_alpha, rms_eps=ocfg.rms_eps, rope_theta=ocfg.rope_theta)


def _flat(d, names):
    return torch.cat([d[k].double().flatten().cpu() for k in names])


def _cos_rel(a, b):
    return ((a @ b) / (a.norm() * b.norm())).item(), ((a - b).norm() / b.norm()).item()


# name, head_dim, learner, alpha, N, B, fuse, share_prompts, compact_scored_rows, kl_beta, clip_eps
CASES = [
    ("classic_hd32_pg", 32, "pg", 0.01, 6, 2, 1, False, True, 0.0, 0.0),
    ("classic_hd64_grpo", 64, "grpo", -0.05, 6, 3, 1, False, True, 0.0, 0.0),
    ("packed_compact_grpo", 128, "grpo", 0.01, 8, 4, 1, True, True, 0.0, 0.0),
    ("packed_full_pg", 128, "pg", -0.05, 8, 4, 1, True, False, 0.0, 0.0),
    ("fused_packed_grpo", 128, "grpo", 0.01, 22, 4, 2, True, True, 0.0, 0.0),
    ("fused_classic_pg", 64, "pg", -0.05, 22, 4, 2, False, True, 0.0, 0.0),
    ("kl_clip_grpo", 128, "grpo", 0.01, 8, 4, 2, True, True, 0.2, 0.1),
]


@pytest.mark.parametrize("name,hd,kind,alpha,N,B,fuse,share,compact,beta,clip", CASES, ids=[c[0] for c in CASES])
def test_entropy_learner_vs_oracle(cuda, name, hd, kind, alpha, N, B, fuse, share, compact, beta, clip):
    from distrl_llm_b200.learner import GRPOLearner, IdTokenizer, Learner
    from distrl_llm_b200.policy import Policy
    nq, nkv = {32: (4, 2), 64: (4, 2), 128: (2, 1)}[hd]
    ocfg = lo.OracleConfig(vocab=2048, hidden=256, inter=512, n_layers=2, n_q_heads=nq, n_kv_heads=nkv, head_dim=hd,
                           lora_r=16, lora_alpha=16)
    params, nf4 = lo.make_params(ocfg, seed=8, lora_b_std=0.05 if beta else 0.01)
    # lm_head x 8 (exact in bf16): logits of std ~3, so that the softmax is far from uniform and the entropy gradient
    # p (ln p + H) is not negligible
    params["lm_head"] = params["lm_head"] * 8
    P, T = 16, 40
    rng = np.random.default_rng(5)
    prompts, answers = [], []
    for _ in range((N + 3) // 4):
        pr = rng.integers(1, ocfg.vocab, size=int(rng.integers(P // 2, P + 1))).tolist()
        for _ in range(4):
            prompts.append(pr)
            answers.append(rng.integers(1, ocfg.vocab, size=int(rng.integers(T // 4, T + 1))).tolist())
    prompts, answers = prompts[:N], answers[:N]
    rewards = rng.normal(size=N) * 0.1
    if N > 2 * B:
        rewards[B + 1] = 0.0               # micro-batch 1 is skipped by the reference's predicate (quirk Q1)
    pol = Policy.from_params(_mk_cfg(ocfg), params, nf4, cuda, max_batch=fuse * B, P=P, T=T)
    cls = Learner if kind == "pg" else GRPOLearner
    ln = cls(pol, IdTokenizer(), {"train_batch_size": B, "max_new_tokens": T, "max_prompt_tokens": P, "lr": 1e-5,
                                  "entropy_alpha": alpha, "kl_beta": beta, "clip_eps": clip, "share_prompts": share,
                                  "compact_scored_rows": compact, "fuse_microbatches": fuse})
    assert ln.log_entropy and ln.fuse_microbatches == fuse
    ids, am, ansm = lo.pad_batch(prompts, answers, P, T)
    ids, am, ansm = ids.to(cuda), am.to(cuda), ansm.to(cuda)
    old = None
    kw = {"kl_beta": beta} if beta else {}
    if clip:
        lp_all = torch.cat([ln.compute_current_policy_probs(pol, prompts[i:i + B], answers[i:i + B])[0] for i in range(0, N, B)])
        g = torch.Generator(device=cuda).manual_seed(0)
        old = (lp_all + 0.25 * torch.randn(lp_all.shape, generator=g, device=cuda)) * ansm.float()
        kw.update(old_lp=old, clip_eps=clip)
    loss = ln.compute_loss(prompts, answers, list(rewards), old_lp=old)
    grads = ln.export_gradients()
    met = ln.last_metrics()
    dparams = {k: (v.detach().to(cuda).requires_grad_(v.requires_grad)) for k, v in params.items()}
    ref_grads, ref_loss = eo.compute_gradients(dparams, ocfg, ids, am, ansm, rewards, P, B, kind, entropy_alpha=alpha, **kw)
    g0, loss0 = lo.compute_gradients(dparams, ocfg, ids, am, ansm, rewards, P, B, kind, **kw)
    names = lo.lora_names(ocfg)
    got = torch.cat([grads[pol.peft_name(i, m, ab)].double().flatten()
                     for i in range(ocfg.n_layers) for m in lo.LORA_MODULES for ab in ("A", "B")])
    ref, ref0 = _flat(ref_grads, names), _flat(g0, names)
    cos, rel = _cos_rel(got, ref)
    moved = ((ref - ref0).norm() / ref.norm()).item()
    nb = (N + B - 1) // B
    loss_tol = 4e-2 * sum(np.abs(rewards[i:i + B]).mean() for i in range(0, N, B)) + 2e-3 + abs(alpha) * 5e-2 * nb
    if clip or beta:
        loss_tol += 5e-2 * abs(ref_loss)
    print(f"{name}: loss {loss:.6f} (oracle {ref_loss:.6f}, without bonus {loss0:.6f}), grad cosine {cos:.6f} "
          f"rel-L2 {rel:.4f}, bonus moves the oracle gradient by {moved:.3f}")
    assert abs(loss - ref_loss) <= loss_tol, (loss, ref_loss)
    assert cos >= (0.995 if clip else 0.999) and rel <= (1e-1 if clip else 3e-2)
    if not (clip or beta):   # with KL + clip active the bonus is a small share of the gradient: agreement only
        assert moved > 3 * 3e-2, "the entropy term must move the gradient well beyond the tolerance"
    # the metric: mean H over the answer tokens of the micro-batches that were trained
    with torch.no_grad():
        H_ref = eo.compute_current_policy_entropy(dparams, ocfg, ids, am, P)
    keep = torch.tensor([bool(np.all(rewards[(i // B) * B:(i // B + 1) * B] != 0)) for i in range(N)], device=cuda)
    m = ansm.bool() & keep[:, None]
    assert met["entropy_tokens"] == int(m.sum())
    assert abs(met["entropy"] - H_ref[m].double().mean().item()) <= 1e-2, (met, H_ref[m].mean().item())
    # per-token H of the scoring API
    lp, mask, ent = ln.compute_current_policy_probs(pol, prompts[:B], answers[:B], return_entropy=True)
    mk = mask.bool()
    dH = (ent[mk] - H_ref[:B][mk]).abs()
    print(f"{name}: per-token |dH| max {dH.max().item():.3e} mean {dH.mean().item():.3e} nats")
    # H comes from bf16 logits of std ~3 (|z| up to ~12, bf16 ulp 0.03-0.06) like lp does; measured on B200: max 6.4e-2,
    # mean <= 1.0e-2 nats over the cases above
    assert dH.max().item() < 1e-1 and dH.mean().item() < 2e-2
    lp_only, _ = ln.compute_current_policy_probs(pol, prompts[:B], answers[:B])
    assert torch.equal(lp, lp_only)


def test_entropy_vs_reference_golden(cuda):
    """Library per-token H on BASELINE config 1 vs the reference helper's values (tests/golden/cfg1_entropy.npz)."""
    import os
    from distrl_llm_b200.learner import Learner, IdTokenizer
    from distrl_llm_b200.policy import Policy
    from tests.golden_utils import load_cfg1
    z, ocfg, params, nf4, prompts, answers = load_cfg1()
    ze = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "cfg1_entropy.npz"))
    assert str(ze["param_sha256"]) == str(z["param_sha256"])
    P, T, B = int(z["P"]), int(z["T"]), int(z["train_batch_size"])
    pol = Policy.from_params(_mk_cfg(ocfg), params, nf4, cuda, max_batch=B, P=P, T=T)
    ln = Learner(pol, IdTokenizer(), {"train_batch_size": B, "max_new_tokens": T, "max_prompt_tokens": P, "lr": 2e-5,
                                      "log_entropy": True})
    ent = torch.cat([ln.compute_current_policy_probs(pol, prompts[i:i + B], answers[i:i + B], return_entropy=True)[2]
                     for i in range(0, len(prompts), B)])
    m = torch.from_numpy(ze["answer_mask"]).bool()
    d = (ent.cpu()[m] - torch.from_numpy(ze["entropy"])[m]).abs()
    print(f"config 1 per-token H vs reference helper: max |dH| {d.max().item():.3e}, mean {d.mean().item():.3e} nats")
    # near-uniform rows (std ~0.2 logits): measured on B200 max 7.8e-5, mean 2.0e-5 nats
    assert d.max().item() < 2e-4


def test_entropy_cfg2_width_vs_oracle(cuda):
    """One full-width Qwen2.5-7B layer through the exact bench path (V = 152064, packed, fused, weight cache) with
    entropy_alpha = 0.01, against the fp32 oracle."""
    from tests.test_gpu_cfg2_shapes import B, GROUP, N, P, T, _build, _check_grads
    from tests.policy_bridge import flat_grad_from_oracle, oracle_config, oracle_params_from_policy
    from distrl_llm_b200.trainer_prep import synthetic_candidates
    cfg, pol, ln = _build(cuda, 1, "grpo", seed=41)
    ln.entropy_alpha, ln.log_entropy = 0.01, True
    ln._ent_accum = torch.zeros(2, device=cuda, dtype=torch.float64)
    _, (prompts, answers, adv) = synthetic_candidates(cfg.vocab, N, P, T, GROUP, seed=77, ragged=True)
    rewards = np.asarray(adv, dtype=np.float64)
    _, loss = ln._compute_gradients(prompts, answers, list(rewards), export=False)
    met = ln.last_metrics()
    torch.cuda.synchronize()
    ocfg = oracle_config(cfg)
    params = oracle_params_from_policy(pol)
    ids, am, ansm = lo.pad_batch(prompts, answers, P, T)
    ids, am, ansm = ids.to(cuda), am.to(cuda), ansm.to(cuda)
    ref_grads, ref_loss = eo.compute_gradients(params, ocfg, ids, am, ansm, rewards, P, B, "grpo", entropy_alpha=0.01)
    # GRPO loss = -mean(adv) - alpha * mean H: the second part carries the bf16-logit error of H
    assert abs(loss - ref_loss) <= 0.01 * 5e-2 * 2 + 1e-6, (loss, ref_loss)
    cos, rel = _check_grads(pol, flat_grad_from_oracle(pol, ref_grads))
    with torch.no_grad():
        H = torch.cat([eo.compute_current_policy_entropy(params, ocfg, ids[i:i + B], am[i:i + B], P) for i in range(0, N, B)])
    h_ref = H[ansm.bool()].double().mean().item()
    print(f"cfg2 width: loss {loss:.6f} (oracle {ref_loss:.6f}), cosine {cos:.6f}, rel-L2 {rel:.4f}, "
          f"entropy {met['entropy']:.5f} (oracle {h_ref:.5f})")
    assert abs(met["entropy"] - h_ref) <= 2e-2


@pytest.mark.parametrize("share", [True, False])
def test_entropy_logging_alone_changes_nothing(cuda, share):
    """log_entropy=True, entropy_alpha=0: loss, gradients and log-probs bit-identical to entropy off."""
    from distrl_llm_b200.learner import GRPOLearner, IdTokenizer
    from distrl_llm_b200.policy import Policy
    ocfg = lo.OracleConfig(vocab=2048, hidden=256, inter=512, n_layers=2, n_q_heads=2, n_kv_heads=1, head_dim=128,
                           lora_r=16, lora_alpha=16)
    params, nf4 = lo.make_params(ocfg, seed=9)
    P, T, B, N = 12, 36, 4, 10
    prompts, answers, rewards = lo.make_batch(ocfg, N, P, T, seed=2, ragged=True, group_size=5, learner="grpo")
    out = []
    for log in (False, True):
        pol = Policy.from_params(_mk_cfg(ocfg), params, nf4, cuda, max_batch=2 * B, P=P, T=T)
        ln = GRPOLearner(pol, IdTokenizer(), {"train_batch_size": B, "max_new_tokens": T, "max_prompt_tokens": P,
                                              "lr": 1e-5, "log_entropy": log, "share_prompts": share})
        lp_cap = torch.zeros(N, T, device=cuda)
        loss = ln.compute_loss(prompts, answers, list(rewards), lp_capture=lp_cap)
        out.append((loss, pol.lora_grad.clone(), lp_cap, ln.last_metrics()))
    (l0, g0, lp0, m0), (l1, g1, lp1, m1) = out
    assert l0 == l1 and torch.equal(g0, g1) and torch.equal(lp0, lp1)
    assert m0 == {} and m1["entropy_tokens"] > 0 and 0 < m1["entropy"] <= math.log(ocfg.vocab)


# ---------------------------------------------------------------------------------------------------
# trainer: two learners on one GPU (P2P harness of test_gpu_trainer.py)
# ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("alpha", [0.01, None], ids=["alpha0.01", "off"])
def test_trainer_two_learners_entropy_metric(cuda, alpha):
    from distrl_llm_b200 import local_rpc, train_distributed
    from distrl_llm_b200.actors import create_actor_and_learner
    from distrl_llm_b200.generator import synthetic_reward_function
    from distrl_llm_b200.trainer import SyntheticDataset, Trainer
    from tests.test_gpu_trainer import BASE
    argv = BASE + ["--number_of_learners", "2", "--max_steps", "2"] + (["--entropy_alpha", str(alpha)] if alpha else [])
    args = train_distributed.build_parser().parse_args(argv)
    config = train_distributed.config_from_args(args)
    config["learner_gpus"] = [0, 0]
    config["stub_generators_share_gpus"] = True
    actors, learners = create_actor_and_learner(2, 2, args.model, None, config)
    t = Trainer(SyntheticDataset(8, 2048, 12, seed=0), SyntheticDataset(2, 2048, 12, seed=1), synthetic_reward_function, config,
                actors=actors, learners=learners)
    steps, _ = t.train()
    assert steps == 2
    flats = local_rpc.get([l.export_flat.remote() for l in learners])
    assert torch.equal(flats[0], flats[1]) and float(flats[0].abs().sum()) > 0
    mets = local_rpc.get([l.last_metrics.remote() for l in learners])
    last = t.history[-1]
    if alpha is None:
        assert all(m == {} for m in mets) and all("entropy" not in h for h in t.history)
    else:
        vocab = local_rpc.get(learners[0].vocab_size.remote())
        n = sum(m["entropy_tokens"] for m in mets)
        want = sum(m["entropy"] * m["entropy_tokens"] for m in mets if m["entropy_tokens"]) / n
        assert n > 0 and last["entropy"] == pytest.approx(want, rel=1e-12)
        assert math.isfinite(last["entropy"]) and 0 < last["entropy"] <= math.log(vocab)
    for h in actors + learners:
        h.shutdown()
