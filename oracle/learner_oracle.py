"""ORACLE — TEST INFRASTRUCTURE ONLY.  CPU/torch restatement of the reference learner hot path.

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs may import
this module; the product path (distrl_llm_b200/*) never does.

Every function cites the reference code it restates (paths relative to /root/reference, BY571/DistRL-LLM
@ a1099fd).  Pinning: tests/test_oracle.py checks this module against tests/golden/*.npz, which were
produced by oracle/make_golden.py running the reference's OWN `Learner` / `GRPOLearner` code verbatim
(third-party imports stubbed, HF Qwen2ForCausalLM + a torch LoRA wrapper as `policy`).

What is NOT pinned by the reference (arithmetic lives in un-vendored dependencies, SURVEY.md §8c):
  * model forward: restated from HF transformers 5.5 `Qwen2ForCausalLM` (eager attention) — pinned
    against HF itself through the golden vectors;
  * NF4: restated from the QLoRA / bitsandbytes 0.45.2 `quantize_4bit(quant_type="nf4",
    blocksize=64)` published format (no double quantisation) — "parity unpinned" vs real bnb files;
  * optimizer: bnb Adam8bit is restated as fp32 torch.optim.Adam (8-bit state not reproducible) —
    post-step weights "parity unpinned";
  * KL-to-reference term: absent from the reference (beta=0 reproduces it exactly);
  * clipped-ratio surrogate / inner epochs (old_lp, clip_eps): absent from the reference (its ratio is identically 1);
    clip_eps=0 or old_lp=None reproduces it exactly — the oracle restates THIS repo's definition, "parity unpinned".
"""
from __future__ import annotations

import hashlib
import math
from dataclasses import dataclass

import numpy as np
import torch

LORA_MODULES = ("q", "k", "v", "o", "gate", "up", "down")  # helper.py:29-37 target_modules


@dataclass
class OracleConfig:
    vocab: int
    hidden: int
    inter: int
    n_layers: int
    n_q_heads: int
    n_kv_heads: int
    head_dim: int
    lora_r: int
    lora_alpha: float
    rms_eps: float = 1e-6
    rope_theta: float = 1e6

    @property
    def lora_scale(self) -> float:
        return self.lora_alpha / self.lora_r  # PEFT: scaling = lora_alpha / r (use_rslora=False, helper.py:44)

    def module_shapes(self):
        """(in, out) of each LoRA target module."""
        H, I = self.hidden, self.inter
        qd, kd = self.n_q_heads * self.head_dim, self.n_kv_heads * self.head_dim
        return {"q": (H, qd), "k": (H, kd), "v": (H, kd), "o": (qd, H), "gate": (H, I), "up": (H, I), "down": (I, H)}


# ---------------------------------------------------------------------------------------------------
# NF4 (bitsandbytes [3P] format restated; see header)
# ---------------------------------------------------------------------------------------------------
NF4_LEVELS = np.array(
    [-1.0, -0.6961928009986877, -0.5250730514526367, -0.39491748809814453, -0.28444138169288635,
     -0.18477343022823334, -0.09105003625154495, 0.0, 0.07958029955625534, 0.16093020141124725,
     0.24611230194568634, 0.33791524171829224, 0.44070982933044434, 0.5626170039176941,
     0.7229568362236023, 1.0], dtype=np.float32)


def nf4_quantize(w: np.ndarray):
    """w: float32 array, size % 64 == 0 -> (packed uint8 [n/2], absmax float32 [n/64])."""
    flat = w.astype(np.float32).reshape(-1, 64)
    absmax = np.abs(flat).max(axis=1)
    inv = np.where(absmax > 0, 1.0 / np.maximum(absmax, 1e-45), 0.0).astype(np.float32)
    x = flat * inv[:, None]
    mid = 0.5 * (NF4_LEVELS[:-1] + NF4_LEVELS[1:])
    codes = (x[..., None] > mid[None, None]).sum(-1).astype(np.uint8)
    packed = ((codes[:, 0::2] << 4) | codes[:, 1::2]).reshape(-1)  # even element in the high nibble
    return packed, absmax.astype(np.float32)


def nf4_dequantize(packed: np.ndarray, absmax: np.ndarray, shape) -> torch.Tensor:
    """-> bf16 tensor of `shape`: bf16(level[code] * absmax) exactly like bnb's dequantize to bf16."""
    hi, lo = packed >> 4, packed & 15
    vals = np.stack([NF4_LEVELS[hi], NF4_LEVELS[lo]], -1).reshape(-1, 64) * absmax[:, None].astype(np.float32)
    return torch.from_numpy(vals.reshape(shape).astype(np.float32)).to(torch.bfloat16)


# ---------------------------------------------------------------------------------------------------
# model forward (restates transformers Qwen2ForCausalLM, eager attention, + PEFT LoRA formula)
# ---------------------------------------------------------------------------------------------------
def _rmsnorm(x, w, eps):
    # Qwen2RMSNorm.forward: fp32 variance, weight * hidden.to(input_dtype)
    var = x.float().pow(2).mean(-1, keepdim=True)
    xh = (x.float() * torch.rsqrt(var + eps)).to(x.dtype)
    return w * xh


def _rotate_half(x):
    h = x.shape[-1] // 2
    return torch.cat([-x[..., h:], x[..., :h]], -1)


def _lora_linear(x, W, b, A, B, s):
    # PEFT LoRA Linear forward: base(x) + lora_B(lora_A(dropout(x))) * scaling   (dropout 0, helper.py:39)
    y = x @ W.T
    if b is not None:
        y = y + b
    return y + (x @ A.T) @ B.T * s


def model_forward(params: dict, cfg: OracleConfig, ids: torch.Tensor, attn_mask: torch.Tensor,
                  dtype=torch.float32, lora_off=False) -> torch.Tensor:
    """Logits [B, L, V].  `params`: base tensors ('embed','final_norm','lm_head', 'l{i}.wq' ...,
    'l{i}.bq'/bk/bv, 'l{i}.ln1/ln2') and LoRA tensors 'l{i}.{mod}.A' [r,in] / '.B' [out,r].
    position_ids = arange(L) even under left padding (reference passes none, distributed_actor.py:241-243;
    transformers Qwen2Model.forward builds arange)."""
    B, L = ids.shape
    dev = ids.device
    s = 0.0 if lora_off else cfg.lora_scale  # lora_off: adapter disabled = reference policy of the KL term
    hd, nq, nkv = cfg.head_dim, cfg.n_q_heads, cfg.n_kv_heads
    p = lambda name: params[name].to(dtype) if params[name].dtype.is_floating_point else params[name]
    x = p("embed")[ids]
    pos = torch.arange(L, device=dev).float()
    inv = 1.0 / (cfg.rope_theta ** (torch.arange(0, hd, 2, device=dev).float() / hd))
    fr = pos[:, None] * inv[None]
    emb = torch.cat([fr, fr], -1)
    cos, sin = emb.cos().to(dtype)[None, None], emb.sin().to(dtype)[None, None]
    causal = torch.tril(torch.ones(L, L, dtype=torch.bool, device=dev))
    ok = causal[None, None] & attn_mask.bool()[:, None, None, :]
    neg = torch.finfo(dtype).min
    bias = torch.zeros(B, 1, L, L, dtype=dtype, device=dev).masked_fill(~ok, neg)
    for i in range(cfg.n_layers):
        g = lambda n: p(f"l{i}.{n}")
        h = _rmsnorm(x, g("ln1"), cfg.rms_eps)
        q = _lora_linear(h, g("wq"), g("bq"), g("q.A"), g("q.B"), s).view(B, L, nq, hd).transpose(1, 2)
        k = _lora_linear(h, g("wk"), g("bk"), g("k.A"), g("k.B"), s).view(B, L, nkv, hd).transpose(1, 2)
        v = _lora_linear(h, g("wv"), g("bv"), g("v.A"), g("v.B"), s).view(B, L, nkv, hd).transpose(1, 2)
        q = q * cos + _rotate_half(q) * sin
        k = k * cos + _rotate_half(k) * sin
        k = k.repeat_interleave(nq // nkv, dim=1)
        v = v.repeat_interleave(nq // nkv, dim=1)
        att = (q @ k.transpose(-1, -2)) * (hd ** -0.5) + bias
        att = torch.softmax(att.float(), -1).to(dtype)
        o = (att @ v).transpose(1, 2).reshape(B, L, nq * hd)
        x = x + _lora_linear(o, g("wo"), None, g("o.A"), g("o.B"), s)
        h = _rmsnorm(x, g("ln2"), cfg.rms_eps)
        gate = _lora_linear(h, g("wg"), None, g("gate.A"), g("gate.B"), s)
        up = _lora_linear(h, g("wu"), None, g("up.A"), g("up.B"), s)
        x = x + _lora_linear(torch.nn.functional.silu(gate) * up, g("wd"), None, g("down.A"), g("down.B"), s)
    x = _rmsnorm(x, p("final_norm"), cfg.rms_eps)
    return x @ p("lm_head").T


# ---------------------------------------------------------------------------------------------------
# learner math
# ---------------------------------------------------------------------------------------------------
def pad_batch(prompt_ids, answer_ids, P, T, pad_id=0):
    """BaseLearner.compute_current_policy_probs tokenise+pad (distributed_actor.py:217-239) on token-id
    lists: prompts LEFT-padded / right-truncated to exactly P, answers RIGHT-padded / truncated to T."""
    B = len(prompt_ids)
    ids = np.full((B, P + T), pad_id, dtype=np.int64)
    mask = np.zeros((B, P + T), dtype=np.int64)
    for i in range(B):
        p = list(prompt_ids[i])[:P]
        a = list(answer_ids[i])[:T]
        ids[i, P - len(p):P] = p
        mask[i, P - len(p):P] = 1
        ids[i, P:P + len(a)] = a
        mask[i, P:P + len(a)] = 1
    return torch.from_numpy(ids), torch.from_numpy(mask), torch.from_numpy(mask[:, P:].copy())


def compute_current_policy_probs(params, cfg, ids, attn_mask, P, dtype=torch.float32, lora_off=False):
    """distributed_actor.py:241-261: logits -> shift (:245-246) -> slice to the answer (:248-249) ->
    per-row log_softmax + gather (:252-259).  Returns action_log_probs [B, T] (fp32 like autocast's
    log_softmax)."""
    logits = model_forward(params, cfg, ids, attn_mask, dtype, lora_off)
    logits = logits[:, :-1, :]
    targets = ids[:, 1:]
    logits = logits[:, P - 1:]
    targets = targets[:, P - 1:]
    lp = torch.log_softmax(logits.float(), dim=-1)
    return torch.gather(lp, 2, targets.unsqueeze(-1)).squeeze(-1)


def compute_loss(params, cfg, ids, attn_mask, answer_mask, rewards, P, train_batch_size, learner="pg",
                 dtype=torch.float32, reference_quirks=True, kl_beta=0.0, old_lp=None, clip_eps=0.0, lp_capture=None):
    """Learner.compute_loss (distributed_actor.py:349-395) / GRPOLearner.compute_loss (:440-493).
    Accumulates .grad on the LoRA tensors of `params` (those with requires_grad) and returns the float
    the reference returns: the SUM over micro-batches of the per-micro-batch mean loss (quirk Q2)."""
    rewards = torch.as_tensor(np.asarray(rewards), dtype=torch.float64).to(ids.device)  # :350 / :441 -> float64 tensor .to("cuda")
    N = ids.shape[0]
    nb = (N + train_batch_size - 1) // train_batch_size  # :354-356
    total = 0.0
    for i in range(nb):
        sl = slice(i * train_batch_size, min((i + 1) * train_batch_size, N))
        r = rewards[sl]
        if reference_quirks and bool(r.all() == 0):  # :367 / :459 — skips when ANY reward is exactly 0 (quirk Q1)
            continue
        lp = compute_current_policy_probs(params, cfg, ids[sl], attn_mask[sl], P, dtype)
        m = answer_mask[sl]
        if lp_capture is not None:
            lp_capture[sl] = lp.detach()
        if old_lp is not None and clip_eps > 0:
            # NOT in the reference (its ratio is exp(lp - lp.detach()) == 1, :467; SURVEY.md 8(f) N4; parity unpinned):
            # PPO / GRPO clipped surrogate against the log-probs of the policy that generated the batch,
            #   min(rho * A, clip(rho, 1-eps, 1+eps) * A),  rho = exp(lp - old_lp),
            # normalised like the reference's loss (mask, / len, mean over the micro-batch)
            rho = torch.exp(lp - old_lp[sl].to(lp.device))
            a = r[:, None].to(lp.dtype)
            surr = torch.minimum(rho * a, torch.clamp(rho, 1 - clip_eps, 1 + clip_eps) * a)
            loss = -((surr * m).sum(-1) / m.sum(-1)).mean()
        elif learner == "pg":
            per_seq = (lp * m).sum(-1) / m.sum(-1)  # :375
            loss = -(per_seq * r).mean()
        else:
            imp = torch.exp(lp - lp.detach())  # :467
            per_seq = (imp * m).sum(-1) / m.sum(-1)  # :470
            loss = -(per_seq * r).mean()
        if kl_beta:
            # NOT in the reference (parity unpinned): KL(pi||pi_ref) with the k3 estimator, pi_ref = adapter off,
            # normalised exactly like the policy term (mask, /len, mean over the micro-batch)
            with torch.no_grad():
                q = compute_current_policy_probs(params, cfg, ids[sl], attn_mask[sl], P, dtype, lora_off=True)
            d = q - lp
            loss = loss + kl_beta * (((torch.exp(d) - d - 1) * m).sum(-1) / m.sum(-1)).mean()
        loss = loss / nb  # :375+:382 / :470+:479
        loss.backward()  # :385 / :483
        total += loss.item() * nb  # :387-389 / :485-487
    return total


def lora_names(cfg: OracleConfig):
    return [f"l{i}.{m}.{ab}" for i in range(cfg.n_layers) for m in LORA_MODULES for ab in ("A", "B")]


def compute_gradients(params, cfg, ids, attn_mask, answer_mask, rewards, P, train_batch_size, learner, **kw):
    """BaseLearner._compute_gradients (distributed_actor.py:283-294): zero_grad, compute_loss, export
    {name: grad (zeros if None)}."""
    for n in lora_names(cfg):
        params[n].grad = None
    loss = compute_loss(params, cfg, ids, attn_mask, answer_mask, rewards, P, train_batch_size, learner, **kw)
    grads = {n: (params[n].grad.clone() if params[n].grad is not None else torch.zeros_like(params[n]))
             for n in lora_names(cfg)}
    return grads, loss


def merge_gradients(grad_dicts):
    """BaseLearner.apply_merged_gradients merge part (distributed_actor.py:311-323): elementwise mean."""
    n = len(grad_dicts)
    out = {k: torch.zeros_like(v) for k, v in grad_dicts[0].items()}
    for g in grad_dicts:
        for k in g:
            out[k] += g[k]
    for k in out:
        out[k] /= n
    return out


def adam_step(params, grads, state, lr, betas=(0.9, 0.999), eps=1e-8, weight_decay=0.0):
    """optimizer.step() (:332/:414/:512) restated as fp32 Adam(W) (see header: Adam8bit unpinned).
    `state`: {'step': int, name: (m, v)} updated in place."""
    state["step"] = state.get("step", 0) + 1
    t = state["step"]
    b1, b2 = betas
    for n, g in grads.items():
        p = params[n].data
        m, v = state.setdefault(n, (torch.zeros_like(p), torch.zeros_like(p)))
        if weight_decay:
            p.mul_(1 - lr * weight_decay)
        m.lerp_(g, 1 - b1)
        v.mul_(b2).addcmul_(g, g, value=1 - b2)
        denom = (v.sqrt() / math.sqrt(1 - b2 ** t)).add_(eps)
        p.addcdiv_(m, denom, value=-(lr / (1 - b1 ** t)))


def split_evenly(n_items, n_learners):
    """Trainer.train multi-learner split (distributed_trainer.py:312-322): even chunks, remainder to the
    first learners. Returns [(start, size)]."""
    sizes = [n_items // n_learners] * n_learners
    for i in range(n_items % n_learners):
        sizes[i] += 1
    out, start = [], 0
    for s in sizes:
        out.append((start, s))
        start += s
    return out


# ---------------------------------------------------------------------------------------------------
# advantages / top-k (Trainer.train, distributed_trainer.py:262-294)
# ---------------------------------------------------------------------------------------------------
def group_advantages(batch_reward: np.ndarray, learner: str):
    """batch_reward [C, 2] float64 (format, accuracy).  GRPO (:273,:276): (s-mean)/(std+1e-8);
    PG (:267,:274,:278-279): rewards = s, baseline = mean(s)."""
    s = batch_reward.sum(axis=1)
    baseline = np.mean(s)
    if learner == "grpo":
        return (s - np.mean(s)) / (np.std(s) + 1e-8), baseline
    return s, baseline


def topk_filter(values: np.ndarray, topk: int, stable=True):
    """:287 `np.argsort(rewards)[-topk:]` (ascending).  numpy's default introsort is not stable; the
    oracle and the CUDA kernel both use the stable order (ties keep candidate order) — documented
    divergence that can only permute equal-valued candidates."""
    return np.argsort(values, kind="stable" if stable else None)[-topk:]


# ---------------------------------------------------------------------------------------------------
# synthetic parameters (SURVEY.md §8d "Synthetic inputs")
# ---------------------------------------------------------------------------------------------------
def make_params(cfg: OracleConfig, seed=0, quantize_base=True, lora_b_std=0.01, device="cpu"):
    """Random-init base (N(0, 0.02^2), HF initializer_range) rounded through NF4 (so the dense weights the
    oracle/HF consume are exactly what the CUDA path dequantises), norms ~ 1, LoRA A kaiming-uniform(a=sqrt5),
    B ~ N(0, lora_b_std^2) (non-zero on purpose: with PEFT's B=0 init dA would be identically 0).
    Returns (params, nf4) where nf4[name] = (packed, absmax) for each base matrix."""
    g = torch.Generator().manual_seed(seed)
    H, I, V = cfg.hidden, cfg.inter, cfg.vocab
    qd, kd = cfg.n_q_heads * cfg.head_dim, cfg.n_kv_heads * cfg.head_dim
    params, nf4 = {}, {}

    def dense(name, shape, std=0.02, quant=False):
        w = torch.randn(*shape, generator=g) * std
        if quant and quantize_base:
            packed, absmax = nf4_quantize(w.numpy())
            absmax = torch.from_numpy(absmax).to(torch.bfloat16).float().numpy()  # bf16-representable scales
            nf4[name] = (packed, absmax)
            w = nf4_dequantize(packed, absmax, shape).float()
        else:
            w = w.to(torch.bfloat16).float()
        params[name] = w.to(device)

    dense("embed", (V, H))
    dense("lm_head", (V, H))
    params["final_norm"] = (1 + 0.1 * torch.randn(H, generator=g)).to(torch.bfloat16).float().to(device)
    shapes = cfg.module_shapes()
    wname = {"q": "wq", "k": "wk", "v": "wv", "o": "wo", "gate": "wg", "up": "wu", "down": "wd"}
    for i in range(cfg.n_layers):
        for m in LORA_MODULES:
            fin, fout = shapes[m]
            dense(f"l{i}.{wname[m]}", (fout, fin), quant=True)
            bound = 1.0 / math.sqrt(fin)  # kaiming_uniform(a=sqrt(5)) on [r, in] -> U(-1/sqrt(in), 1/sqrt(in))
            A = (torch.rand(cfg.lora_r, fin, generator=g) * 2 - 1) * bound
            Bm = torch.randn(fout, cfg.lora_r, generator=g) * lora_b_std
            params[f"l{i}.{m}.A"] = A.to(torch.bfloat16).float().to(device).requires_grad_(True)
            params[f"l{i}.{m}.B"] = Bm.to(torch.bfloat16).float().to(device).requires_grad_(True)
        for b, n in (("bq", qd), ("bk", kd), ("bv", kd)):
            params[f"l{i}.{b}"] = (torch.randn(n, generator=g) * 0.02).to(torch.bfloat16).float().to(device)
        params[f"l{i}.ln1"] = (1 + 0.1 * torch.randn(H, generator=g)).to(torch.bfloat16).float().to(device)
        params[f"l{i}.ln2"] = (1 + 0.1 * torch.randn(H, generator=g)).to(torch.bfloat16).float().to(device)
    return params, nf4


def params_digest(params, nf4):
    """sha256 over every parameter (fp32 bytes) and NF4 code / scale array of make_params' output, in name order."""
    h = hashlib.sha256()
    for k in sorted(params):
        h.update(k.encode())
        h.update(params[k].detach().cpu().float().numpy().tobytes())
    for k in sorted(nf4):
        h.update(k.encode())
        h.update(np.ascontiguousarray(nf4[k][0]).tobytes())
        h.update(np.ascontiguousarray(nf4[k][1]).tobytes())
    return h.hexdigest()


def make_batch(cfg: OracleConfig, n_seq, P, T, seed=0, ragged=True, group_size=None, learner="grpo"):
    """Synthetic (prompt ids, answer ids, rewards) following SURVEY.md §8d: ids ~ U[1, V), ragged
    lengths (prompt ~ U[P/2, P], completion ~ U[T/4, T]) or full length; rewards = format in
    {0, .1, .2} w.p. (.5,.3,.2) + accuracy ~ Bernoulli(.25), turned into advantages per group (degenerate
    groups are redrawn)."""
    rng = np.random.default_rng(seed)
    prompts, answers = [], []
    for _ in range(n_seq):
        pl = int(rng.integers(max(1, P // 2), P + 1)) if ragged else P
        tl = int(rng.integers(max(1, T // 4), T + 1)) if ragged else T
        prompts.append(rng.integers(1, cfg.vocab, size=pl).tolist())
        answers.append(rng.integers(1, cfg.vocab, size=tl).tolist())
    gsz = group_size or n_seq
    rewards = []
    for _ in range(0, n_seq, gsz):
        while True:
            fmt = rng.choice([0.0, 0.1, 0.2], size=gsz, p=[0.5, 0.3, 0.2])
            acc = (rng.random(gsz) < 0.25).astype(np.float64)
            br = np.stack([fmt, acc], -1)
            if np.std(br.sum(1)) > 0:
                break
        vals, base = group_advantages(br, learner)
        rewards.extend((vals if learner == "grpo" else vals - base).tolist())
    return prompts, answers, np.asarray(rewards[:n_seq], dtype=np.float64)
