#!/usr/bin/env python
"""bench.py — learner tokens processed/sec (GRPO step, Qwen2.5-7B LoRA) on B200.

Contract: python bench.py --gpus N --steps K --warmup W [--impl reference] [--config cfg2|cfg3|cfg4|cfg5]
  [--dump-outputs DIR]  (N > 1: launched by torch.distributed.run, one rank per GPU).

Workloads (BASELINE.json configs; SURVEY.md 8d):
  cfg2 (default, the headline): GRPO learner, Qwen2.5-7B-shaped random-init NF4 base + rank-16 LoRA, group_size 8,
        64 completions of length 512 (P = 350, micro-batch 8 -> 8 reference micro-batches) PER GPU (weak scaling).
  cfg3: 256 completions of length 1024 = 16 problems x 16 candidates, split evenly over the N learners like the
        reference's Trainer (distributed_trainer.py:310-322); quoted at N = 2 (strong scaling in N).
  cfg4: 1024 sampled completions of length 2048 = 4 problems x 256 candidates; group advantages on all 256 and the
        top-k = 128 subselect per problem through the G9 kernel (distributed_trainer.py:262-294) -> 512 sequences scored,
        split evenly over the N learners; quoted at N = 4.
  cfg5: full pipeline (stub generators -> rewards -> advantages -> learners -> adapter hand-off), trainer steps/s:
        `python -m distrl_llm_b200.train_distributed --bench` prints that line; see there.
A "step" = one learner update: zero_grad, the reference micro-batches (forward, fused log-prob/loss, backward into LoRA
grads) as model passes of --fuse_microbatches micro-batches each (gradient accumulation is linear, identical result) in
the packed shared-prompt layout, (P2P reduce +) Adam on the LoRA parameters, refresh of the bf16 LoRA operands.
  value  : completion tokens scored+updated / s with the batch already resident in HBM
  e2e    : same through the reference-shaped public API (GRPOLearner.train(candidates) / compute_gradients +
           apply_merged_gradients) with HOST token-id lists: CPU padding + packing, pinned H2D copies, D2H of the loss
           (cfg3/cfg4: plus the advantage / top-k kernel and the learner split) inside the timed region
  N > 1  : gradient mean + Adam through the one-shot P2P reduce kernel over NVLink; time = max over ranks; after the
           timed region the ranks' parameters are checked for bit-identity and against NCCL-mean + Adam ("exchange").
--impl reference: the reference learner's CPU path (the pinned torch oracle port of its code on all host cores) timed on
bounded samples of the same workload (one 8-sequence micro-batch through 1/2/3-layer full-width slices, one slice per
step) and extrapolated to 28 layers x n micro-batches; see run_reference().
--impl torch_gpu (optional comparator, SURVEY.md 8d): the same oracle port run on ONE B200 in dense bf16 autocast.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

CATS = ["gemm", "gemm_lora_skinny", "gemm_dw", "nf4_dequant", "attn_fwd", "attn_bwd", "row_kernels", "logprob", "misc"]
METRIC = "learner tokens processed/sec (GRPO step, Qwen2.5-7B LoRA)"
UNIT = "completion tokens/s"

# name -> (problems, candidates per problem, top-k, T, scaling, quoted at N)
PRESETS = {
    "cfg2": dict(n_prob=8, cand=8, topk=8, T=512, scaling="weak", quoted_n=1),
    "cfg3": dict(n_prob=16, cand=16, topk=16, T=1024, scaling="strong", quoted_n=2),
    "cfg4": dict(n_prob=4, cand=256, topk=128, T=2048, scaling="strong", quoted_n=4),
}


def workload(args):
    return dict(n_seq=args.seqs, P=args.prompt_len, T=args.new_tokens, B=args.micro_batch, group=args.group_size,
                rank=args.lora_rank)


# ---------------------------------------------------------------------------------------------------
# clocks sampler (B200_PROFILING.md "clocks DURING the timed region")
# ---------------------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        self.proc = None
        self.lines = []
        self.index = index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for ln in self.proc.stdout:
            self.lines.append(ln.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1]))
            except ValueError:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[3:7]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        busy = [s for s in sm if s > 0]
        return {"sm_mhz": float(np.median(busy)) if busy else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ---------------------------------------------------------------------------------------------------
# algorithmic work (SURVEY.md 8d)
# ---------------------------------------------------------------------------------------------------
P_LAYERS, P_LM = 6_525_288_448, 544_997_376


def flops_per_sequence(P, T, r=16):
    """Reference layout: every (prompt, completion) pair is its own P+T row block; lm_head only at the T scored rows."""
    L = P + T
    p_lora = r * 90_112 * 28
    return L * (4 * P_LAYERS + 6 * p_lora) + T * 4 * P_LM + 3 * 28 * 2 * L * L * 3584


def flops_packed_step(n_seq, group, P, T, r=16):
    """Packed shared-prompt layout: the prompt rows of a group are computed once (identical result).  Rows through the
    layer stack = G*P + n*T; attention pairs are causal-exact: a prompt row p sees p+1 keys, completion token t sees
    P+t+1; attention cost 4*3584 FLOP per (query, key) pair per layer forward, x3 for forward + backward (survey)."""
    G = n_seq // group
    p_lora = r * 90_112 * 28
    rows = G * P + n_seq * T
    pairs = G * P * (P + 1) / 2 + n_seq * (T * P + T * (T + 1) / 2)
    return rows * (4 * P_LAYERS + 6 * p_lora) + n_seq * T * 4 * P_LM + 3 * 28 * 4 * 3584 * pairs


def host_threads():
    """All the host cores the CPU arm can use: torchrun exports OMP_NUM_THREADS=1, which would silently turn the
    reference arm into a single-thread run (measured 3.3 instead of 12.9 tok/s).  One thread per physical core."""
    forced = int(os.environ.get("B200RL_CPU_THREADS", "0"))
    return forced if forced > 0 else max(1, (os.cpu_count() or 2) // 2)


# ---------------------------------------------------------------------------------------------------
# CPU path (oracle port of the reference learner) on bounded samples
# ---------------------------------------------------------------------------------------------------
class CpuArm:
    """The reference learner's math (oracle/learner_oracle.py = pinned restatement of distributed_actor.py:215-261,
    :440-493) on the host cores, for ONE full micro-batch (B sequences x (P+T) tokens, all P+T positions through the
    lm_head like the reference, :241-243) through an nl-layer full-width, full-vocab slice of the model.
    Arithmetic: the reference runs its hot loop under torch.autocast(bf16) (:462); on CPUs with AMX that is the fast
    path, elsewhere fp32 is faster — a 2048^3 matmul probe picks the faster of the two so the arm is timed at its best.
    Gradient checkpointing (helper.py:42, +1 forward per layer in the reference) is OFF in this port: favours the arm."""

    def __init__(self, w, threads, n_rows=None, max_layers=3, dtype="auto"):
        from oracle import learner_oracle as lo
        self.lo = lo
        torch.set_num_threads(threads)
        self.threads = torch.get_num_threads()
        self.w = w
        self.B = n_rows or w["B"]
        if dtype == "auto":
            dtype = self._probe()
        self.dtype = {"bf16": torch.bfloat16, "fp32": torch.float32}[dtype]
        self.dtype_name = dtype
        # B200RL_CPU_ARM_SHAPE="vocab,hidden,inter,q_heads,kv_heads": debug / CI only (tests/test_host_logic.py exercises the
        # arm's bookkeeping on a tiny model); the benchmark always runs the full Qwen2.5-7B width and vocabulary
        shape = [int(x) for x in os.environ.get("B200RL_CPU_ARM_SHAPE", "152064,3584,18944,28,4").split(",")]
        mk = lambda nl: lo.OracleConfig(vocab=shape[0], hidden=shape[1], inter=shape[2], n_layers=nl, n_q_heads=shape[3],
                                        n_kv_heads=shape[4], head_dim=shape[1] // shape[3], lora_r=w["rank"], lora_alpha=16)
        cfg = mk(max_layers)
        params, _ = lo.make_params(cfg, seed=1, quantize_base=False)
        # parameters are converted ONCE (the reference's model already holds its weights in the compute dtype)
        self.params = {k: (v.detach().to(self.dtype).requires_grad_(v.requires_grad) if v.dtype.is_floating_point else v)
                       for k, v in params.items()}
        self.cfgs = {nl: mk(nl) for nl in range(1, max_layers + 1)}
        prompts, answers, rewards = lo.make_batch(self.cfgs[1], self.B, w["P"], w["T"], seed=2, ragged=False,
                                                  group_size=self.B, learner="grpo")
        self.batch = lo.pad_batch(prompts, answers, w["P"], w["T"]) + (rewards,)
        self.samples = {}   # nl -> [seconds]

    @staticmethod
    def _probe():
        """bf16 when the host has a bf16 matrix unit (AMX-BF16 / AVX512-BF16: then it is the faster arm, measured 14.8 s vs
        26.0 s per 1-layer sample on this pool's 64-core hosts), else fp32.  Decided from the CPU flags, not from a timing
        probe (a probe taken while the GPU arm's threads are still winding down picked fp32 once)."""
        try:
            flags = open("/proc/cpuinfo").read()
            if "amx_bf16" in flags or "avx512_bf16" in flags:
                return "bf16"
        except OSError:
            pass
        return "fp32"

    def sample(self, nl):
        ids, am, ansm, rewards = self.batch
        t0 = time.perf_counter()
        self.lo.compute_gradients(self.params, self.cfgs[nl], ids, am, ansm, rewards, self.w["P"], self.B, "grpo",
                                  dtype=self.dtype)
        dt = time.perf_counter() - t0
        self.samples.setdefault(nl, []).append(dt)
        return dt

    def extrapolate(self):
        """Least-squares t = head + per_layer * nl over the samples -> seconds per full learner step, tokens/s."""
        xs = np.array([nl for nl, v in self.samples.items() for _ in v], dtype=np.float64)
        ys = np.array([t for v in self.samples.values() for t in v], dtype=np.float64)
        if len(set(xs.tolist())) >= 2:
            per_layer, head = np.polyfit(xs, ys, 1)
        else:   # a single layer count: attribute everything to the layers (upper bound on the arm's speed is kept honest below)
            per_layer, head = ys.mean() / xs.mean(), 0.0
        per_layer, head = max(per_layer, 1e-9), max(head, 0.0)
        t_mb = head + 28 * per_layer
        w = self.w
        nb = (w["n_seq"] + w["B"] - 1) // w["B"]
        t_step = t_mb * nb * (w["B"] / self.B)
        tok_s = w["n_seq"] * w["T"] / t_step
        desc = (f"oracle port of the reference learner ({self.dtype_name} on {self.threads} host threads, no gradient "
                f"checkpointing): one full micro-batch ({self.B}x{w['P'] + w['T']} tokens, lm_head on all positions) fwd+bwd "
                f"through full-width/full-vocab slices of "
                + ", ".join(f"{nl} layer(s): {np.mean(v):.1f}s x{len(v)}" for nl, v in sorted(self.samples.items()))
                + f"; fit head {head:.1f}s + {per_layer:.2f}s/layer, extrapolated to 28 layers x {nb} micro-batches")
        return tok_s, desc, t_step


DUMP_SAMPLE = 1 << 22   # positions kept per flat LoRA-sized buffer: 3 x 16 MB of float32


def step_outputs(pol):
    """What the last learner step hands its caller: the loss (sum over the micro-batches, float64) and the updated adapter,
    plus the Adam moments, which carry that step's gradient (the optimizer step zeroes the gradient buffer itself).  The
    flat buffers hold ~40M values at the Qwen2.5-7B shape, so a fixed sample of DUMP_SAMPLE positions (seed 0) is kept."""
    n = pol.lora_flat.numel()
    idx = torch.randperm(n, generator=torch.Generator().manual_seed(0))[:DUMP_SAMPLE].sort().values.to(pol.device)
    out = {"loss": pol.loss_accum, "lora": pol.lora_flat[idx], "adam_m": pol.adam_m[idx], "adam_v": pol.adam_v[idx]}
    return {k: v.cpu().numpy() for k, v in out.items()}


def config_dict(args):
    preset = PRESETS.get(args.config)
    if args.config == "cfg2":
        what = (f"group_size={args.group_size}, {args.seqs} completions len={args.new_tokens} per GPU "
                f"(P={args.prompt_len}, micro-batch {args.micro_batch})")
        gb = args.seqs * args.gpus
    else:
        kept = preset["n_prob"] * preset["topk"]
        what = (f"{preset['n_prob']} problems x {preset['cand']} sampled completions len={args.new_tokens}"
                + (f", group advantages on all {preset['cand']} then top-k={preset['topk']} per problem (G9 kernel) -> {kept} sequences scored"
                   if preset["topk"] < preset["cand"] else f" = {kept} sequences")
                + f", split evenly over {args.gpus} learner(s) like distributed_trainer.py:310-322 (P={args.prompt_len}, micro-batch {args.micro_batch})")
        gb = kept
    return {"workload": f"{args.config}: GRPO learner step, Qwen2.5-7B-shaped random-init NF4 base + rank-{args.lora_rank} LoRA, " + what
                        + (", RAGGED lengths (prompt ~ U[P/2,P], completion ~ U[T/4,T]); value counts real completion tokens" if getattr(args, "ragged", False) else ""),
            "global_batch": gb, "seq_len": args.prompt_len + args.new_tokens,
            "parallelism": f"dp{args.gpus}" if args.gpus > 1 else "single learner",
            "passes": f"{getattr(args, 'fuse_microbatches', 1)} reference micro-batches of {args.micro_batch} per model pass (gradient accumulation is linear: identical result)",
            "layout": "classic [B, P+T] rows" if getattr(args, "no_share_prompts", False) else
                      "packed shared-prompt rows (each group's prompt processed once; identical gradients)",
            "weights": {"auto": "NF4 at the boundary; resident bf16 image of the dequantised base (15.2 GB) inside",
                        "cache": "NF4 at the boundary; resident bf16 image of the dequantised base (15.2 GB) inside",
                        "scratch": "NF4 dequantised into a scratch before each GEMM",
                        "inkernel": "NF4 dequantised inside the GEMM mainloop (no bf16 copy of the base)"}[getattr(args, "weights", "auto")],
            "l2": "per-step activations and weights (>30 GB) far exceed the 126 MB L2; no flush needed"}


def run_reference(args, rank, world):
    """Reference arm: every step times ONE bounded sample (a full micro-batch through an nl-layer slice, nl cycling over
    1,2,3), `ms_per_step` is the measured time of those samples, `value` the tokens/s extrapolated from the fit over all
    timed samples to the full 28-layer, n-micro-batch step of the SAME config as the b200 arm."""
    w = workload(args)
    if rank != 0:
        return
    arm = CpuArm(w, host_threads(), n_rows=args.cpu_rows, max_layers=3, dtype=args.cpu_dtype)
    for i in range(args.warmup):
        arm.sample(1 + i % 3)
    arm.samples = {}
    t_all = []
    for i in range(args.steps):
        t_all.append(arm.sample(1 + i % 3))
    tok, desc, t_step = arm.extrapolate()
    line = {"impl": "reference", "metric": METRIC, "value": tok, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": float(np.mean(t_all)) * 1e3, "higher_is_better": True,
            "scaling": "weak" if args.config == "cfg2" else "strong", "vs_baseline": None,
            "dtype": "bf16" if arm.dtype_name == "bf16" else "f32", "data": "synthetic", "config": config_dict(args),
            "step_is": "one bounded sample (a full micro-batch through a 1/2/3-layer slice); value is extrapolated, see cpu_baseline.sample",
            "extrapolated_ms_per_full_step": t_step * 1e3,
            "cpu_baseline": {"value": tok, "unit": UNIT, "cores": arm.threads, "kind": "port", "sample": desc},
            "e2e": {"value": tok, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


def run_torch_gpu(args):
    """Optional comparator (SURVEY.md 8d "torch-GPU"): the oracle port of the reference learner, unchanged, on ONE B200
    with dense bf16 weights under torch autocast — what the reference's torch path would do on this GPU without
    Unsloth/bnb (not installable here).  Full 28 layers, the reference's padded [B, P+T] layout, lm_head on all
    positions, eager attention, no gradient checkpointing (fits in 180 GB)."""
    from oracle import learner_oracle as lo
    w = workload(args)
    dev = torch.device("cuda", 0)
    cfg = lo.OracleConfig(vocab=152064, hidden=3584, inter=18944, n_layers=args.layers, n_q_heads=28, n_kv_heads=4,
                          head_dim=128, lora_r=w["rank"], lora_alpha=16)
    g = torch.Generator(device=dev).manual_seed(0)
    params = {}

    def dense(name, shape, std=0.02, grad=False):
        params[name] = (torch.randn(*shape, generator=g, device=dev) * std).to(torch.bfloat16).requires_grad_(grad)
    dense("embed", (cfg.vocab, cfg.hidden)); dense("lm_head", (cfg.vocab, cfg.hidden))
    params["final_norm"] = torch.ones(cfg.hidden, device=dev, dtype=torch.bfloat16)
    wname = {"q": "wq", "k": "wk", "v": "wv", "o": "wo", "gate": "wg", "up": "wu", "down": "wd"}
    for i in range(cfg.n_layers):
        for m, (fin, fout) in cfg.module_shapes().items():
            dense(f"l{i}.{wname[m]}", (fout, fin))
            params[f"l{i}.{m}.A"] = ((torch.rand(cfg.lora_r, fin, generator=g, device=dev) * 2 - 1) * fin ** -0.5).requires_grad_(True)
            params[f"l{i}.{m}.B"] = (torch.randn(fout, cfg.lora_r, generator=g, device=dev) * 0.01).requires_grad_(True)
        for b, n in (("bq", cfg.n_q_heads * cfg.head_dim), ("bk", cfg.n_kv_heads * cfg.head_dim), ("bv", cfg.n_kv_heads * cfg.head_dim)):
            dense(f"l{i}.{b}", (n,))
        params[f"l{i}.ln1"] = torch.ones(cfg.hidden, device=dev, dtype=torch.bfloat16)
        params[f"l{i}.ln2"] = torch.ones(cfg.hidden, device=dev, dtype=torch.bfloat16)
    prompts, answers, rewards = lo.make_batch(cfg, w["n_seq"], w["P"], w["T"], seed=2, ragged=False, group_size=w["group"], learner="grpo")
    ids, am, ansm = (t.to(dev) for t in lo.pad_batch(prompts, answers, w["P"], w["T"]))
    lora = [params[n] for n in lo.lora_names(cfg)]
    opt = torch.optim.Adam(lora, lr=2e-5)

    def step():
        lo.compute_gradients(params, cfg, ids, am, ansm, rewards, w["P"], w["B"], "grpo", dtype=torch.bfloat16)
        opt.step()
    for _ in range(args.warmup):
        step()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        step()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / args.steps
    tok = w["n_seq"] * w["T"] / (ms / 1e3)
    print(json.dumps({"impl": "torch_gpu", "metric": METRIC, "value": tok, "unit": UNIT, "n_gpus": 1, "steps": args.steps,
                      "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "dtype": "bf16", "data": "synthetic",
                      "config": config_dict(args), "what": "oracle port of the reference learner (torch eager, dense bf16 weights, "
                      "padded [B,P+T] layout, lm_head on all positions, no checkpointing) on one B200 — optional comparator, "
                      "not the reference arm", "max_mem_gb": torch.cuda.max_memory_allocated() / 2 ** 30}), flush=True)


# ---------------------------------------------------------------------------------------------------
# synthetic trainer-side payload for cfg3 / cfg4: raw rewards -> (G9 kernel) advantages + top-k -> merge -> split
# ---------------------------------------------------------------------------------------------------
def raw_candidates(vocab, n_prob, cand, P, T, seed):
    """The reference's `candidates` payload BEFORE the advantage block (distributed_trainer.py:252-261): per problem `cand`
    completions (token-id lists) and rewards [cand, 2] = (format, accuracy), SURVEY.md 8d distribution.  Groups whose
    normalised advantages would contain an exact 0 are redrawn (quirk Q1 would skip those micro-batches)."""
    rng = np.random.default_rng(seed)
    c = {"answers": [], "problem": [], "rewards": []}
    for _ in range(n_prob):
        prompt = rng.integers(1, vocab, size=P).tolist()
        c["problem"].append([prompt] * cand)
        ans = rng.integers(1, vocab, size=(cand, T))
        c["answers"].append([a.tolist() for a in ans])
        while True:
            fmt = rng.choice([0.0, 0.1, 0.2], size=cand, p=[0.5, 0.3, 0.2])
            acc = (rng.random(cand) < 0.25).astype(np.float64)
            s = fmt + acc
            if np.std(s) > 0 and np.all((s - np.mean(s)) / (np.std(s) + 1e-8) != 0):
                break
        c["rewards"].append(np.stack([fmt, acc], -1))
    return [c]


# ---------------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference", "torch_gpu"])
    ap.add_argument("--config", default="cfg2", choices=["cfg2", "cfg3", "cfg4"], help="BASELINE.json config (cfg2 = headline)")
    ap.add_argument("--seqs", type=int, default=64, help="cfg2: sequences per GPU")
    ap.add_argument("--new_tokens", type=int, default=None)
    ap.add_argument("--prompt_len", type=int, default=350)
    ap.add_argument("--micro_batch", type=int, default=8)
    ap.add_argument("--group_size", type=int, default=8)
    ap.add_argument("--lora_rank", type=int, default=16)
    ap.add_argument("--layers", type=int, default=28, help="debug only: anything but 28 is not the benchmark")
    ap.add_argument("--cpu_rows", type=int, default=8, help="sequences in the CPU sample micro-batch (8 = a full reference micro-batch)")
    ap.add_argument("--cpu_dtype", default="auto", choices=["auto", "bf16", "fp32"])
    ap.add_argument("--no_cpu_baseline", action="store_true")
    ap.add_argument("--fuse_microbatches", type=int, default=2, help="reference micro-batches per model pass (identical gradients; 1 = one pass per micro-batch like the reference)")
    ap.add_argument("--ragged", action="store_true", help="cfg2 only: ragged synthetic lengths (prompt ~ U[P/2,P], completion ~ U[T/4,T]); value counts REAL completion tokens")
    ap.add_argument("--no_share_prompts", action="store_true", help="classic [B, P+T] layout (every prompt recomputed per completion)")
    ap.add_argument("--weights", default="auto", choices=["auto", "cache", "scratch", "inkernel"],
                    help="NF4 base: resident bf16 cache (auto/cache), dequant into a scratch before each GEMM, or inside the GEMM mainloop")
    ap.add_argument("--lean", action="store_true", help="long configs (cfg4): one e2e warm-up, no repeat of the device timing, one exchange-timing step")
    ap.add_argument("--no_verify_exchange", action="store_true", help="N > 1: skip the post-run parameter identity / NCCL cross-check")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step computed (see step_outputs) as DIR/<name>.npy; --impl b200, one GPU")
    args = ap.parse_args()
    if args.dump_outputs and (args.impl != "b200" or args.gpus != 1):
        ap.error("--dump-outputs needs --impl b200 and --gpus 1")
    preset = PRESETS[args.config]
    if args.new_tokens is None:
        args.new_tokens = preset["T"]
    if args.config != "cfg2":
        args.seqs = preset["n_prob"] * preset["topk"]     # global kept sequences (split over the learners)
        args.group_size = preset["topk"]
    if args.warmup < 3 and args.impl == "b200":
        args.warmup = 3  # timing rule: W >= 3

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    if args.impl == "torch_gpu":
        if rank == 0:
            run_torch_gpu(args)
        return
    assert world == args.gpus, f"--gpus {args.gpus} but WORLD_SIZE={world} (launch with torch.distributed.run)"

    import torch.distributed as dist
    from distrl_llm_b200 import _capi, ops, trainer_prep
    from distrl_llm_b200.learner import GRPOLearner, IdTokenizer
    from distrl_llm_b200.policy import LMConfig, Policy
    from distrl_llm_b200.p2p import P2PGroup

    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        # stdout carries exactly one JSON line: NCCL prints its version banner to stdout when the first communicator
        # is created (NCCL_DEBUG=VERSION/WARN in this image), so fd 1 points at stderr until that has happened
        sys.stdout.flush()
        _saved_fd = os.dup(1)
        os.dup2(2, 1)
        try:
            dist.init_process_group("nccl", device_id=dev)
            dist.barrier()
            torch.cuda.synchronize()
        finally:
            sys.stdout.flush()
            os.dup2(_saved_fd, 1)
            os.close(_saved_fd)
    w = workload(args)
    cfg = LMConfig.qwen25_7b(lora_r=args.lora_rank)
    cfg.n_layers = args.layers
    P, T, B = w["P"], w["T"], w["B"]
    group = None
    kw = {}
    FK = max(1, args.fuse_microbatches)
    try:   # long-sequence configs (T = 2048: 38k rows per fused pass) may not leave room for 2 micro-batches per pass
        from distrl_llm_b200.policy import largest_pass_that_fits
        free_b, _ = torch.cuda.mem_get_info(dev)
        FK = largest_pass_that_fits(cfg, B, P, T, FK, free_b, reserve_bytes=24 << 30)   # NF4 + bf16 cache + lm_head/embed
        args.fuse_microbatches = FK
    except Exception as e:  # sizing is best-effort; the allocation itself still fails loudly
        print(f"[bench] pass sizing skipped: {e}", file=sys.stderr)
    if world > 1:
        group, kw = P2PGroup.from_torch_distributed(cfg, FK * B, P, T, dev)
    kw["cache_weights"] = {"auto": "auto", "cache": True, "scratch": False, "inkernel": "inkernel"}[args.weights]
    pol = Policy.random_init(cfg, dev, FK * B, P, T, seed=1234, **kw)   # same base + LoRA on every learner
    if group is not None:
        group.attach(pol)
    config = {"train_batch_size": B, "max_new_tokens": T, "max_prompt_tokens": P, "lr": 2e-5}
    learner = GRPOLearner(pol, IdTokenizer(), config, gpu_id=local)
    if group is not None:
        learner.enable_p2p(group)

    # ---- this learner's batch --------------------------------------------------------------------------------
    if args.config == "cfg2":
        # SURVEY.md 8d: ids ~ U[1,V), full-length prompts/completions, rewards -> group advantages; every learner its own
        N = w["n_seq"]
        cands, flat = trainer_prep.synthetic_candidates(cfg.vocab, N, P, T, args.group_size, seed=1234 + rank, ragged=args.ragged)
        prompts, answers, adv = flat
        raw = None
        tokens_global = (N * T if not args.ragged else int(sum(len(a) for a in answers))) * world
    else:
        # the Trainer's side of the step (distributed_trainer.py:262-342), identical on every rank (same seed): raw rewards
        # -> G9 kernel (advantages on all candidates, top-k) -> merge -> even split -> this rank's chunk
        raw = raw_candidates(cfg.vocab, preset["n_prob"], preset["cand"], P, T, seed=4321)

        def trainer_side():
            c = [dict(problem=raw[0]["problem"], answers=raw[0]["answers"], rewards=[r.copy() for r in raw[0]["rewards"]])]
            c = trainer_prep.apply_advantages_and_topk(c, "grpo", preset["topk"], dev)
            pr, an, rw = trainer_prep.merge_candidates(c)
            return trainer_prep.split_for_learners(pr, an, rw, world)[rank]
        prompts, answers, adv = trainer_side()
        adv = np.asarray(adv, dtype=np.float64)
        N = len(prompts)
        cands = None
        tokens_global = preset["n_prob"] * preset["topk"] * T
    assert np.all(np.asarray(adv) != 0), "synthetic advantages must be non-zero (quirk Q1 would skip work)"
    nb = (N + B - 1) // B
    # device-resident copy for the `value` measurement
    ids_h, am_h, ansm_h = learner._encode(prompts, answers)
    d_ids, d_am, d_ansm = (None, None, None)
    d_adv = torch.from_numpy(np.asarray(adv, dtype=np.float64)).to(dev)

    share = learner.share_prompts and not args.no_share_prompts
    learner.share_prompts = share
    assert learner.fuse_microbatches == FK
    if not share:
        d_ids, d_am, d_ansm = ids_h.to(dev), am_h.to(dev), ansm_h.to(dev)
    # passes of FK reference micro-batches each (learner.compute_loss does the same planning on the e2e path)
    bounds = [(i * B, min((i + 1) * B, N)) for i in range(nb)]
    passes, cur = [], []
    for (s_, e_) in bounds:
        if e_ - s_ == B and FK > 1:
            cur.append((s_, e_))
            if len(cur) == FK:
                passes.append(cur); cur = []
        else:
            passes.append([(s_, e_)])
    if cur:
        passes.append(cur)
    pass_rng = [(g[0][0], g[-1][1], len(g)) for g in passes]      # contiguous because only full micro-batches fuse
    d_adv_k = [d_adv[s_:e_] * float(k) for (s_, e_, k) in pass_rng]
    packed = []
    rows_per_step = 0
    if share:  # packed shared-prompt layout, device-resident for the `value` measurement
        from distrl_llm_b200 import packing
        for (s_, e_, k) in pass_rng:
            packed.append(packing.PackedDevice(packing.pack_microbatch(ids_h[s_:e_].numpy(), am_h[s_:e_].numpy(), P, T), dev))
            rows_per_step += packed[-1].host.rows
        torch.cuda.synchronize()
    else:
        rows_per_step = N * (P + T)

    ev_pre = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    timing_on = [False]

    def device_step():
        if timing_on[0]:
            ev_pre[0].record()
        pol.zero_grad()
        pol.loss_accum.zero_()
        for i, (s, e, k) in enumerate(pass_rng):
            if share:
                pol.microbatch_packed(packed[i], d_adv_k[i], nb, True, backward=True)
            else:
                pol.microbatch(d_ids[s:e], d_am[s:e], d_ansm[s:e], d_adv_k[i], P, T, nb, True, backward=True)
        if timing_on[0]:
            ev_pre[1].record()
        if group is not None:
            group.reduce_adam_step(pol, learner.lr, 0.0, timing=timing_on[0])
        else:
            pol.optimizer_step(learner.lr)

    def e2e_step():
        if raw is not None:      # cfg3 / cfg4: the trainer-side advantage + top-k kernel and the split are part of the step
            pr, an, rw = trainer_side()
        else:
            pr, an, rw = prompts, answers, adv
        if group is not None:
            loss = learner.compute_loss(pr, an, rw)
            learner.apply_merged_gradients()
        elif cands is not None:
            loss = learner.train(cands)
        else:
            loss = learner.compute_loss(pr, an, rw)
            pol.optimizer_step(learner.lr)
        return loss

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps, sample_clocks=False):
        sampler = ClockSampler(local) if sample_clocks and rank == 0 else None
        barrier()
        if sampler:
            sampler.start()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        l0 = _capi.lib().b200rl_launch_count()
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        barrier()
        ms = e0.elapsed_time(e1)
        clocks = sampler.stop() if sampler else None
        launches = _capi.lib().b200rl_launch_count() - l0
        if world > 1:
            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = t.item()
        return ms / steps, clocks, launches

    for _ in range(args.warmup):
        device_step()
    if os.environ.get("B200RL_PROFILE_ONE_STEP"):
        # ncu --profile-from-start off: exactly one learner step between cudaProfilerStart/Stop
        torch.cuda.synchronize()
        torch.cuda.profiler.start()
        device_step()
        torch.cuda.synchronize()
        torch.cuda.profiler.stop()
        return
    ms_dev, clocks, launches = timed(device_step, args.steps, sample_clocks=True)
    if args.dump_outputs:   # before the e2e and diagnostic steps below move the adapter on
        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, arr in step_outputs(pol).items():
            np.save(os.path.join(args.dump_outputs, name + ".npy"), arr)
    for _ in range(1 if args.lean else 2):
        e2e_step()
    ms_e2e, _, _ = timed(e2e_step, args.steps)
    ms_dev2 = None
    if not args.lean:
        ms_dev2, _, _ = timed(device_step, args.steps)   # diagnostic: same region without the nvidia-smi sampler

    # ---- N > 1: where the exchange time goes, and is the result right? ---------------------------------------------
    exchange = None
    if group is not None:
        barrier()
        timing_on[0] = True
        comp, waits, reds, refr = [], [], [], []
        for _ in range(1 if args.lean else 3):
            device_step()
            wait_ms, red_ms, refresh_ms = group.exchange_ms()
            comp.append(ev_pre[0].elapsed_time(ev_pre[1])); waits.append(wait_ms); reds.append(red_ms); refr.append(refresh_ms)
        timing_on[0] = False
        mine = torch.tensor([np.median(comp), np.median(waits), np.median(reds), np.median(refr)], device=dev, dtype=torch.float64)
        allr = [torch.zeros_like(mine) for _ in range(world)]
        dist.all_gather(allr, mine)
        allr = torch.stack(allr).cpu().numpy()
        nv_bytes = group.nvlink_bytes_per_step()
        exchange = {"compute_ms_per_rank": [round(float(x), 2) for x in allr[:, 0]],
                    "wait_for_slowest_ms_per_rank": [round(float(x), 3) for x in allr[:, 1]],
                    "reduce_adam_and_closing_barrier_ms": round(float(allr[:, 2].max()), 3),
                    "zero_grad_and_operand_refresh_ms": round(float(allr[:, 3].max()), 3),
                    "nvlink_bytes_per_gpu_per_step": int(nv_bytes),
                    "nvlink_gbs_per_direction": round(nv_bytes / 2 / (float(allr[:, 2].max()) / 1e3) / 1e9, 1),
                    "nvlink_peak_gbs_per_direction": 900.0,
                    "note": "reduce time includes the closing flag barrier; the wait column is rank skew (max-over-ranks compute), not link time"}
        if not args.no_verify_exchange:
            # (1) every learner holds the same parameters, bit for bit
            hi, lo_ = pol.lora_flat.clone(), pol.lora_flat.clone()
            dist.all_reduce(hi, op=dist.ReduceOp.MAX); dist.all_reduce(lo_, op=dist.ReduceOp.MIN)
            identical = bool(torch.equal(hi, lo_))
            # (2) one more step, cross-checked against NCCL mean + the single-learner Adam kernel
            p0, m0, v0 = pol.lora_flat.clone(), pol.adam_m.clone(), pol.adam_v.clone()
            learner.compute_loss(prompts, answers, adv)
            g = pol.lora_grad.clone()
            learner.apply_merged_gradients()
            dist.all_reduce(g, op=dist.ReduceOp.SUM)
            g /= world
            ops.adamw_step(p0, m0, v0, g, pol.opt_step, learner.lr)
            torch.cuda.synchronize()
            group.check()
            # every learner owns the Adam moments of ITS 1/N slice only (the fused kernel updates m, v there and pushes the
            # new parameters to all peers), so the single-learner replay is comparable on the owned slice; bit-identity across
            # ranks (checked above) extends it to the whole buffer
            from distrl_llm_b200.p2p import owned_slice
            lo_i, hi_i = owned_slice(group.numel, world, rank)
            dmax = (p0[lo_i:hi_i] - pol.lora_flat[lo_i:hi_i]).abs().max().reshape(1)
            dist.all_reduce(dmax, op=dist.ReduceOp.MAX)
            diff = float(dmax)
            exchange.update({"params_bit_identical_across_ranks": identical, "max_abs_diff_vs_nccl_mean_adam": diff,
                             "lr": learner.lr})
            assert identical, "learners diverged after the P2P exchange"
            assert diff <= 5e-6, f"P2P reduce+Adam differs from NCCL mean + Adam by {diff}"

    # per-category CUDA-event profile of ONE extra step (same stream; events between consecutive launches)
    import ctypes as C
    _capi.check(_capi.lib().b200rl_model_profile(pol.handle, 1))
    device_step()
    ms_c, wk_c, cnt_c = (C.c_double * 9)(), (C.c_double * 9)(), (C.c_longlong * 9)()
    _capi.check(_capi.lib().b200rl_model_profile_read(pol.handle, ms_c, wk_c, cnt_c))
    _capi.check(_capi.lib().b200rl_model_profile(pol.handle, 0))
    prof = {CATS[i]: {"ms": ms_c[i], "work": wk_c[i], "launches": cnt_c[i]} for i in range(9)}

    value = tokens_global / (ms_dev / 1e3)
    e2e_val = tokens_global / (ms_e2e / 1e3)
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak_tf = peaks.get("bf16_tflops_sustained", 1400.0)
    gemm = prof["gemm"]
    ach_tf = gemm["work"] / (gemm["ms"] / 1e3) / 1e12 if gemm["ms"] > 0 else 0.0
    lscale = args.layers / 28.0 if args.layers != 28 else 1.0
    n_global = tokens_global // T if not args.ragged else w["n_seq"] * world
    ref_flops = flops_per_sequence(P, T, args.lora_rank) * n_global * lscale
    packed_flops = flops_packed_step(n_global, args.group_size, P, T, args.lora_rank) * lscale
    traffic = None
    traffic_src = None
    for name in ("r2_gemm_dram_traffic.json", "r1_gemm_dram_traffic.json"):
        try:  # dram__bytes_read + dram__bytes_write per GEMM launch from the committed ncu --set full capture
            traffic = json.load(open(os.path.join(ROOT, "profiles", name)))["per_launch_traffic_bytes"]
            traffic_src = name
            break
        except Exception:
            pass
    roofline = {"bound": "tensor", "kernel": "gemm_pair_kernel<256> (tcgen05 cta_group::2, base+LoRA mainloop)",
                "achieved": round(ach_tf, 1), "peak": peak_tf, "unit": "TFLOP/s", "frac": round(ach_tf / peak_tf, 4),
                "peak_source": "MEASURED_PEAKS.json bf16_tflops_sustained" if peaks else "fallback 1.4 PF sustained",
                "traffic": traffic, "traffic_unit": f"bytes per GEMM launch (ncu dram read+write, profiles/{traffic_src})",
                "gemm_share_of_step": round(gemm["ms"] / max(sum(p["ms"] for p in prof.values()), 1e-9), 4),
                "avg_launch_ms": round(gemm["ms"] / max(gemm["launches"], 1), 4),
                "flops_per_launch": gemm["work"] / max(gemm["launches"], 1),
                "how": "CUDA events between consecutive launches on the launching stream, one profiled step after the timed region"}
    # whole-step roofline (attention + LoRA-GEMM roofline of north_star): algorithmic FLOPs / measured sustained bf16 peak
    step_roofline = {"algorithmic_flops_reference_layout": ref_flops, "algorithmic_flops_packed_layout": packed_flops,
                     "tok_s_at_sustained_peak_reference_layout": round(tokens_global / (ref_flops / world / (peak_tf * 1e12)), 1),
                     "tok_s_at_sustained_peak_packed_layout": round(tokens_global / (packed_flops / world / (peak_tf * 1e12)), 1),
                     "frac_of_packed_roofline": round(value / (tokens_global / (packed_flops / world / (peak_tf * 1e12))), 4),
                     "frac_of_reference_layout_roofline": round(value / (tokens_global / (ref_flops / world / (peak_tf * 1e12))), 4),
                     "rows_through_the_layers_per_step_per_gpu": int(rows_per_step)}
    if share:
        h2d = int(sum(pk.h2d_bytes for pk in packed) + N * 8)
    else:
        h2d = int(ids_h.numel() * 4 + am_h.numel() * 4 + ansm_h.numel() * 4 + N * 8)
    if raw is not None:
        h2d += int(preset["n_prob"] * preset["cand"] * 2 * 8)     # raw rewards to the G9 kernel
    d2h = 8 if raw is None else 8 + int(preset["n_prob"] * (preset["topk"] * 12 + 8))   # loss (+ top-k indices / values / baselines)
    if rank == 0:
        cpu = None
        if world == 1 and not args.no_cpu_baseline and args.layers == 28:   # rank 0 at N = 1 only (a bounded sample)
            arm = CpuArm(w, host_threads(), n_rows=args.cpu_rows, max_layers=2, dtype=args.cpu_dtype)
            arm.sample(1); arm.sample(2)
            tok_s, desc, _ = arm.extrapolate()
            cpu = {"value": tok_s, "unit": UNIT, "cores": arm.threads, "kind": "port", "sample": desc}
            del arm
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": ms_dev, "higher_is_better": True, "scaling": preset["scaling"], "vs_baseline": None,
                "dtype": "bf16", "data": "synthetic", "config": config_dict(args),
                "e2e": {"value": e2e_val, "unit": UNIT, "ms_per_step": ms_e2e,
                        "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h},
                "ms_per_step_no_sampler": ms_dev2, "gpu_launches": int(launches), "clocks": clocks, "roofline": roofline,
                "step_roofline": step_roofline, "exchange": exchange, "cpu_baseline": cpu,
                "profile_ms": {k: round(v["ms"], 3) for k, v in prof.items()},
                "profile_launches": {k: int(v["launches"]) for k, v in prof.items()}}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
