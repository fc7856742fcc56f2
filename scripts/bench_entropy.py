"""Cost of the per-token entropy in G7: the plain log-prob kernel (b200rl_logprob_slots) and its entropy variant
(b200rl_logprob_entropy, bonus gradient on) timed alternately in one process on the same logits.

R = 8192 rows x V = 152064 (Qwen2.5 vocabulary) bf16 = 2.5 GB of logits, more than L2 holds, so every pass streams
from HBM.  Two modes: scoring only (reads R*V*2 bytes) and write-grad (reads and overwrites them in place:
2*R*V*2 bytes).  CUDA events around `iters` back-to-back launches, after warm-ups; the plain and entropy kernels
alternate for `rounds` rounds and the median per-launch time of each is reported.

Usage: python scripts/bench_entropy.py --out DIR   (writes DIR/bench_entropy.json and prints it)
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def card():
    """Name and power limit of GPU 0, read in the same run as the measurement."""
    info = {"name": torch.cuda.get_device_name(0)}
    try:
        out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        name, power, sm = [x.strip() for x in out.split(",")]
        info.update(smi_name=name, power_limit=power, max_sm_clock=sm)
    except Exception as e:   # noqa: BLE001  (reported, not hidden)
        info["power_limit"] = f"unavailable ({e})"
    return info


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rows", type=int, default=8192)
    ap.add_argument("--vocab", type=int, default=152064)
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=7)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--out", required=True)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_entropy needs a CUDA device")
    from distrl_llm_b200._capi import check, lib, ptr, stream
    dev = torch.device("cuda:0")
    R, V = a.rows, a.vocab
    T = 512
    Bm = R // T
    g = torch.Generator(device=dev).manual_seed(0)
    logits = (torch.randn(R, V, generator=g, device=dev) * 3).to(torch.bfloat16)
    targets = torch.randint(0, V, (R,), generator=g, device=dev, dtype=torch.int32)
    coef = torch.full((R,), -1e-4, device=dev)
    mask = torch.ones(Bm, T, device=dev, dtype=torch.int32)
    lens = torch.full((Bm,), T, device=dev, dtype=torch.int32)
    lp = torch.empty(R, device=dev)
    ent = torch.empty(R, device=dev)

    def plain(wg):
        check(lib().b200rl_logprob_slots(ptr(logits), V, ptr(targets), ptr(coef), None, None, None, 0.0, ptr(lp), R, V, wg,
                                         None, stream()), "logprob_slots")

    def entropy(wg):
        check(lib().b200rl_logprob_entropy(ptr(logits), V, ptr(targets), ptr(coef), None, None, None, 0.0, ptr(lp), R, V, wg,
                                           None, ptr(mask), ptr(lens), Bm, T, 1, 0.01, ptr(ent), stream()), "logprob_entropy")

    def timed(fn, wg):
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        for _ in range(a.iters):
            fn(wg)
        e.record()
        e.synchronize()
        return s.elapsed_time(e) / a.iters

    result = {"card": card(), "rows": R, "vocab": V, "iters": a.iters, "rounds": a.rounds,
              "logits_bytes": R * V * 2, "l2_note": "2.5 GB of logits > 126 MB L2: every pass streams from HBM"}
    for mode, wg, nbytes in (("score", 0, R * V * 2), ("write_grad", 1, 2 * R * V * 2)):
        for _ in range(a.warmup):
            plain(wg)
            entropy(wg)
        torch.cuda.synchronize()
        tp, te = [], []
        for _ in range(a.rounds):
            tp.append(timed(plain, wg))
            te.append(timed(entropy, wg))
        mp, me = statistics.median(tp), statistics.median(te)
        result[mode] = {"bytes": nbytes, "plain_ms": mp, "entropy_ms": me, "ratio": me / mp,
                        "plain_GBps": nbytes / mp / 1e6, "entropy_GBps": nbytes / me / 1e6,
                        "plain_ms_all": tp, "entropy_ms_all": te}
    os.makedirs(a.out, exist_ok=True)
    with open(os.path.join(a.out, "bench_entropy.json"), "w") as f:
        json.dump(result, f, indent=1)
    print(json.dumps(result))


if __name__ == "__main__":
    main()
