"""ORACLE — TEST INFRASTRUCTURE ONLY.  Generates tests/golden/cfg1_entropy.npz: per-token policy entropy on BASELINE
config 1 computed by the REFERENCE's own helper, BaseLearner.compute_entropy_bonus (distributed_actor.py:266-281).

The reference never calls that helper (its call sites are commented out, :377-379 and :472-480), so there is no
reference loss to pin; what is pinned is the per-token definition H = -sum_v p_v ln p_v of the rows the learner scores.
Recipe (same stubs, parameters and batch as oracle/make_golden.py, config 1):
  * the stock HF Qwen2ForCausalLM + LoRA policy of make_golden.build_hf_policy, fp32;
  * the slicing of compute_current_policy_probs restated (:245-249: shift by one, keep the answer positions) and the
    fp32 log_softmax over the full vocabulary;
  * compute_entropy_bonus(log_probs[i, t][None, None], alpha=1) for every scored position: with one position its
    `entropy.mean()` is that position's H;
  * the helper's own aggregate over micro-batch 0 (train_batch_size rows, all T positions, pad included) with
    alpha = 0.01, exactly as the commented call at :377-378 would have produced it.

Usage: python oracle/make_golden_entropy.py   (writes tests/golden/cfg1_entropy.npz; needs /root/reference)
"""
from __future__ import annotations

import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from oracle import learner_oracle as lo  # noqa: E402
from oracle import make_golden as mg  # noqa: E402


def main():
    assert os.path.isdir(mg.REF), f"{mg.REF} not found: goldens can only be generated where the reference is"
    mg.install_stubs()
    sys.path.insert(0, mg.REF)
    import distributed_actor as da  # the reference module, unmodified

    torch.manual_seed(0)
    # BASELINE config 1, as in make_golden.main()
    cfg = lo.OracleConfig(vocab=512, hidden=128, inter=256, n_layers=2, n_q_heads=4, n_kv_heads=2, head_dim=32,
                          lora_r=16, lora_alpha=16)
    P, T, B = 16, 32, 2
    seed = 1234
    params, nf4 = lo.make_params(cfg, seed=seed)
    prompts, answers, _ = lo.make_batch(cfg, 4, P, T, seed=1, ragged=True)
    ids, am, ansm = lo.pad_batch(prompts, answers, P, T)
    policy = mg.build_hf_policy(cfg, params)
    policy.eval()
    with torch.no_grad():
        logits = policy(input_ids=ids, attention_mask=am).logits
        logits = logits[:, :-1, :]          # :245
        logits = logits[:, P - 1:]          # :248
        logp = torch.log_softmax(logits.float(), dim=-1)
        n, t = logp.shape[:2]
        H = np.zeros((n, t), dtype=np.float32)
        for i in range(n):
            for j in range(t):
                H[i, j] = float(da.BaseLearner.compute_entropy_bonus(logp[i, j][None, None], 1.0))
        agg = float(da.BaseLearner.compute_entropy_bonus(logp[:B], 0.01))
    fixtures = {"P": P, "T": T, "train_batch_size": B, "param_seed": np.int64(seed),
                "param_sha256": np.array(lo.params_digest(params, nf4)),
                "entropy": H, "answer_mask": ansm.numpy().astype(np.int8),
                "bonus_mb0_alpha": np.float64(0.01), "bonus_mb0": np.float64(agg)}
    out = os.path.join(ROOT, "tests", "golden", "cfg1_entropy.npz")
    np.savez_compressed(out, **fixtures)
    print("wrote", out, os.path.getsize(out), "bytes")


if __name__ == "__main__":
    main()
