"""train_distributed: the reference's CLI surface (train_distributed.py:9-85) in front of the B200 learner.

Every flag of the reference is accepted with the same name, type and default, and lands in the same flat `config` dict the
Trainer and the actors read (:51-81).  Additions (all optional):
  --stub                 synthetic token-id dataset + StubGenerator actors + synthetic rewards (no dataset, tokenizer or vLLM
                         needed: this image has no network); implied by a `random:*` model
  --kl_beta / --clip_eps / --inner_epochs     KL-to-reference weight, clipped-ratio surrogate, epochs per batch (N4)
  --entropy_alpha / --log_entropy   entropy bonus weight (> 0 rewards entropy) / log the mean per-token policy entropy
  --overlap_generation   generate batch k+1 while the learners train on batch k (N3)
  --adapter_sync         memory (default: device-to-device hand-off, N1) | file (PEFT directory like the reference)
  --max_steps, --bench   stop after that many trainer steps / print ONE JSON line with trainer steps per second
                         (BASELINE config 5: "full pipeline ... end-to-end steps/sec")
Example (BASELINE config 5 shape on 8 GPUs, stub generators):
  python -m distrl_llm_b200.train_distributed --model random:qwen2.5-7b --learner grpo --number_of_actors 4 \\
      --number_of_learners 4 --batch_size 512 --learner_chunk_size 0 --max_lora_rank 16 --bench --max_steps 3
"""
from __future__ import annotations

import argparse
import json
import time


def build_parser():
    ap = argparse.ArgumentParser()
    # ---- the reference's flags (train_distributed.py:11-36), same defaults ----
    ap.add_argument("--model", type=str, default="unsloth/Qwen2.5-7B-Instruct-bnb-4bit")
    ap.add_argument("--dataset", type=str, default="HuggingFaceH4/MATH-500")
    ap.add_argument("--run_name", type=str)
    ap.add_argument("--project_name", type=str, default="math-reasoning")
    ap.add_argument("--lora_save_path", type=str, default="lora_request_math")
    ap.add_argument("--lr", type=float, default=2e-5)
    ap.add_argument("--max_new_tokens", type=int, default=1200)
    ap.add_argument("--max_prompt_tokens", type=int, default=350)
    ap.add_argument("--temperature", type=float, default=1.2)
    ap.add_argument("--episodes", type=int, default=15)
    ap.add_argument("--num_candidates", type=int, default=16)
    ap.add_argument("--batch_size", type=int, default=30)
    ap.add_argument("--learner_chunk_size", type=int, default=8)
    ap.add_argument("--train_batch_size", type=int, default=8)
    ap.add_argument("--save_every", type=int, default=100)
    ap.add_argument("--eval_every", type=int, default=10)
    ap.add_argument("--number_of_actors", type=int, default=2)
    ap.add_argument("--number_of_learners", type=int, default=1)
    ap.add_argument("--learner", type=str, choices=["pg", "grpo"], default="pg")
    ap.add_argument("--max_lora_rank", type=int, default=32)
    ap.add_argument("--lora_alpha", type=int, default=16)
    ap.add_argument("--lora_dropout", type=float, default=0)
    ap.add_argument("--topk", type=int, default=16)
    ap.add_argument("--actor_gpu_usage", type=float, default=0.91)
    ap.add_argument("--learner_gpu_usage", type=float, default=0.35)
    # ---- additions ----
    ap.add_argument("--stub", action="store_true")
    ap.add_argument("--kl_beta", type=float, default=0.0)
    ap.add_argument("--clip_eps", type=float, default=0.0)
    ap.add_argument("--inner_epochs", type=int, default=1)
    ap.add_argument("--entropy_alpha", type=float, default=0.0)
    ap.add_argument("--log_entropy", action="store_true")
    ap.add_argument("--overlap_generation", action="store_true")
    ap.add_argument("--adapter_sync", choices=["memory", "file"], default="memory")
    ap.add_argument("--fuse_microbatches", type=int, default=2)
    ap.add_argument("--max_steps", type=int, default=0)
    ap.add_argument("--dataset_size", type=int, default=0, help="--stub: synthetic problems (default: enough for max_steps)")
    ap.add_argument("--bench", action="store_true")
    return ap


def config_from_args(args):
    """The reference's `config` dict (train_distributed.py:51-81) plus the optional keys above."""
    cfg = {k: getattr(args, k) for k in (
        "run_name", "project_name", "lora_save_path", "lr", "max_prompt_tokens", "max_new_tokens", "episodes",
        "num_candidates", "batch_size", "train_batch_size", "temperature", "save_every", "eval_every", "model", "dataset",
        "number_of_actors", "number_of_learners", "learner", "max_lora_rank", "topk", "learner_chunk_size",
        "actor_gpu_usage", "learner_gpu_usage", "lora_alpha", "lora_dropout")}
    cfg["use_vllm"] = True
    cfg.update(kl_beta=args.kl_beta, clip_eps=args.clip_eps, inner_epochs=args.inner_epochs,
               entropy_alpha=args.entropy_alpha, log_entropy=args.log_entropy,
               overlap_generation=args.overlap_generation, adapter_sync=args.adapter_sync,
               fuse_microbatches=args.fuse_microbatches, max_steps=args.max_steps or None)
    return cfg


def main(argv=None):
    args = build_parser().parse_args(argv)
    config = config_from_args(args)
    from .trainer import SyntheticDataset, Trainer
    stub = args.stub or args.model.startswith("random:")
    if stub:
        from .actors import model_config
        from .generator import synthetic_reward_function as reward_function
        mc = model_config(args.model, args.max_lora_rank, args.lora_alpha) if args.model.startswith("random:") else None
        vocab = mc.vocab if mc is not None else 32000
        n = args.dataset_size or max(args.batch_size * max(args.max_steps, 1), args.batch_size)
        train_ds = SyntheticDataset(n, vocab, args.max_prompt_tokens, seed=0)
        test_ds = SyntheticDataset(max(args.batch_size // 4, 1), vocab, args.max_prompt_tokens, seed=1)
    else:   # the reference's data path (train_distributed.py:38-48); needs `datasets`, a tokenizer and network / a cache
        from datasets import load_dataset   # noqa: F401  (absent in this image: fails loudly here)
        raise SystemExit("real datasets / vLLM generators need Ray + vLLM wiring (INTEGRATION.md); use --stub here")
    trainer = Trainer(train_ds, test_ds, reward_function, config)
    t0 = time.time()
    steps, _ = trainer.train()
    wall = time.time() - t0
    if args.bench:
        h = [m for m in trainer.history if "loss" in m]
        upd = [m["timing/update_duration"] for m in h]
        gen = [m["timing/generation_duration"] for m in h]
        tokens = sum(m["mean_token_length"] for m in h)   # informational
        print(json.dumps({"metric": "full pipeline trainer steps/sec (generate -> reward -> advantages -> learners -> adapter hand-off)",
                          "value": steps / wall, "unit": "steps/s", "steps": steps, "wall_s": wall,
                          "timing/update_duration_mean_s": sum(upd) / max(len(upd), 1),
                          "timing/generation_duration_mean_s": sum(gen) / max(len(gen), 1),
                          "mean_token_length": tokens / max(len(h), 1), "generators": "stub" if stub else "vllm",
                          "config": {k: config[k] for k in ("model", "learner", "number_of_actors", "number_of_learners", "batch_size",
                                                            "num_candidates", "topk", "max_new_tokens", "max_prompt_tokens",
                                                            "train_batch_size", "learner_chunk_size", "overlap_generation", "adapter_sync")}}),
              flush=True)
    return trainer


if __name__ == "__main__":
    main()
