"""Trainer: the reference's orchestration loop (distributed_trainer.py:13-415) around the B200 learner.

Same constructor, same method names, same call ORDER on the actors — generate on every actor and learner chunk
(:178-203), rewards on the driver (:205-219), advantages + top-k (:262-294), then `train` on one learner (:306-307) or
merge -> even split -> `compute_gradients` on every learner -> `apply_merged_gradients` (:308-342), `save_adapter`
(:346), metrics (:348-366), `evaluate` (:384-415), `save_checkpoint` (:373-380) — and the same metric names, so a
maintainer of the reference finds everything where it was.  What differs, on purpose:
  * actor handles come from Ray when it is installed, else from local_rpc (one thread per actor in this process);
  * the advantage / top-k block runs in the fp64 G9 CUDA kernel (trainer_prep.apply_advantages_and_topk);
  * with the P2P exchange enabled, `compute_gradients` leaves the gradients on the device (returns {}), and
    `apply_merged_gradients` is called on EVERY learner (the fused reduce + Adam needs all of them; fixes quirk Q4);
  * `save_adapter` publishes the adapter in memory (adapter_sync.py, SURVEY.md 8(f) N1) unless config["adapter_sync"]
    == "file";
  * config["overlap_generation"] (SURVEY.md 8(f) N3, default off = the reference's strictly serial loop): the next
    batch is generated while the learners update on the current one (the generators then run one adapter version
    behind — the clipped-ratio objective of config["clip_eps"] is made for exactly that).
"""
from __future__ import annotations

import os
import time

import numpy as np

from . import local_rpc, trainer_prep

try:  # pragma: no cover - Ray is not installed in the build image
    import ray as _ray
    _get = _ray.get
except Exception:  # noqa: BLE001
    _ray = None
    _get = local_rpc.get


class SyntheticDataset:
    """`datasets.Dataset` look-alike for the two calls the trainer makes (`shuffle()`, `iter(batch_size=...)`): prompts
    are token-id lists (IdTokenizer passthrough), solutions are ints."""

    def __init__(self, n, vocab, max_prompt_tokens, seed=0, min_len_frac=0.5):
        rng = np.random.default_rng(seed)
        lo = max(1, int(max_prompt_tokens * min_len_frac))
        self.rows = [{"problem": rng.integers(1, vocab, size=int(rng.integers(lo, max_prompt_tokens + 1))).tolist(),
                      "solution": int(rng.integers(0, 1000))} for _ in range(n)]
        self._rng = rng

    def __len__(self):
        return len(self.rows)

    def shuffle(self):
        self._rng.shuffle(self.rows)
        return self

    def iter(self, batch_size):
        for i in range(0, len(self.rows), batch_size):
            chunk = self.rows[i:i + batch_size]
            yield {k: [r[k] for r in chunk] for k in chunk[0]}


class Trainer:
    def __init__(self, dataset, test_dataset, reward_function, config, actors=None, learners=None, log=None):
        """actors / learners: lists of actor handles (`handle.method.remote(...)`); when omitted they are created by
        actors.create_actor_and_learner(config) like the reference (:31-33)."""
        self.dataset, self.test_dataset = dataset, test_dataset
        self.reward_function = reward_function
        self.config = config
        if actors is None or learners is None:
            from .actors import create_actor_and_learner
            actors, learners = create_actor_and_learner(config["number_of_actors"], config["number_of_learners"],
                                                        config["model"], None, config)
        self.actors, self.learners = actors, learners
        self.num_actors, self.num_learners = len(actors), len(learners)
        self.episodes = config["episodes"]
        self.batch_size = config["batch_size"]
        self.learner_chunk_size = config["learner_chunk_size"]
        self.num_candidates = config["num_candidates"]
        self.save_every = config["save_every"]
        self.eval_every = config["eval_every"]
        self.topk = config["topk"]
        self.run_name = config.get("run_name")
        self.run_directory = f"run_{self.run_name}"
        self.learner_type = config["learner"]
        self.prep_device = config.get("prep_device", "cuda:0")
        self.overlap = bool(config.get("overlap_generation", False))
        self.max_steps = config.get("max_steps")          # bench / tests: stop after this many trainer steps
        self.history = []
        self._log = log or (lambda metrics, step: self.history.append(dict(metrics, step=step)))
        self.eval_n = 8                                   # reference: SamplingParams(temperature=0.6, top_p=0.95, n=8) (:53-58)

    # ---- host-side batch chunking (reference :77-169), parity-pinned by tests/golden/trainer_chunks.json ----------
    @staticmethod
    def calculate_chunk_sizes(batch_size, num_actors, num_learners=1, learner_chunk_size=1):
        """Problems per actor, then per learner.  Learners take `learner_chunk_size` each, actors share the rest
        (remainder to the first ones); when the batch is too small actors are served first with one problem each and the
        learners split what is left."""
        if batch_size <= 0 or num_learners <= 0 or num_actors < 0:
            raise ValueError("Batch size, number of learners and number of actors must be positive")
        if batch_size < num_actors + learner_chunk_size * num_learners:
            print(f"Warning: Batch size ({batch_size}) is smaller than actors + learners need "
                  f"({num_actors + learner_chunk_size * num_learners})")
            if batch_size >= num_actors:
                spare = batch_size - num_actors
                if spare > 0:
                    learner_chunk_size = max(1, spare // num_learners)
                    num_learners = min(num_learners, spare // learner_chunk_size)
                else:
                    num_learners = 0
            else:
                num_actors, num_learners = batch_size, 0
        for_actors = batch_size - learner_chunk_size * num_learners
        chunks = [for_actors // num_actors + (1 if i < for_actors % num_actors else 0) for i in range(num_actors)]
        return chunks + [learner_chunk_size] * num_learners

    @staticmethod
    def split_dict_lists(data, chunk_sizes):
        if isinstance(chunk_sizes, int):
            chunk_sizes = [chunk_sizes]
        n = len(next(iter(data.values())))
        if any(len(v) != n for v in data.values()):
            raise ValueError("All lists in the dictionary must have the same length")
        if sum(chunk_sizes) != n:
            raise ValueError(f"Sum of chunk sizes ({sum(chunk_sizes)}) must equal the length of lists ({n})")
        out, start = [], 0
        for size in chunk_sizes:
            out.append({k: v[start:start + size] for k, v in data.items()})
            start += size
        return out

    def merge_candidates(self, candidates):
        return trainer_prep.merge_candidates(candidates)   # drops 'baselines' like the reference (quirk Q5)

    # ---- generation + rewards (reference :171-219) --------------------------------------------------------------------
    def _start_round(self, batch, sampling_params=None):
        sizes = self.calculate_chunk_sizes(len(batch["problem"]), self.num_actors, self.num_learners, self.learner_chunk_size)
        chunks = self.split_dict_lists(batch, sizes)
        futures = [a.generate.remote(t, sampling_params) for a, t in zip(self.actors, chunks[:self.num_actors])]
        n_l = len(sizes) - min(self.num_actors, len(sizes))           # learner chunks that survived a small batch
        futures += [l.generate.remote(t, sampling_params) for l, t in zip(self.learners, chunks[len(chunks) - n_l:])] if n_l else []
        return futures, time.time()

    def _finish_round(self, started):
        futures, t0 = started
        generations = [g for g in _get(futures, timeout=240) if g["problem"]]
        return generations, time.time() - t0

    def _compute_round_rewards(self, candidate_data):
        t0 = time.time()
        for cand in candidate_data:
            cand["rewards"] = [self.reward_function(a, s) for a, s in zip(cand["answers"], cand["solution"])]
        return candidate_data, time.time() - t0

    def _generate_all_candidates(self, batch, sampling_params=None):
        cands, gen_s = self._finish_round(self._start_round(batch, sampling_params))
        cands, rew_s = self._compute_round_rewards(cands)
        return cands, gen_s, rew_s

    # ---- one policy update (reference :302-346) ---------------------------------------------------------------------
    def _update(self, candidates):
        loss = self._update_learners(candidates)
        self._update_metrics = {}
        if self.config.get("log_entropy") or self.config.get("entropy_alpha", 0.0):
            # token-weighted mean per-token policy entropy over every learner's trained tokens
            ms = [m for m in _get([l.last_metrics.remote() for l in self.learners]) if m.get("entropy_tokens", 0) > 0]
            n = sum(m["entropy_tokens"] for m in ms)
            self._update_metrics["entropy"] = sum(m["entropy"] * m["entropy_tokens"] for m in ms) / n if n else float("nan")
        return loss

    def _update_learners(self, candidates):
        if self.num_learners == 1:
            return _get(self.learners[0].train.remote(candidates))
        problems, answers, rewards = self.merge_candidates(candidates)
        chunks = trainer_prep.split_for_learners(problems, answers, rewards, self.num_learners)
        futures = [l.compute_gradients.remote(c) for l, c in zip(self.learners, chunks)]
        gradients, losses = [], []
        for f in futures:
            g, loss = _get(f, timeout=240)
            gradients.append(g)
            losses.append(loss)
        if all(len(g) == 0 for g in gradients):     # P2P mode: the fused reduce + Adam runs on every learner
            _get([l.apply_merged_gradients.remote(None) for l in self.learners])
        else:                                       # reference exchange: list of dicts to learner 0 only (:342)
            _get(self.learners[0].apply_merged_gradients.remote(gradients))
        return sum(losses) / len(losses)

    def save_adapter(self):
        _get(self.learners[0].save_adapter.remote())

    def _save_checkpoint(self, path):
        """reference :373-380 (learner 0 writes the adapter); with several learners the others add their slice of the Adam
        moments (the fused exchange keeps them sharded)."""
        _get(self.learners[0].save_checkpoint.remote(path))
        if self.num_learners > 1:
            _get([l.save_optimizer_state.remote(path) for l in self.learners[1:]])

    # ---- the loop (reference :232-382) ----------------------------------------------------------------------------------
    def train(self):
        step = samples = 0
        if self.eval_every > 0:
            self.evaluate(step)
        t_run = time.time()
        for episode in range(self.episodes):
            self.dataset = self.dataset.shuffle()
            loader = iter(self.dataset.iter(batch_size=self.batch_size))
            batch = next(loader, None)
            started = self._start_round(batch) if batch is not None else None
            while batch is not None:
                step += 1
                samples += len(batch["problem"])
                candidates, gen_s = self._finish_round(started)
                candidates, rew_s = self._compute_round_rewards(candidates)
                nxt = next(loader, None)
                if self.overlap and nxt is not None:      # N3: generate batch k+1 while the learners train on batch k
                    started = self._start_round(nxt)
                m = self._reward_metrics(candidates)
                candidates = trainer_prep.apply_advantages_and_topk(candidates, self.learner_type, self.topk, self.prep_device)
                t0 = time.time()
                loss = self._update(candidates)
                upd_s = time.time() - t0
                self.save_adapter()
                m.update(self._update_metrics)
                m.update({"loss": loss, "episode": episode, "total_batch_steps": step, "total_samples_processed": samples,
                          "timing/update_duration": upd_s, "timing/reward_duration": rew_s, "timing/generation_duration": gen_s})
                self._log(m, step)
                if self.eval_every > 0 and step % self.eval_every == 0:
                    self.evaluate(step)
                if step % self.save_every == 0:
                    self._save_checkpoint(os.path.join(self.run_directory, f"model_{step}"))
                if self.max_steps and step >= self.max_steps:
                    return step, time.time() - t_run
                if not self.overlap and nxt is not None:
                    started = self._start_round(nxt)
                batch = nxt
            if not self.max_steps:
                self._save_checkpoint(os.path.join(self.run_directory, f"model_{step}"))
        return step, time.time() - t_run

    @staticmethod
    def _reward_metrics(candidates):
        fmt, acc, mx, mn, tl = [], [], [], [], []
        for cand in candidates:
            for r, tok in zip(cand["rewards"], cand["token_lengths"]):
                fmt.append(np.mean(r[:, 0])); acc.append(np.mean(r[:, 1])); mx.append(np.max(r[:, 1])); mn.append(np.min(r[:, 1]))
                tl.append(np.mean(tok))
        return {"mean_format_reward": float(np.mean(fmt)), "mean_accuracy_reward": float(np.mean(acc)),
                "min_accuracy_reward": float(np.mean(mn)), "max_accuracy_reward": float(np.mean(mx)),
                "mean_token_length": float(np.mean(tl))}

    def evaluate(self, total_steps):
        """reference :384-415: mean-of-n pass@1 and best-of-n on the test split."""
        t0 = time.time()
        passed = best = problems = 0
        lengths = []
        params = type("SamplingParams", (), {"n": self.eval_n, "temperature": 0.6, "top_p": 0.95})()
        for batch in self.test_dataset.iter(batch_size=self.batch_size):
            cands, _, _ = self._generate_all_candidates(batch, params)
            for cand in cands:
                for r, tok in zip(cand["rewards"], cand["token_lengths"]):
                    lengths.append(np.mean(tok)); passed += np.mean(r[:, 1]); best += np.max(r[:, 1]); problems += 1
        if problems:
            self._log({f"eval/pass@1(mean{self.eval_n})": passed / problems, f"eval/BoN({self.eval_n})": best / problems,
                       "eval/mean_token_length": float(np.mean(lengths)), "timing/eval_duration": time.time() - t0}, total_steps)
