"""Learner / GRPOLearner: same method surface as the reference's Ray actors
(distributed_actor.py:196-514), with the learner math running in libb200rl (sm_100a CUDA).

Method-by-method mirror (reference line numbers in each docstring).  Differences that are deliberate
and documented in DESIGN.md:
  * token ids may be passed instead of strings (tokenizer = IdTokenizer) — removes quirk Q6;
  * the loss scalar is accumulated on the device, one .item() per compute_loss instead of one per
    micro-batch (:387 / :485);
  * multi-learner mode: compute_gradients leaves the gradients in a peer-mapped device buffer and
    apply_merged_gradients runs the fused P2P reduce + Adam on EVERY learner (fixes quirk Q4); the
    reference's dict-of-CPU-tensors exchange is still available (export_gradients / a list of dicts
    passed to apply_merged_gradients) and is what the parity tests use.
There is no CPU or torch fallback: constructing a learner without libb200rl / a B200 raises.
"""
from __future__ import annotations

import numpy as np
import torch

from . import ops, packing
from .policy import LMConfig, Policy

try:  # Ray is the reference's process model; optional here (not installed in the build image)
    import ray  # type: ignore

    def _remote(cls):
        return ray.remote(num_gpus=1, num_cpus=1)(cls)
except Exception:  # pragma: no cover
    ray = None

    def _remote(cls):
        return cls


class IdTokenizer:
    """Token-id passthrough with the reference's padding rules (distributed_actor.py:217-229):
    batch_encode_plus(items, padding='max_length', padding_side=..., max_length=..., truncation=True)."""

    def __init__(self, pad_id=0):
        self.pad_token_id = pad_id

    def batch_encode_plus(self, items, return_tensors="pt", padding="max_length", padding_side="right",
                          max_length=None, truncation=True):
        n = len(items)
        ids = np.full((n, max_length), self.pad_token_id, dtype=np.int32)
        mask = np.zeros((n, max_length), dtype=np.int32)
        for i, it in enumerate(items):
            it = list(it)[:max_length]
            if not it:
                continue
            if padding_side == "left":
                ids[i, max_length - len(it):] = it
                mask[i, max_length - len(it):] = 1
            else:
                ids[i, :len(it)] = it
                mask[i, :len(it)] = 1
        return {"input_ids": torch.from_numpy(ids), "attention_mask": torch.from_numpy(mask)}


class BaseLearner:
    """reference BaseLearner (distributed_actor.py:196-333)."""

    learner_type = "pg"

    def __init__(self, policy: Policy, tokenizer, config: dict, gpu_id=0, generator=None, reference_quirks=True):
        self.policy = policy
        self.tokenizer = tokenizer
        self.model_gpu_id = gpu_id                                # :28 (informational)
        self.update_batch_size = config["train_batch_size"]       # :29
        self.max_new_tokens = config["max_new_tokens"]            # :31
        self.max_prompt_tokens = config["max_prompt_tokens"]      # :213
        self.lr = config["lr"]                                    # :210
        self.weight_decay = config.get("weight_decay", 0.0)       # commented out in the reference (:210)
        self.kl_beta = float(config.get("kl_beta", 0.0))          # KL-to-reference weight; 0 = reference behaviour
        # SURVEY.md 8(f) N4 (absent from the reference, whose ratio exp(lp - lp.detach()) is identically 1, :467):
        # clipped-ratio surrogate against the log-probs of the policy that generated the batch, over `inner_epochs`
        # optimizer steps per batch.  Defaults (0, 1) are exactly the reference's single step.
        self.clip_eps = float(config.get("clip_eps", 0.0))
        self.inner_epochs = max(1, int(config.get("inner_epochs", 1)))
        self.last_epoch_losses = []
        # entropy bonus (reference: compute_entropy_bonus, distributed_actor.py:266-281, call sites commented out at
        # :377-379 / :472-480, config key at :437): loss -= entropy_alpha * mean_i(sum_t mask H / len_i) per micro-batch, so
        # alpha > 0 rewards entropy (DESIGN.md).  log_entropy: report the mean per-token entropy of the trained tokens in
        # last_metrics(); implied by entropy_alpha != 0.
        self.entropy_alpha = float(config.get("entropy_alpha", 0.0))
        self.log_entropy = bool(config.get("log_entropy", False)) or self.entropy_alpha != 0.0
        self._metrics = {}
        self._ent_accum = torch.zeros(2, device=policy.device, dtype=torch.float64) if self.log_entropy else None
        self._ent_buf = None
        # packed shared-prompt layout (packing.py): identical results, each distinct prompt of a micro-batch is
        # processed once; needs the tcgen05 attention kernels (head_dim 128)
        self.share_prompts = bool(config.get("share_prompts", policy.cfg.head_dim == 128))
        # packed layout only: do not store pad tokens at all (packing.py; SURVEY 8(f) N2).  Same surviving rows, same positions.
        self.ragged_rows = bool(config.get("ragged_rows", True))
        # head (final norm, lm_head, log-softmax, lm_head dX) on the completion tokens that carry loss only; False =
        # all max_new_tokens positions of every sequence like the reference (:245-260), masked afterwards
        self.compact_scored_rows = bool(config.get("compact_scored_rows", True))
        # Pass fusion: the reference accumulates gradients over micro-batches of train_batch_size sequences
        # (:354-389) because a pass has to fit a 24-80 GB GPU.  The accumulated gradient is linear in the per-sequence
        # coefficients, so k full micro-batches can go through the model as ONE pass with every advantage (and the KL
        # weight) scaled by k -- coef = -(k A)/(len * kB * nb) = -A/(len * B * nb) -- with identical results: weights are
        # streamed once per k micro-batches and the GEMM M dimension fills its last tile.  k is bounded by the capacity
        # the policy was built with (max_batch // train_batch_size) and by config["fuse_microbatches"] (0 = auto).
        cap = max(1, policy.max_batch // max(1, self.update_batch_size))
        want = int(config.get("fuse_microbatches", 0))
        self.fuse_microbatches = cap if want <= 0 else max(1, min(want, cap))
        self.lora_save_path = config.get("lora_save_path", "lora_request_math")
        self.reference_quirks = reference_quirks
        self.generator = generator
        self.p2p = None  # set by enable_p2p() / p2p_open_handles()
        self._p2p_group = None
        self._p2p_handles = None
        self._publisher = None            # adapter_sync.AdapterPublisher once a generator asked for the adapter
        self.adapter_sync = config.get("adapter_sync", "memory")   # "memory" (default once a publisher exists) | "file"
        self.model_name = config.get("model")
        self._stager = packing.PinnedStager(policy.device)   # reusable pinned staging for the per-pass H2D copies

    # ---- tokenise + pad (:217-239) ------------------------------------------------------------
    def _encode(self, messages, answers):
        P, T = self.max_prompt_tokens, self.max_new_tokens
        inputs = self.tokenizer.batch_encode_plus(messages, return_tensors="pt", padding="max_length",
                                                  padding_side="left", max_length=P, truncation=True)
        tok_ans = self.tokenizer.batch_encode_plus(answers, return_tensors="pt", max_length=T,
                                                   padding="max_length", padding_side="right", truncation=True)
        ids = torch.cat([inputs["input_ids"], tok_ans["input_ids"]], dim=1).to(torch.int32)
        am = torch.cat([inputs["attention_mask"], tok_ans["attention_mask"]], dim=1).to(torch.int32)
        return ids, am, tok_ans["attention_mask"].to(torch.int32)

    def _h2d(self, t):
        return self._stager.to_device(t)

    def compute_current_policy_probs(self, policy, messages, answers, return_entropy=False):
        """(:215-261) -> (action_log_probs [B,T] fp32, answer_mask [B,T]) on the device; scoring only.
        return_entropy: (lp, mask, entropy [B,T] fp32 in nats), computed in the same pass over the logits."""
        ids, am, ansm = self._encode(messages, answers)
        B = ids.shape[0]
        lp = torch.empty(B, self.max_new_tokens, device=policy.device, dtype=torch.float32)
        ekw = {}
        if return_entropy:
            ekw["ent_out"] = torch.empty(B, self.max_new_tokens, device=policy.device, dtype=torch.float32)
        if self.share_prompts:
            pk = self._pack(ids, am)
            policy.microbatch_packed(pk, None, 1, False, backward=False, lp_out=lp, **ekw)
            mask = pk.answer_mask
        else:
            mask = self._h2d(ansm)
            policy.microbatch(self._h2d(ids), self._h2d(am), mask, None, self.max_prompt_tokens,
                              self.max_new_tokens, 1, False, backward=False, lp_out=lp, **ekw)
        return (lp, mask, ekw["ent_out"]) if return_entropy else (lp, mask)

    def _pack(self, ids, am):
        host = packing.pack_microbatch(ids.numpy(), am.numpy(), self.max_prompt_tokens, self.max_new_tokens,
                                       ragged=self.ragged_rows, compact_scored=self.compact_scored_rows)
        return packing.PackedDevice(host, self.policy.device, stager=self._stager)

    # ---- loss + backward (:349-395 PG, :440-493 GRPO) ---------------------------------------------
    def compute_loss(self, messages, answers, rewards, old_lp=None, lp_capture=None):
        """old_lp [n, T] f32 device tensor (+ self.clip_eps > 0): clipped-ratio surrogate; lp_capture [n, T]: filled with
        the current per-token log-probs of every trained sequence (the next inner epoch's old_lp).  Both None = reference."""
        rewards = np.asarray([float(r) for r in rewards], dtype=np.float64)   # :350 / :441 (float64)
        n = len(messages)
        clip = self.clip_eps if old_lp is not None else 0.0
        nb = (n + self.update_batch_size - 1) // self.update_batch_size      # :354-356
        pol = self.policy
        pol.zero_grad()                                                       # :358 / :450
        pol.loss_accum.zero_()
        ent_accum = self._ent_accum
        if ent_accum is not None:
            ent_accum.zero_()
            if self._ent_buf is None:
                self._ent_buf = torch.empty(pol.max_batch * self.max_new_tokens, device=pol.device, dtype=torch.float32)
        grpo = self.learner_type == "grpo"
        B = self.update_batch_size
        # plan the passes: runs of up to `fuse_microbatches` FULL micro-batches that survive the skip predicate
        passes, cur = [], []
        for i in range(nb):
            s, e = i * B, min((i + 1) * B, n)
            # :367 / :459  `if batch_rewards.all() == 0: continue` — true when ANY reward is exactly 0 (quirk Q1)
            if self.reference_quirks and not bool(np.all(rewards[s:e] != 0)):
                continue
            if e - s == B and self.fuse_microbatches > 1:
                cur.append((s, e))
                if len(cur) == self.fuse_microbatches:
                    passes.append(cur)
                    cur = []
            else:
                passes.append([(s, e)])
        if cur:
            passes.append(cur)
        for group in passes:
            k = len(group)
            idx = [j for (s, e) in group for j in range(s, e)]
            msgs, answ = [messages[j] for j in idx], [answers[j] for j in idx]
            r = rewards[idx] * float(k)          # see __init__: k fused micro-batches
            beta = self.kl_beta * k
            ekw = {}
            if ent_accum is not None:    # alpha scaled like the advantages and kl_beta (see __init__)
                ekw = dict(entropy_alpha=self.entropy_alpha * k, ent_out=self._ent_buf[:len(idx) * self.max_new_tokens],
                           ent_accum=ent_accum)
            ids, am, ansm = self._encode(msgs, answ)
            didx = torch.as_tensor(idx, device=pol.device) if (old_lp is not None or lp_capture is not None) else None
            olp = old_lp.index_select(0, didx).contiguous() if old_lp is not None else None
            lp_now = torch.empty(len(idx), self.max_new_tokens, device=pol.device, dtype=torch.float32) if lp_capture is not None else None
            if self.share_prompts:
                pk = self._pack(ids, am)
                ref_lp = None
                if self.kl_beta != 0.0:
                    ref_lp = torch.empty(len(idx), self.max_new_tokens, device=pol.device, dtype=torch.float32)
                    pol.microbatch_packed(pk, None, 1, False, backward=False, lp_out=ref_lp, lora_off=True)
                pol.microbatch_packed(pk, self._h2d(torch.from_numpy(r)), nb, grpo, backward=True, ref_lp=ref_lp,
                                      kl_beta=beta, lp_out=lp_now, old_lp=olp, clip_eps=clip, **ekw)
            else:
                d_ids, d_am, d_ansm = self._h2d(ids), self._h2d(am), self._h2d(ansm)
                ref_lp = None
                if self.kl_beta != 0.0:
                    # reference policy = the frozen base with the adapter disabled (one extra forward, no backward)
                    ref_lp = torch.empty(len(idx), self.max_new_tokens, device=pol.device, dtype=torch.float32)
                    pol.microbatch(d_ids, d_am, d_ansm, None, self.max_prompt_tokens, self.max_new_tokens, 1, False,
                                   backward=False, lp_out=ref_lp, lora_off=True)
                pol.microbatch(d_ids, d_am, d_ansm, self._h2d(torch.from_numpy(r)), self.max_prompt_tokens,
                               self.max_new_tokens, nb, grpo, backward=True, ref_lp=ref_lp, kl_beta=beta, lp_out=lp_now,
                               old_lp=olp, clip_eps=clip, **ekw)
            if lp_capture is not None:
                lp_capture.index_copy_(0, didx, lp_now)
        if ent_accum is None:
            self._metrics = {}
            return float(pol.loss_accum.item())   # sum of per-micro-batch losses (quirk Q2), one sync
        loss, h_sum, n_tok = torch.cat([pol.loss_accum, ent_accum]).tolist()   # still one sync
        self._metrics = {"entropy": h_sum / n_tok if n_tok > 0 else float("nan"), "entropy_tokens": int(n_tok)}
        return loss

    def last_metrics(self):
        """Metrics of the last compute_loss / train / compute_gradients (first inner epoch): {"entropy": mean per-token
        entropy in nats over the answer tokens trained, "entropy_tokens": their count}; {} when entropy logging is off."""
        return dict(self._metrics)

    def _train_epochs(self, problems, answers, rewards):
        """One optimizer step per inner epoch on the same batch (reference: exactly one, :407-415 / :507-513).  Epoch 0 is
        the reference's step (ratio == 1) and records the per-token log-probs; later epochs use them as the old policy of
        the clipped surrogate.  Returns the first epoch's loss (the number the reference returns)."""
        old = None
        self.last_epoch_losses = []
        metrics = {}
        for epoch in range(self.inner_epochs):
            capture = None
            if epoch == 0 and self.inner_epochs > 1 and self.clip_eps > 0:
                capture = torch.zeros(len(problems), self.max_new_tokens, device=self.policy.device, dtype=torch.float32)
            loss = self.compute_loss(problems, answers, rewards, old_lp=old, lp_capture=capture)
            if epoch == 0:
                metrics = self._metrics
            self.policy.optimizer_step(self.lr, weight_decay=self.weight_decay)
            self.last_epoch_losses.append(loss)
            if capture is not None:
                old = capture
        self._metrics = metrics
        return self.last_epoch_losses[0]

    # ---- gradient export / merge (:283-333) --------------------------------------------------------
    def export_gradients(self):
        """{PEFT name: CPU tensor} (:289-293) from ONE device->host copy of the flat buffer."""
        host = self.policy.lora_grad.detach().cpu()
        return {k: v.clone() for k, v in self.policy.named_views(host).items()}

    def _compute_gradients(self, problems, answers, rewards, export=True):
        loss = self.compute_loss(problems, answers, rewards)   # zero_grad + compute_loss (:285-286)
        return (self.export_gradients() if export else {}), loss

    def compute_gradients(self, candidates):
        """(:296-300). With P2P enabled the gradients stay on the device (returns ({}, loss))."""
        problems, answers, rewards = candidates
        return self._compute_gradients(problems, answers, rewards, export=self.p2p is None)

    def apply_merged_gradients(self, gradients_list=None):
        """(:302-333). Reference path: list of gradient dicts -> mean -> Adam. P2P path: fused one-shot
        reduce + Adam + write-back on every learner (gradients_list ignored)."""
        pol = self.policy
        if self.p2p is not None:
            self.p2p.reduce_adam_step(pol, self.lr, self.weight_decay)
            return
        if not gradients_list:
            print("No gradients to merge.")
            return
        n = len(gradients_list)
        merged = None
        for g in gradients_list:   # :316-319 (sum) ... :322-323 (divide)
            flat = torch.zeros(pol.lora_numel, dtype=torch.float32)
            views = pol.named_views(flat)
            for k, v in g.items():
                views[k].copy_(v)
            merged = flat if merged is None else merged + flat
        merged /= n
        pol.lora_grad.copy_(merged.to(pol.device))                    # :326-328
        pol.optimizer_step(self.lr, weight_decay=self.weight_decay)   # :331-333

    def enable_p2p(self, group):
        self.p2p = group

    # Ray flow (INTEGRATION.md): create_for_p2p() builds the policy on IPC-exportable buffers; the driver gathers every
    # learner's handles with p2p_export_handles() and broadcasts the list to p2p_open_handles().  Those two RPC rounds
    # are also the host-side rendezvous that keeps the GPU flag barrier of attach() short.
    @classmethod
    def create_for_p2p(cls, rank, world, device, build_policy, tokenizer, config, numel, **kw):
        """Learner `rank` of `world` for the fused P2P reduce + Adam exchange.  `numel` = p2p.lora_numel(cfg, ...);
        `build_policy(lora_flat=..., lora_grad=...)` must construct the Policy on the given buffers (e.g.
        `lambda **b: Policy.random_init(cfg, device, max_batch, P, T, **b)`)."""
        from .p2p import P2PGroup
        group = P2PGroup(rank, world, device)
        handles, bufs = group.alloc_local(numel)
        self = cls(build_policy(**bufs), tokenizer, config, gpu_id=rank, **kw)
        self._p2p_group, self._p2p_handles = group, handles
        return self

    def p2p_export_handles(self):
        if self._p2p_handles is None:
            raise RuntimeError("this learner was not built with create_for_p2p(): it has no exportable buffers")
        return self._p2p_handles

    def p2p_open_handles(self, all_handles, host_rendezvous=None):
        if self._p2p_group is None:
            raise RuntimeError("this learner was not built with create_for_p2p()")
        self._p2p_group.open_peers(all_handles)
        self._p2p_group.attach(self.policy, host_rendezvous=host_rendezvous)
        self.p2p = self._p2p_group

    # same-process harness (actors.create_actor_and_learner without Ray): the groups exchange plain pointers
    def p2p_local_group(self):
        return self._p2p_group

    def p2p_attach_local(self):
        self._p2p_group.attach(self.policy, host_rendezvous=lambda: None)
        self.p2p = self._p2p_group

    def vocab_size(self):
        return self.policy.cfg.vocab

    def warmup(self):
        """Run one throw-away micro-batch (forward, backward, optimizer kernels) and restore the state.  CUDA loads a
        kernel's code at its first launch and that load synchronises with the device, so learners that SHARE a device (one
        process, one stream each — tests) must have launched every kernel once before the first P2P barrier spins on it."""
        pol = self.policy
        flat, m, v, step = pol.lora_flat.clone(), pol.adam_m.clone(), pol.adam_v.clone(), pol.opt_step
        metrics = self._metrics
        B = min(self.update_batch_size, pol.max_batch)
        msgs = [[1, 2, 3]] * B
        answ = [[4, 5, 6, 7]] * B
        self.compute_loss(msgs, answ, [1.0] * B)   # launches the entropy kernels too when they are enabled
        self._metrics = metrics
        pol.optimizer_step(self.lr)
        pol.lora_flat.copy_(flat); pol.adam_m.copy_(m); pol.adam_v.copy_(v)
        pol.opt_step = step
        pol.lora_grad.zero_()
        pol.sync_lora()
        torch.cuda.current_stream(pol.device).synchronize()

    def export_flat(self):
        """The flat fp32 adapter on the host (tests / debugging)."""
        torch.cuda.current_stream(self.policy.device).synchronize()
        if self.p2p is not None:
            self.p2p.check()
        return self.policy.lora_flat.detach().cpu().clone()

    # ---- adapter hand-off to the generators (SURVEY.md 8(f) N1) -------------------------------------------------------
    def adapter_publisher(self):
        """Create (once) the in-memory publisher of this learner's adapter and return its picklable description for the
        generators' AdapterSubscriber (adapter_sync.py).  From then on save_adapter() publishes instead of writing files."""
        if self._publisher is None:
            from .adapter_sync import AdapterPublisher
            self._publisher = AdapterPublisher(self.policy)
            self._publisher.publish()
        return self._publisher.describe()

    # ---- misc actor surface --------------------------------------------------------------------------
    def generate(self, messages, sampling_params=None):
        """(:174-180) generation is the generator's job (vLLM or a stub), not part of the hot path.  The reference's
        Trainer always sends the learners a chunk of `learner_chunk_size` problems (distributed_trainer.py:187-197); a
        learner without a generator accepts only the empty chunk (`--learner_chunk_size 0`)."""
        if self.generator is None:
            if len(messages.get("problem", [])) == 0:
                return dict(messages, answers=[], token_lengths=[])
            raise RuntimeError("this learner has no generator attached: run the trainer with learner_chunk_size=0 "
                               "(all problems go to the generators) or pass generator=... to the learner")
        return self.generator.generate(messages, sampling_params)

    def save_checkpoint(self, path):
        """(:263-264) `self.policy.save_pretrained(path)` on a PEFT model = an adapter directory.  Written here in the
        same on-disk format (adapter_model.safetensors with PEFT's saved key names + adapter_config.json), plus the
        torch-pickled dict with the in-memory names the gradient exchange uses (T2) and — what the reference lacks
        (no resume path, README TODO; SURVEY.md 8(f) N4) — the optimizer state: Adam moments and the step counter."""
        import os
        os.makedirs(path, exist_ok=True)
        sd = self.policy.lora_state_dict()
        torch.save(sd, os.path.join(path, "adapter_model.pt"))
        write_peft_adapter(path, sd, self.policy.cfg, base_model=self.model_name)
        self.save_optimizer_state(path)

    def save_optimizer_state(self, path):
        """Adam moments + step counter.  Single learner: the whole state in optimizer_state.pt.  With the fused P2P exchange
        every learner holds the moments of ITS 1/N slice only (csrc/optim.cu), so each learner writes its slice
        (optimizer_state.rank{r}of{n}.pt; the Trainer calls this on every learner) and load_checkpoint merges what it finds."""
        import os
        os.makedirs(path, exist_ok=True)
        pol = self.policy
        meta = {"opt_step": int(pol.opt_step), "lr": self.lr, "weight_decay": self.weight_decay, "betas": (0.9, 0.999),
                "eps": 1e-8, "lora_numel": int(pol.lora_numel)}
        if self.p2p is None:
            torch.save(dict(meta, adam_m=pol.adam_m.detach().cpu(), adam_v=pol.adam_v.detach().cpu()),
                       os.path.join(path, "optimizer_state.pt"))
            return
        from .p2p import owned_slice
        lo, hi = owned_slice(self.p2p.numel, self.p2p.world, self.p2p.rank)
        torch.save(dict(meta, lo=lo, hi=hi, adam_m=pol.adam_m[lo:hi].detach().cpu(), adam_v=pol.adam_v[lo:hi].detach().cpu()),
                   os.path.join(path, f"optimizer_state.rank{self.p2p.rank}of{self.p2p.world}.pt"))

    def load_checkpoint(self, path):
        """Resume from a directory written by save_checkpoint (adapter + optimizer state) or by PEFT / the reference itself
        (adapter only: the Adam moments and the step counter then restart from zero, as for a fresh optimizer).
        In multi-learner mode call it on every learner (they hold identical replicas)."""
        import os
        sd, conf = read_peft_adapter(path)
        cfg = self.policy.cfg
        if int(conf.get("r", cfg.lora_r)) != cfg.lora_r:
            raise ValueError(f"adapter rank {conf.get('r')} != policy rank {cfg.lora_r}")
        if "lora_alpha" in conf and float(conf["lora_alpha"]) != float(cfg.lora_alpha):
            raise ValueError(f"adapter lora_alpha {conf['lora_alpha']} != policy lora_alpha {cfg.lora_alpha} (the scale alpha/r would change silently)")
        want = {"q_proj", "k_proj", "v_proj", "o_proj", "gate_proj", "up_proj", "down_proj"}
        if "target_modules" in conf and set(conf["target_modules"]) != want:
            raise ValueError(f"adapter target_modules {sorted(conf['target_modules'])} != {sorted(want)} (helper.py:29-37)")
        self.policy.load_lora_state(sd)
        pol = self.policy
        import glob
        pol.adam_m.zero_()
        pol.adam_v.zero_()
        pol.opt_step = 0
        opt = os.path.join(path, "optimizer_state.pt")
        slices = sorted(glob.glob(os.path.join(path, "optimizer_state.rank*of*.pt")))
        for f in ([opt] if os.path.exists(opt) else slices):   # whole state, or the per-learner slices of a P2P run
            st = torch.load(f, map_location="cpu")
            if int(st["lora_numel"]) != int(pol.lora_numel):
                raise ValueError("optimizer state belongs to a different adapter layout")
            lo, hi = int(st.get("lo", 0)), int(st.get("hi", pol.lora_numel))
            pol.adam_m[lo:hi].copy_(st["adam_m"].to(pol.device))
            pol.adam_v[lo:hi].copy_(st["adam_v"].to(pol.device))
            pol.opt_step = int(st["opt_step"])
        pol.lora_grad.zero_()

    def save_adapter(self):
        """(:84-86) `save_lora(self.policy, self.lora_save_path)`: makes the current adapter available to the generators
        (`load_lora`, :150).  With an in-memory publisher (adapter_publisher()) that is one device-to-device copy and a
        version bump; otherwise (or with config["adapter_sync"] == "file") the PEFT adapter directory vLLM loads."""
        if self._publisher is not None and self.adapter_sync != "file":
            return self._publisher.publish()
        import os
        os.makedirs(self.lora_save_path, exist_ok=True)
        write_peft_adapter(self.lora_save_path, self.policy.lora_state_dict(), self.policy.cfg, base_model=self.model_name)


def read_peft_adapter(path):
    """Inverse of write_peft_adapter: {in-memory PEFT name (`...lora_A.default.weight`): fp32 CPU tensor} and the
    adapter_config dict, from a PEFT adapter directory (also one written by PEFT / the reference itself)."""
    import json
    import os
    from safetensors.torch import load_file
    conf = json.load(open(os.path.join(path, "adapter_config.json")))
    raw = load_file(os.path.join(path, "adapter_model.safetensors"))
    out = {}
    for k, v in raw.items():
        if k.endswith(".lora_A.weight") or k.endswith(".lora_B.weight"):
            k = k[:-len("weight")] + "default.weight"
        out[k] = v.to(torch.float32)
    return out, conf


def write_peft_adapter(path, lora_state, cfg, base_model=None):
    """PEFT adapter directory from {in-memory PEFT name: tensor}: `...lora_A.default.weight` is stored as
    `...lora_A.weight` (PEFT strips the adapter name on save), fp32 tensors, and the adapter_config.json vLLM / PEFT
    need to rebuild the LoRA (r, alpha, target modules; helper.py:25-45)."""
    import json
    import os
    from safetensors.torch import save_file
    tensors = {k.replace(".default.weight", ".weight"): v.detach().to(torch.float32).contiguous().cpu() for k, v in lora_state.items()}
    save_file(tensors, os.path.join(path, "adapter_model.safetensors"), metadata={"format": "pt"})
    conf = {"peft_type": "LORA", "task_type": "CAUSAL_LM", "base_model_name_or_path": base_model, "inference_mode": True,
            "r": int(cfg.lora_r), "lora_alpha": float(cfg.lora_alpha), "lora_dropout": 0.0, "bias": "none",
            "fan_in_fan_out": False, "init_lora_weights": True, "modules_to_save": None, "use_rslora": False,
            "target_modules": ["q_proj", "k_proj", "v_proj", "o_proj", "gate_proj", "up_proj", "down_proj"]}
    with open(os.path.join(path, "adapter_config.json"), "w") as f:
        json.dump(conf, f, indent=1)


class Learner(BaseLearner):
    """reference Learner (PG), distributed_actor.py:336-416."""

    learner_type = "pg"

    def train(self, candidates):
        """(:397-416): flatten, subtract the per-problem baseline (`r - b`, :406), compute_loss, step."""
        problems, answers, rewards = [], [], []
        for cand in candidates:
            for a, p, r, b in zip(cand["answers"], cand["problem"], cand["rewards"], cand["baselines"]):
                problems.extend(p)
                answers.extend(a)
                rewards.extend(np.asarray(r) - b)
        return self._train_epochs(problems, answers, rewards)


class GRPOLearner(BaseLearner):
    """reference GRPOLearner, distributed_actor.py:419-514."""

    learner_type = "grpo"

    def train(self, candidates):
        """(:495-514)"""
        problems, answers, rewards = [], [], []
        for cand in candidates:
            for a, p, r in zip(cand["answers"], cand["problem"], cand["rewards"]):
                problems.extend(p)
                answers.extend(a)
                rewards.extend(r)
        return self._train_epochs(problems, answers, rewards)


RemoteLearner = _remote(Learner) if ray is not None else Learner
RemoteGRPOLearner = _remote(GRPOLearner) if ray is not None else GRPOLearner
