"""ORACLE — TEST INFRASTRUCTURE ONLY.  Per-token policy entropy and the entropy bonus, on top of learner_oracle.

Reference: BaseLearner.compute_entropy_bonus (distributed_actor.py:266-281), whose call sites are commented out
(:377-379 PG, :472-480 GRPO).  What is pinned and what is not:
  * per-token entropy H = -sum_v p_v ln p_v of the rows compute_current_policy_probs scores (fp32 log_softmax, temperature
    1): pinned to the reference helper itself through tests/golden/cfg1_entropy.npz (oracle/make_golden_entropy.py);
  * the loss term restates THIS repo's definition (masked, per-sequence mean, mean over the micro-batch, alpha > 0
    rewards entropy; DESIGN.md), "parity unpinned" like the KL and clipped-ratio terms.

The loss is linear in its terms, so the entropy term is computed and back-propagated after learner_oracle.compute_loss
over the same micro-batches; the accumulated .grad is the gradient of the sum.
"""
from __future__ import annotations

import numpy as np
import torch

from oracle import learner_oracle as lo


def answer_log_softmax(params, cfg, ids, attn_mask, P, dtype=torch.float32):
    """The slicing of compute_current_policy_probs (distributed_actor.py:245-249) -> fp32 log_softmax [B, T, V]."""
    logits = lo.model_forward(params, cfg, ids, attn_mask, dtype)
    return torch.log_softmax(logits[:, :-1, :][:, P - 1:].float(), dim=-1)


def entropy_from_log_probs(logp):
    """H = -sum_v p_v ln p_v over the last dim (compute_entropy_bonus, distributed_actor.py:277-278, before its mean)."""
    return -(logp.exp() * logp).sum(-1)


def compute_current_policy_entropy(params, cfg, ids, attn_mask, P, dtype=torch.float32):
    """Per-token entropy [B, T] in nats (fp32) of the full-vocabulary softmax of every scored row."""
    return entropy_from_log_probs(answer_log_softmax(params, cfg, ids, attn_mask, P, dtype))


def entropy_loss(params, cfg, ids, attn_mask, answer_mask, rewards, P, train_batch_size, entropy_alpha,
                 dtype=torch.float32, reference_quirks=True):
    """Back-propagates the entropy term of every micro-batch compute_loss trains (same skip predicate, quirk Q1 :367 /
    :459; same 1/nb scaling :382 / :479):  L_H = -alpha * mean_i( sum_t mask H / len_i ).  Returns sum over micro-batches
    of L_H (before /nb), the part it adds to the reference's returned loss (quirk Q2)."""
    rewards = torch.as_tensor(np.asarray(rewards), dtype=torch.float64)
    N = ids.shape[0]
    nb = (N + train_batch_size - 1) // train_batch_size
    total = 0.0
    for i in range(nb):
        sl = slice(i * train_batch_size, min((i + 1) * train_batch_size, N))
        if reference_quirks and bool(rewards[sl].all() == 0):
            continue
        H = compute_current_policy_entropy(params, cfg, ids[sl], attn_mask[sl], P, dtype)
        m = answer_mask[sl]
        loss = -entropy_alpha * ((H * m).sum(-1) / m.sum(-1)).mean() / nb
        loss.backward()
        total += loss.item() * nb
    return total


def compute_gradients(params, cfg, ids, attn_mask, answer_mask, rewards, P, train_batch_size, learner, entropy_alpha=0.0,
                      **kw):
    """learner_oracle.compute_gradients with the entropy bonus added: ({name: grad}, loss)."""
    for n in lo.lora_names(cfg):
        params[n].grad = None
    loss = lo.compute_loss(params, cfg, ids, attn_mask, answer_mask, rewards, P, train_batch_size, learner, **kw)
    if entropy_alpha:
        loss += entropy_loss(params, cfg, ids, attn_mask, answer_mask, rewards, P, train_batch_size, entropy_alpha,
                             dtype=kw.get("dtype", torch.float32), reference_quirks=kw.get("reference_quirks", True))
    grads = {n: (params[n].grad.clone() if params[n].grad is not None else torch.zeros_like(params[n]))
             for n in lo.lora_names(cfg)}
    return grads, loss
