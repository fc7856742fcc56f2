"""Device-resident state of one learner: NF4 base weights, flat fp32 LoRA parameters / gradients /
Adam moments, the workspace, and the handle of the C++ model driver (csrc/model.cu).

Plays the role of `self.policy` + `self.optimizer` in the reference's BaseLearner
(distributed_actor.py:50-82, :209-211) — but every tensor op goes through libb200rl (no torch math).
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass

import torch

from . import _capi, ops
from ._capi import LayerWeights, ModelConfig, check, lib, ptr, stream

LORA_MODULES = ("q", "k", "v", "o", "gate", "up", "down")  # reference helper.py:29-37
_PEFT = {"q": "self_attn.q_proj", "k": "self_attn.k_proj", "v": "self_attn.v_proj", "o": "self_attn.o_proj",
         "gate": "mlp.gate_proj", "up": "mlp.up_proj", "down": "mlp.down_proj"}


@dataclass
class LMConfig:
    vocab: int
    hidden: int
    inter: int
    n_layers: int
    n_q_heads: int
    n_kv_heads: int
    head_dim: int
    lora_r: int = 16
    lora_alpha: float = 16.0
    rms_eps: float = 1e-6
    rope_theta: float = 1e6

    @property
    def lora_scale(self):
        return self.lora_alpha / self.lora_r

    @property
    def qd(self):
        return self.n_q_heads * self.head_dim

    @property
    def kd(self):
        return self.n_kv_heads * self.head_dim

    def module_shapes(self):
        H, I = self.hidden, self.inter
        return {"q": (H, self.qd), "k": (H, self.kd), "v": (H, self.kd), "o": (self.qd, H),
                "gate": (H, I), "up": (H, I), "down": (I, H)}

    @staticmethod
    def from_hf_config(hf, lora_r=16, lora_alpha=16.0):
        """From a transformers Qwen2Config-like object or dict (config.json of the checkpoint the reference loads,
        distributed_actor.py:58-66)."""
        g = (lambda k, d=None: hf.get(k, d)) if isinstance(hf, dict) else (lambda k, d=None: getattr(hf, k, d))
        nq = g("num_attention_heads")
        hd = g("head_dim") or g("hidden_size") // nq
        theta = g("rope_theta")
        if theta is None and g("rope_parameters"):
            rp = g("rope_parameters")
            theta = rp.get("rope_theta") if isinstance(rp, dict) else getattr(rp, "rope_theta", None)
        return LMConfig(vocab=g("vocab_size"), hidden=g("hidden_size"), inter=g("intermediate_size"),
                        n_layers=g("num_hidden_layers"), n_q_heads=nq, n_kv_heads=g("num_key_value_heads") or nq,
                        head_dim=hd, lora_r=lora_r, lora_alpha=lora_alpha, rms_eps=g("rms_norm_eps", 1e-6),
                        rope_theta=float(theta or 1e6))

    @staticmethod
    def qwen25_7b(lora_r=16, lora_alpha=16.0):
        return LMConfig(vocab=152064, hidden=3584, inter=18944, n_layers=28, n_q_heads=28, n_kv_heads=4,
                        head_dim=128, lora_r=lora_r, lora_alpha=lora_alpha)


class LoraLayout:
    """Names and offsets of every LoRA tensor inside the flat fp32 buffer, without a model behind it (what a generator
    needs to view a pulled adapter under PEFT names; csrc/model.cu build_groups() is the authority for the order:
    for layer: for module in (q,k,v,o,gate,up,down): A [r, in] then B [out, r]; total padded to a multiple of 4)."""

    def __init__(self, cfg: "LMConfig"):
        self.cfg = cfg
        self.offsets = {}
        off = 0
        shapes = cfg.module_shapes()
        for i in range(cfg.n_layers):
            for m in LORA_MODULES:
                fin, fout = shapes[m]
                self.offsets[(i, m, "A")] = (off, (cfg.lora_r, fin)); off += cfg.lora_r * fin
                self.offsets[(i, m, "B")] = (off, (fout, cfg.lora_r)); off += fout * cfg.lora_r
        self.numel = (off + 3) // 4 * 4

    @staticmethod
    def peft_name(i, m, ab):
        return f"base_model.model.model.layers.{i}.{_PEFT[m]}.lora_{ab}.default.weight"

    def named_views(self, flat):
        return {self.peft_name(i, m, ab): flat[off:off + shp[0] * shp[1]].view(*shp)
                for (i, m, ab), (off, shp) in self.offsets.items()}


class _RawCuda:
    """Wrap a raw device pointer (library-owned, e.g. an IPC-mapped peer buffer) as a torch tensor."""

    def __init__(self, ptr_, nbytes):
        self.__cuda_array_interface__ = {"shape": (nbytes,), "typestr": "|u1", "data": (int(ptr_), False), "version": 2}


def tensor_from_ptr(ptr_, numel, dtype, device):
    nbytes = numel * torch.empty((), dtype=dtype).element_size()
    return torch.as_tensor(_RawCuda(ptr_, nbytes), device=device).view(dtype)


def workspace_bytes(cfg: "LMConfig", max_batch, P, T):
    """Activation workspace a Policy(cfg, max_batch, P, T) allocates (b200rl_model_workspace_bytes; host-only call)."""
    _capi.load_library()
    L = P + T
    ccfg = ModelConfig(cfg.vocab, cfg.hidden, cfg.inter, cfg.n_layers, cfg.n_q_heads, cfg.n_kv_heads, cfg.head_dim,
                       cfg.lora_r, cfg.lora_scale, cfg.rms_eps, cfg.rope_theta, max_batch * L, max_batch, L, max_batch * T)
    return int(lib().b200rl_model_workspace_bytes(C.byref(ccfg)))


def largest_pass_that_fits(cfg: "LMConfig", micro_batch, P, T, want, free_bytes, reserve_bytes=0):
    """Largest k <= want such that the workspace of k micro-batches per pass fits in 80 % of what is left of
    free_bytes after reserve_bytes (weights, cache, optimizer state)."""
    k = max(1, int(want))
    while k > 1 and workspace_bytes(cfg, k * micro_batch, P, T) > 0.8 * (free_bytes - reserve_bytes):
        k -= 1
    return k


class Policy:
    """NF4 base + LoRA causal LM on one GPU. `lora_flat` layout (fp32), matching csrc/model.cu:
    for layer in layers: for mod in (q,k,v,o,gate,up,down): A [r, in] then B [out, r]."""

    def __init__(self, cfg: LMConfig, device, max_batch, max_prompt_tokens, max_new_tokens,
                 lora_flat=None, lora_grad=None, cache_weights="auto"):
        _capi.load_library()
        check(lib().b200rl_check_device(), "check_device")
        self.cfg = cfg
        self.device = torch.device(device)
        self.max_batch, self.P, self.T = max_batch, max_prompt_tokens, max_new_tokens
        L = max_prompt_tokens + max_new_tokens
        self.ccfg = ModelConfig(cfg.vocab, cfg.hidden, cfg.inter, cfg.n_layers, cfg.n_q_heads, cfg.n_kv_heads,
                                cfg.head_dim, cfg.lora_r, cfg.lora_scale, cfg.rms_eps, cfg.rope_theta,
                                max_batch * L, max_batch, L, max_batch * max_new_tokens)
        n = lib().b200rl_model_lora_numel(C.byref(self.ccfg))
        if n <= 0:
            raise RuntimeError("libb200rl: " + lib().b200rl_last_error().decode())
        self.lora_numel = int(n)
        f32 = dict(device=self.device, dtype=torch.float32)
        self.lora_flat = lora_flat if lora_flat is not None else torch.zeros(n, **f32)
        self.lora_grad = lora_grad if lora_grad is not None else torch.zeros(n, **f32)
        self.adam_m = torch.zeros(n, **f32)
        self.adam_v = torch.zeros(n, **f32)
        self.opt_step = 0
        self.layers = []      # per layer dict of device tensors
        self.embed = self.final_norm = self.lm_head = None
        self.handle = None
        self.workspace = None
        self.cache_weights = cache_weights   # True / False / "auto": resident bf16 copy of the dequantised base; "inkernel": no copy at all
        self.weight_cache = None
        self.loss_accum = torch.zeros(1, device=self.device, dtype=torch.float64)
        # offsets of every LoRA tensor in the flat buffer
        self.offsets = {}
        off = 0
        shapes = cfg.module_shapes()
        for i in range(cfg.n_layers):
            for m in LORA_MODULES:
                fin, fout = shapes[m]
                self.offsets[(i, m, "A")] = (off, (cfg.lora_r, fin)); off += cfg.lora_r * fin
                self.offsets[(i, m, "B")] = (off, (fout, cfg.lora_r)); off += fout * cfg.lora_r
        assert off <= self.lora_numel

    # ---- construction ------------------------------------------------------------------------
    def _finish(self):
        cfg = self.cfg
        wl = (LayerWeights * cfg.n_layers)()
        for i, L in enumerate(self.layers):
            wl[i] = LayerWeights(ptr(L["qkv_p"]), ptr(L["qkv_a"]), ptr(L["o_p"]), ptr(L["o_a"]),
                                 ptr(L["gu_p"]), ptr(L["gu_a"]), ptr(L["down_p"]), ptr(L["down_a"]),
                                 ptr(L["qkv_bias"]), ptr(L["ln1"]), ptr(L["ln2"]))
        nbytes = lib().b200rl_model_workspace_bytes(C.byref(self.ccfg))
        if nbytes <= 0:
            raise RuntimeError("libb200rl: " + lib().b200rl_last_error().decode())
        self.workspace = torch.empty(int(nbytes) + 1024, device=self.device, dtype=torch.uint8)
        base = self.workspace.data_ptr()
        aligned = (base + 1023) // 1024 * 1024
        h = C.c_void_p()
        check(lib().b200rl_model_create(C.byref(self.ccfg), wl, ptr(self.embed), ptr(self.final_norm),
                                        ptr(self.lm_head), ptr(self.lora_flat),
                                        ptr(self.lora_grad), aligned, int(nbytes), C.byref(h)), "model_create")
        self.handle = h
        self._attach_weight_cache()
        self.sync_lora()

    def _attach_weight_cache(self):
        """Keep the dequantised base resident in HBM when it fits comfortably ("auto": cache <= 1/3 of the free
        memory).  The NF4 tensors stay the source of truth; the cache only removes the per-micro-batch dequant passes."""
        want = self.cache_weights
        if want == "inkernel":   # no cache: the GEMMs expand the NF4 codes inside their mainloop (north_star)
            check(lib().b200rl_model_set_nf4_inkernel(self.handle, 1), "model_set_nf4_inkernel")
            return
        need = int(lib().b200rl_model_weight_cache_bytes(C.byref(self.ccfg)))
        if want == "auto":
            free, _ = torch.cuda.mem_get_info(self.device)
            want = need * 3 <= free
        if not want:
            return
        self.weight_cache = torch.empty(need + 1024, device=self.device, dtype=torch.uint8)
        base = self.weight_cache.data_ptr()
        check(lib().b200rl_model_set_weight_cache(self.handle, (base + 1023) // 1024 * 1024, need), "model_set_weight_cache")

    def __del__(self):
        try:
            if self.handle:
                lib().b200rl_model_destroy(self.handle)
                self.handle = None
        except Exception:
            pass

    @classmethod
    def random_init(cls, cfg: LMConfig, device, max_batch, P, T, seed=1234, lora_b_std=0.01, **kw):
        """Random-init weights of the given architecture, generated and NF4-quantised on the GPU
        (SURVEY.md §8d synthetic inputs: base N(0, 0.02^2), LoRA A kaiming-uniform, B ~ N(0, 0.01^2))."""
        self = cls(cfg, device, max_batch, P, T, **kw)
        g = torch.Generator(device=self.device).manual_seed(seed)
        bf = dict(device=self.device, dtype=torch.bfloat16)

        def rnd(*shape, std=0.02):
            return (torch.randn(*shape, generator=g, device=self.device) * std).to(torch.bfloat16)

        def quant(rows, cols):
            w = rnd(rows, cols)
            p, a = ops.nf4_quantize(w)
            return p, a

        H, I = cfg.hidden, cfg.inter
        self.embed = rnd(cfg.vocab, H)
        self.lm_head = rnd(cfg.vocab, H)
        self.final_norm = torch.ones(H, **bf)
        for _ in range(cfg.n_layers):
            L = {}
            L["qkv_p"], L["qkv_a"] = quant(cfg.qd + 2 * cfg.kd, H)
            L["o_p"], L["o_a"] = quant(H, cfg.qd)
            L["gu_p"], L["gu_a"] = quant(2 * I, H)
            L["down_p"], L["down_a"] = quant(H, I)
            L["qkv_bias"] = rnd(cfg.qd + 2 * cfg.kd)
            L["ln1"] = torch.ones(H, **bf)
            L["ln2"] = torch.ones(H, **bf)
            self.layers.append(L)
        shapes = cfg.module_shapes()
        for (i, m, ab), (off, shp) in self.offsets.items():
            fin, fout = shapes[m]
            n = shp[0] * shp[1]
            if ab == "A":
                bound = fin ** -0.5
                v = (torch.rand(n, generator=g, device=self.device) * 2 - 1) * bound
            else:
                v = torch.randn(n, generator=g, device=self.device) * lora_b_std
            self.lora_flat[off:off + n] = v.to(torch.bfloat16).float()
        self._finish()
        return self

    @classmethod
    def from_params(cls, cfg: LMConfig, params: dict, nf4: dict, device, max_batch, P, T, **kw):
        """Build from a named-tensor dict (the oracle's / golden fixtures' naming): dense tensors for
        embed / lm_head / norms / biases / LoRA, and nf4[name] = (packed uint8, absmax f32) numpy arrays
        for each base matrix 'l{i}.wq' ... The fused qkv / gate|up matrices are row concatenations, and
        NF4 blocks (64 consecutive values of a row-major matrix) never straddle rows (in % 64 == 0)."""
        import numpy as np
        self = cls(cfg, device, max_batch, P, T, **kw)
        dev = self.device

        def bf(t):
            return torch.as_tensor(t).to(dev, torch.bfloat16).contiguous()

        def cat_nf4(names):
            p = np.concatenate([nf4[n][0] for n in names])
            a = np.concatenate([nf4[n][1] for n in names])
            return torch.from_numpy(p).to(dev), torch.from_numpy(a.astype(np.float32)).to(dev)

        self.embed = bf(params["embed"])
        self.lm_head = bf(params["lm_head"])
        self.final_norm = bf(params["final_norm"])
        for i in range(cfg.n_layers):
            L = {}
            L["qkv_p"], L["qkv_a"] = cat_nf4([f"l{i}.wq", f"l{i}.wk", f"l{i}.wv"])
            L["o_p"], L["o_a"] = cat_nf4([f"l{i}.wo"])
            L["gu_p"], L["gu_a"] = cat_nf4([f"l{i}.wg", f"l{i}.wu"])
            L["down_p"], L["down_a"] = cat_nf4([f"l{i}.wd"])
            L["qkv_bias"] = bf(torch.cat([torch.as_tensor(params[f"l{i}.b{x}"]).float() for x in "qkv"]))
            L["ln1"] = bf(params[f"l{i}.ln1"])
            L["ln2"] = bf(params[f"l{i}.ln2"])
            self.layers.append(L)
        for (i, m, ab), (off, shp) in self.offsets.items():
            t = torch.as_tensor(params[f"l{i}.{m}.{ab}"]).detach().float().reshape(-1)
            self.lora_flat[off:off + t.numel()] = t.to(dev)
        self._finish()
        return self

    @classmethod
    def from_hf_state_dict(cls, cfg: LMConfig, sd: dict, device, max_batch, P, T, lora_seed=0, lora_state=None, **kw):
        """Build from a Hugging Face Qwen2-family state dict (`model.layers.{i}.self_attn.q_proj.weight`, ...), dense
        bf16/fp16/fp32 tensors.  The seven linear weights of every layer are NF4-quantised ON THE GPU at load time
        (blocksize 64, fp32 absmax) -- what `load_in_4bit=True` does in the reference (distributed_actor.py:58-66) -- and
        fused row-wise into qkv / gate|up.  LoRA: PEFT's default init (A kaiming-uniform(a=sqrt 5) = U(+-1/sqrt(in)),
        B = 0) from `lora_seed`, or `lora_state` = {PEFT name: tensor} (see peft_name) to resume an adapter."""
        self = cls(cfg, device, max_batch, P, T, **kw)
        dev = self.device

        def get(name):
            if name not in sd:
                raise KeyError(f"state dict has no '{name}'")
            return sd[name]

        def bf(t):
            return t.detach().to(dev, torch.bfloat16).contiguous()

        def quant(names):
            w = torch.cat([bf(get(n)) for n in names], dim=0).contiguous()
            if w.shape[1] % 64:
                raise ValueError(f"{names[0]}: in_features {w.shape[1]} is not a multiple of the NF4 block (64)")
            return ops.nf4_quantize(w)

        self.embed = bf(get("model.embed_tokens.weight"))
        self.lm_head = bf(sd["lm_head.weight"]) if "lm_head.weight" in sd else self.embed   # tied embeddings
        self.final_norm = bf(get("model.norm.weight"))
        if tuple(self.embed.shape) != (cfg.vocab, cfg.hidden):
            raise ValueError(f"embed_tokens is {tuple(self.embed.shape)}, config says {(cfg.vocab, cfg.hidden)}")
        for i in range(cfg.n_layers):
            a, m = f"model.layers.{i}.self_attn.", f"model.layers.{i}.mlp."
            L = {}
            L["qkv_p"], L["qkv_a"] = quant([a + "q_proj.weight", a + "k_proj.weight", a + "v_proj.weight"])
            L["o_p"], L["o_a"] = quant([a + "o_proj.weight"])
            L["gu_p"], L["gu_a"] = quant([m + "gate_proj.weight", m + "up_proj.weight"])
            L["down_p"], L["down_a"] = quant([m + "down_proj.weight"])
            if a + "q_proj.bias" in sd:
                L["qkv_bias"] = torch.cat([bf(get(a + x + "_proj.bias")) for x in "qkv"]).contiguous()
            else:   # Llama-style: no qkv bias
                L["qkv_bias"] = torch.zeros(cfg.qd + 2 * cfg.kd, device=dev, dtype=torch.bfloat16)
            L["ln1"] = bf(get(f"model.layers.{i}.input_layernorm.weight"))
            L["ln2"] = bf(get(f"model.layers.{i}.post_attention_layernorm.weight"))
            self.layers.append(L)
        g = torch.Generator(device=dev).manual_seed(lora_seed)
        shapes = cfg.module_shapes()
        for (i, mod, ab), (off, shp) in self.offsets.items():
            n = shp[0] * shp[1]
            if lora_state is not None:
                t = lora_state[self.peft_name(i, mod, ab)].detach().float().reshape(-1)
                assert t.numel() == n, (self.peft_name(i, mod, ab), tuple(t.shape), shp)
                self.lora_flat[off:off + n] = t.to(dev)
            elif ab == "A":
                bound = shapes[mod][0] ** -0.5
                self.lora_flat[off:off + n] = (torch.rand(n, generator=g, device=dev) * 2 - 1) * bound
        self._finish()
        return self

    @classmethod
    def from_pretrained(cls, path, device, max_batch, P, T, lora_r=16, lora_alpha=16.0, **kw):
        """Local checkpoint directory with config.json + *.safetensors (dense weights).  Returns (policy, cfg)."""
        import glob
        import json
        import os
        from safetensors.torch import load_file
        cfg = LMConfig.from_hf_config(json.load(open(os.path.join(path, "config.json"))), lora_r, lora_alpha)
        sd = {}
        files = sorted(glob.glob(os.path.join(path, "*.safetensors")))
        if not files:
            raise FileNotFoundError(f"no *.safetensors under {path}")
        for f in files:
            sd.update(load_file(f))
        return cls.from_hf_state_dict(cfg, sd, device, max_batch, P, T, **kw), cfg

    # ---- hot path ------------------------------------------------------------------------------
    def sync_lora(self):
        check(lib().b200rl_model_sync_lora(self.handle, stream()), "model_sync_lora")

    @staticmethod
    def _loss_args(nb, grpo, backward, lora_off, ref_lp, kl_beta, old_lp, clip_eps):
        return _capi.LossArgs(int(nb), 1 if grpo else 0, 1 if backward else 0, 1 if lora_off else 0, ptr(ref_lp),
                              float(kl_beta), ptr(old_lp), float(clip_eps))

    @staticmethod
    def _entropy_args(entropy_alpha, ent_out, ent_accum):
        if not entropy_alpha and ent_out is None and ent_accum is None:
            return None
        return _capi.EntropyArgs(float(entropy_alpha), ptr(ent_out), ptr(ent_accum))

    def microbatch(self, ids, attn_mask, answer_mask, adv, P, T, nb, grpo, backward, lp_out=None,
                   lora_off=False, ref_lp=None, kl_beta=0.0, old_lp=None, clip_eps=0.0, entropy_alpha=0.0, ent_out=None,
                   ent_accum=None):
        """One micro-batch through the C++ driver. ids/attn_mask [B, P+T] int32, answer_mask [B,T] int32,
        adv [B] float64 (all on this device). Accumulates into lora_grad and self.loss_accum.
        lora_off: adapter-disabled scoring pass (reference policy); ref_lp + kl_beta: optional KL term;
        old_lp [B,T] + clip_eps: optional clipped-ratio surrogate (b200rl_loss_args);
        ent_out [B,T] f32: per-token entropy; entropy_alpha: entropy bonus weight (needs ent_out); ent_accum f64[2]:
        += {sum mask*H, sum mask} (b200rl_entropy_args)."""
        B = ids.shape[0]
        a = self._loss_args(nb, grpo, backward, lora_off, ref_lp, kl_beta, old_lp, clip_eps)
        e = self._entropy_args(entropy_alpha, ent_out, ent_accum)
        if e is None:
            check(lib().b200rl_model_pass(self.handle, ptr(ids), ptr(attn_mask), ptr(answer_mask), ptr(adv), ptr(lp_out),
                                          ptr(self.loss_accum), B, P, T, C.byref(a), stream()), "model_pass")
            return
        check(lib().b200rl_model_pass_ent(self.handle, ptr(ids), ptr(attn_mask), ptr(answer_mask), ptr(adv), ptr(lp_out),
                                          ptr(self.loss_accum), B, P, T, C.byref(a), C.byref(e), stream()), "model_pass_ent")

    def microbatch_packed(self, packed, adv, nb, grpo, backward, lp_out=None, lora_off=False, ref_lp=None,
                          kl_beta=0.0, old_lp=None, clip_eps=0.0, entropy_alpha=0.0, ent_out=None, ent_accum=None):
        """Same as microbatch() on the packed shared-prompt layout (`packed`: packing.PackedDevice)."""
        a = self._loss_args(nb, grpo, backward, lora_off, ref_lp, kl_beta, old_lp, clip_eps)
        e = self._entropy_args(entropy_alpha, ent_out, ent_accum)
        if e is None:
            check(lib().b200rl_model_pass_packed(self.handle, C.byref(packed.c), ptr(adv), ptr(lp_out),
                                                 ptr(self.loss_accum), C.byref(a), stream()), "model_pass_packed")
            return
        check(lib().b200rl_model_pass_packed_ent(self.handle, C.byref(packed.c), ptr(adv), ptr(lp_out), ptr(self.loss_accum),
                                                 C.byref(a), C.byref(e), stream()), "model_pass_packed_ent")

    def debug_tensor(self, name, layer, shape, dtype=torch.bfloat16):
        p = lib().b200rl_model_debug_ptr(self.handle, name.encode(), layer)
        if not p:
            raise KeyError(name)
        n = 1
        for s in shape:
            n *= s
        return tensor_from_ptr(p, n, dtype, self.device).view(*shape)

    def zero_grad(self):
        self.lora_grad.zero_()

    def optimizer_step(self, lr, betas=(0.9, 0.999), eps=1e-8, weight_decay=0.0):
        """Single-learner fused Adam(W) + zero_grad + refresh of the bf16 LoRA operand copies
        (reference: optimizer.step(); optimizer.zero_grad(), distributed_actor.py:414-415 / :512-513)."""
        self.opt_step += 1
        ops.adamw_step(self.lora_flat, self.adam_m, self.adam_v, self.lora_grad, self.opt_step, lr,
                       betas[0], betas[1], eps, weight_decay, zero_grad=True)
        self.sync_lora()

    # ---- naming (T2: gradient / state dict keyed by PEFT names) -------------------------------------
    @staticmethod
    def peft_name(i, m, ab):
        return f"base_model.model.model.layers.{i}.{_PEFT[m]}.lora_{ab}.default.weight"

    def named_views(self, flat):
        """{PEFT name: view into `flat`} for every LoRA tensor."""
        out = {}
        for (i, m, ab), (off, shp) in self.offsets.items():
            out[self.peft_name(i, m, ab)] = flat[off:off + shp[0] * shp[1]].view(*shp)
        return out

    def load_lora_state(self, state: dict):
        """Copy {PEFT name: tensor} into the flat fp32 master buffer (every LoRA tensor must be present, shapes must
        match) and refresh the bf16 operand copies."""
        views = self.named_views(self.lora_flat)
        missing = [k for k in views if k not in state]
        if missing:
            raise KeyError(f"adapter state lacks {len(missing)} tensors, e.g. {missing[0]}")
        for k, v in views.items():
            t = state[k]
            if tuple(t.shape) != tuple(v.shape):
                raise ValueError(f"{k}: shape {tuple(t.shape)} != {tuple(v.shape)}")
            v.copy_(t.to(device=v.device, dtype=torch.float32))
        self.sync_lora()

    def lora_state_dict(self):
        return {k: v.detach().cpu().clone() for k, v in self.named_views(self.lora_flat).items()}
