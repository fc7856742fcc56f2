/*
 * libb200rl — C ABI of the B200-native GRPO/PG learner hot path.
 *
 * Drop-in boundary for the learner math of BY571/DistRL-LLM (reference @ a1099fd).  The reference
 * has no FFI of its own (pure Python over torch / Unsloth / bitsandbytes); each entry point below
 * names the reference code it replaces (file:line relative to the reference root).  The Python
 * mirror of the reference's Learner / GRPOLearner classes (distrl_llm_b200/learner.py) binds these
 * through ctypes; INTEGRATION.md shows the stub a maintainer would add to distributed_actor.py.
 *
 * Conventions
 *   - every function returns 0 on success, a negative code on failure; b200rl_last_error() returns
 *     a thread-local message.  The Python shim raises RuntimeError, so errors still surface through
 *     ray.get() as RayTaskError like the reference's exceptions do.
 *   - all pointers are DEVICE pointers unless the name ends in _host; the library never allocates
 *     or frees caller-visible memory (exception: b200rl_p2p_alloc, whose buffers must be IPC-exportable).
 *   - `stream` is a cudaStream_t passed as void*; all work is enqueued on it, no hidden syncs.
 *   - bf16 tensors are row-major, 16-byte aligned, leading dimensions multiples of 8.
 */
#ifndef B200RL_H
#define B200RL_H

#ifdef __cplusplus
extern "C" {
#endif

/* ---- runtime ------------------------------------------------------------------------------ */
const char* b200rl_last_error(void);
int b200rl_version(void);
int b200rl_check_device(void); /* 0 iff the current device is sm_100 */

/* ---- G1/G6: tcgen05 GEMM (reference: every nn.Linear / LoRA matmul inside policy(...),
 *      distributed_actor.py:241-243, and their backward, :385 / :483) --------------------------
 * C[M,N] = alpha*(A1[M,K1].B1[N,K1]^T + A2[M,K2].B2[N,K2]^T) (+bias[N]) (+residual[M,N]).
 * mn_major bit0: A stored [K][M]; bit1: B stored [K][N] (read through MN-major UMMA descriptors, no
 * transposes in HBM).  0 = TN (x . W^T), 2 = "dX form" (dY . W, W as stored), 3 = "dW form" (Y^T . U,
 * reduction over tokens); splits>1 writes fp32 partial slabs c_split_stride elements apart.
 * force_bn / max_ctas = 0 for the defaults. */
int b200rl_gemm(const void* A1, long long lda1, const void* B1, long long ldb1, int K1,
                const void* A2, long long lda2, const void* B2, long long ldb2, int K2, void* C,
                long long ldc, int c_fp32, const void* bias, const void* residual, long long ldr,
                float alpha, int M, int N, int mn_major, int splits, long long c_split_stride,
                int force_bn, int max_ctas, void* stream);
/* bisection switch: 1 (default) = CTA-pair (cta_group::2) kernels where applicable, 0 = single-CTA kernels only */
int b200rl_gemm_set_cta_pair(int enable);
/* 1 (default) = the CTA-pair GEMM splits the tiles of its last, partially filled wave along K (gemm2_tcgen05.cu) */
int b200rl_gemm_set_tail_split(int enable);
int b200rl_gemm_set_raster(int gm); /* debug / sweeps: m-blocks per rasterisation group of the CTA-pair GEMM (0 = automatic, gemm_common.cuh raster_group) */
int b200rl_gemm_set_wide(int mode); /* 256 x 512 CTA-pair tiles: 0 never, 1 wherever every pair gets one, 2 (default) only for K-long GEMMs (gemm2_tcgen05.cu) */
/* GEMM with the NF4 base weight dequantised INSIDE the mainloop (north_star; reference: load_in_4bit weights,
 * distributed_actor.py:16-17, :58-66): four producer warps per CTA expand the packed codes of every k-block into the
 * 128B-swizzled shared-memory tile the UMMA reads.  packed / absmax describe W [N, K1] (mn_major 0) or W [K1, N]
 * (mn_major 2) in the layout of b200rl_nf4_quantize.  Bit-identical to b200rl_nf4_dequant + b200rl_gemm. */
int b200rl_gemm_nf4(const void* A1, long long lda1, const void* packed, const float* absmax, int K1, const void* A2,
                    long long lda2, const void* B2, long long ldb2, int K2, void* C, long long ldc, const void* bias,
                    const void* residual, long long ldr, int M, int N, int mn_major, int force_bn, void* stream);
int b200rl_gemm_set_ext(int enable);  /* 1 (default): the model driver computes the LoRA intermediates inside the big GEMMs */
/* Base + LoRA projection in ONE launch (north_star: "LoRA A/B resident in SMEM"): U[M,K2] = ext_alpha * A1.Bext^T is
 * produced by the first work units of the launch ("ext units", one per 256-row block, its own TMEM accumulator) and
 * consumed by the K-extension segment of every tile of that row block: C = A1.B1^T + U.B2^T (+bias) (+residual).
 * mn_major 0 = forward operand layouts (B1 [N,K1], Bext [K2,K1], B2 [N,K2]); 2 = dX form ([K1,N], [K1,K2], [K2,N]).
 * Needs M > 128, N >= 256, K2 in {64, 128}. */
int b200rl_gemm_lora(const void* A1, long long lda1, const void* B1, long long ldb1, int K1, const void* Bext,
                     long long ld_ext, float ext_alpha, void* U, long long ldu, const void* B2, long long ldb2, int K2,
                     void* C, long long ldc, const void* bias, const void* residual, long long ldr, int M, int N,
                     int mn_major, int force_bn, void* stream);
/* G1 + G5 fused (CTA-pair kernel; needs M > 128 and I % 128 == 0, else B200RL_ERR_*):
 * mode 1: gu[M,2I] = A1.B1^T + A2.B2^T (gate rows then up rows of the weight, Qwen2MLP gate_proj|up_proj) and
 *         aux = act[M,I] = silu(gate)*up written by the same epilogue;
 * mode 2: C = dgu[M,2I] from dact = A1.B1 + A2.B2 (B stored [K, I]) and aux = gu[M,2I].
 * Bit-identical to b200rl_gemm followed by b200rl_swiglu_fwd / b200rl_swiglu_bwd. */
int b200rl_gemm_swiglu(int mode, const void* A1, long long lda1, const void* B1, long long ldb1, int K1,
                       const void* A2, long long lda2, const void* B2, long long ldb2, int K2,
                       void* C, long long ldc, void* aux, long long ld_aux, int M, int I, void* stream);
/* G1 grouped dW form (csrc/gemm_dw_grouped.cu): nprob <= 8 independent products C_i = Y_i^T . U_i with the reduction
 * over `tokens` rows, Y_i [tokens, rows_i] (ld ldy_i, rows_i % 8 == 0), U_i [tokens, 64] (ld ldu_i), all bf16 as stored;
 * C_i fp32 [splits][rows_i][64] K-range slabs, split_stride_i elements apart (sum them in order).  One persistent
 * launch.  Returns the number of K-ranges actually written (>= 1), or a negative error code. */
int b200rl_gemm_dw_grouped(int nprob, const void* const* Y, const long long* ldy, const int* rows,
                           const void* const* U, const long long* ldu, float* const* C,
                           const long long* split_stride, int tokens, int splits, void* stream);

/* ---- G2/G3/G5 row kernels (reference: Unsloth RMSNorm / RoPE / SwiGLU inside policy(...)) ---- */
int b200rl_embed(const int* ids, const void* table, void* out, int M, int H, int vocab, void* stream);
int b200rl_rmsnorm_fwd(const void* x, const void* w, void* y, float* rstd, int M, int H, float eps,
                       void* stream);
int b200rl_rmsnorm_bwd(const void* dy, const void* x, const void* w, const float* rstd,
                       const void* dres, void* dx, int M, int H, void* stream);
int b200rl_rope_table(float* cs, int L, int head_dim, float theta, void* stream);
int b200rl_rope(void* qkv, const float* cs, int M, int L, long long row_stride, int n_rot_heads,
                int head_dim, int backward, void* stream);
int b200rl_swiglu_fwd(const void* gu, void* act, int M, int I, void* stream);
int b200rl_swiglu_bwd(const void* gu, const void* dact, void* dgu, int M, int I, void* stream);
/* logits[:, P-1:L-1] row selection of distributed_actor.py:245-249 applied BEFORE lm_head */
int b200rl_gather_rows(const void* x, void* out, int B, int L, int T, int start, int H, void* stream);
int b200rl_scatter_rows(const void* d, void* dx, int B, int L, int T, int start, int H, void* stream);
/* packed layout variants: explicit RoPE positions, indexed gather, CSR scatter-add (fixed order) */
int b200rl_rope_pos(void* qkv, const float* cs, const int* pos, int M, long long row_stride, int n_rot_heads,
                    int head_dim, int backward, void* stream);
int b200rl_gather_rows_idx(const void* x, const int* src, void* out, int R, int H, void* stream);
int b200rl_scatter_add_rows(const void* d, const int* start, const int* list, void* dx, int M, int H, void* stream);

/* ---- G4: causal GQA attention with key-padding mask (reference: attention inside policy(...)
 *      with attention_mask = cat(prompt_mask, answer_mask), distributed_actor.py:236-243) -------- */
int b200rl_attn_fwd(const void* qkv, const int* key_mask, void* out, float* lse, int B, int L,
                    int n_q_heads, int n_kv_heads, int head_dim, float scale, void* stream);
/* bisection switch: 1 (default) = tcgen05/TMEM attention where available (head_dim 128), 0 = mma.sync kernels */
int b200rl_attn_set_prof(void* buf_dev, int which); /* debug: 18 x uint64 per-phase cycle sums of a tcgen05 attention kernel (which: 0 fwd, 1 dQ, 2 dK/dV; NULL = off) */
int b200rl_attn_set_tc(int enable);
int b200rl_attn_bwd(const void* qkv, const int* key_mask, const void* out, const void* dout,
                    const float* lse, float* delta, void* dqkv, int B, int L, int n_q_heads,
                    int n_kv_heads, int head_dim, float scale, void* stream);

/* ---- G4, packed "shared-prompt" layout (head_dim 128): every distinct prompt of a micro-batch is stored once;
 *      completion segments see their prompt segment as a fully visible prefix.  Block descriptors are built on the
 *      host (distrl_llm_b200/packing.py) and passed as device arrays.  lse / delta are [n_q_heads][rows]. */
typedef struct b200rl_attn_qblock {  /* one <=128-query block of a segment (forward and dQ kernels) */
  int q_row0, q_rows;     /* first query row, number of valid query rows */
  int q_local0;           /* index of the first query inside its segment */
  int own_row0, own_len;  /* the segment itself: keys with local index <= query index are visible */
  int pre_row0, pre_len;  /* fully visible prefix (shared prompt), pre_len = 0 for prompt segments */
  int stat0;              /* lse/delta index of (head 0, first query): idx = stat0 + head*rows + r */
} b200rl_attn_qblock;
typedef struct b200rl_attn_kblock {  /* one <=128-key block and ONE query segment that sees it (dK/dV kernel) */
  int k_row0, k_rows, k_local0;
  int q_row0, q_len;      /* the query segment */
  int causal;             /* 1: queries and keys belong to the same segment */
  int stat0;              /* lse/delta index of (head 0, query 0 of the segment) */
  int out_row0;           /* first row of this block's fp32 partial slab */
} b200rl_attn_kblock;
int b200rl_attn_seg_fwd(const void* qkv, const int* key_mask, void* out, float* lse, long long rows,
                        int n_q_heads, int n_kv_heads, float scale, const b200rl_attn_qblock* qblocks_dev,
                        int n_qblocks, void* stream);
int b200rl_attn_seg_bwd(const void* qkv, const int* key_mask, const void* out, const void* dout, const float* lse,
                        float* delta, void* dqkv, float* kv_part, long long rows, int n_q_heads, int n_kv_heads,
                        float scale, const b200rl_attn_qblock* qblocks_dev, int n_qblocks,
                        const b200rl_attn_kblock* kblocks_dev, int n_kblocks, const int* red_start_dev,
                        const int* red_list_dev, void* stream);

/* ---- G7: fused log-softmax + target gather + loss-gradient scale
 *      (distributed_actor.py:252-260 scoring; :375 PG / :467-470 GRPO loss; :382/:479 scaling) --- */
int b200rl_logprob(void* logits, long long ld, const int* targets, const float* coef, float* lp_out,
                   int rows, int V, int write_grad, void* stream);
int b200rl_loss_coef(const int* mask, const double* adv, float* coef, int* lens, int Bm, int T,
                     int nb, void* stream);
int b200rl_loss_value(const float* lp, const int* mask, const double* adv, double* accum, int Bm,
                      int T, int grpo, void* stream);
/* variants with the optional KL(pi || pi_ref) term (k3 estimator exp(q-p)-(q-p)-1 per token, weight beta, same
 * mask / length / batch normalisation as the policy term).  NOT in the reference (its GRPO loss has no KL,
 * distributed_actor.py:467-470): beta = 0 reproduces it exactly; "parity unpinned". */
int b200rl_logprob_kl(void* logits, long long ld, const int* targets, const float* coef, const float* klw,
                      const float* ref_lp, float* lp_out, int rows, int V, int write_grad, void* stream);
int b200rl_loss_coef_kl(const int* mask, const double* adv, float* coef, float* klw, double beta, int* lens,
                        int Bm, int T, int nb, void* stream);
int b200rl_loss_value_kl(const float* lp, const int* mask, const double* adv, const float* ref_lp, double beta,
                         double* accum, int Bm, int T, int grpo, void* stream);

/* clipped-ratio surrogate (SURVEY.md 8(f) N4; the reference's ratio is identically 1, distributed_actor.py:467):
 * old_lp [rows] f32 = log-probs under the policy that generated the batch; clip_eps > 0 turns the per-token loss into
 * -min(rho A, clip(rho, 1-eps, 1+eps) A), rho = exp(lp - old_lp).  old_lp NULL or clip_eps 0 = the plain forms above. */
int b200rl_logprob_clip(void* logits, long long ld, const int* targets, const float* coef, const float* klw,
                        const float* ref_lp, const float* old_lp, double clip_eps, float* lp_out, int rows, int V,
                        int write_grad, void* stream);
/* same with compacted rows: logits / targets hold `rows` live scored rows, slot[rows] maps each to its (i*T + t) entry of
 * the per-token arrays coef / klw / ref_lp / old_lp / lp_out (slot NULL = identity, the call above) */
int b200rl_logprob_slots(void* logits, long long ld, const int* targets, const float* coef, const float* klw,
                         const float* ref_lp, const float* old_lp, double clip_eps, float* lp_out, int rows, int V,
                         int write_grad, const int* slot, void* stream);
int b200rl_loss_value_clip(const float* lp, const int* mask, const double* adv, const float* ref_lp, double beta,
                           const float* old_lp, double clip_eps, double* accum, int Bm, int T, int grpo, void* stream);

/* per-token policy entropy and entropy bonus (reference: BaseLearner.compute_entropy_bonus, distributed_actor.py:266-281,
 * call sites commented out in the PG loss :377-379 and the GRPO loss :472-480).  Same as b200rl_logprob_slots, plus
 *   ent_out [Bm*T] f32 (required): H = -sum_v p_v ln p_v of each scored row, p = softmax(z) at temperature 1, in nats,
 *           written through slot like lp_out;
 *   the bonus gradient e p_v (ln p_v + H) added to dlogits, e = alpha * mask / (len * Bm * nb) from mask [Bm*T] and
 *           lens [Bm] (b200rl_loss_coef*); lens NULL or alpha 0 = no bonus.  alpha > 0 rewards entropy.
 * lp_out is bit-identical to b200rl_logprob_slots'. */
int b200rl_logprob_entropy(void* logits, long long ld, const int* targets, const float* coef, const float* klw,
                           const float* ref_lp, const float* old_lp, double clip_eps, float* lp_out, int rows, int V,
                           int write_grad, const int* slot, const int* mask, const int* lens, int Bm, int T, int nb,
                           double alpha, float* ent_out, void* stream);
/* b200rl_loss_value_clip plus L_H = -alpha (1/Bm) sum_i [len_i>0] (sum_t mask H) / len_i (reference :266-281, :377-379,
 * :472-480); ent [Bm*T] = ent_out above; ent_accum (device f64[2], optional) += {sum mask*H, sum mask}.  One CTA,
 * fixed summation order. */
int b200rl_loss_value_entropy(const float* lp, const int* mask, const double* adv, const float* ref_lp, double beta,
                              const float* old_lp, double clip_eps, double* accum, int Bm, int T, int grpo,
                              const float* ent, double alpha, double* ent_accum, void* stream);

/* ---- G9: group-relative advantages + top-k (distributed_trainer.py:262-294) ---------------- */
int b200rl_group_advantage_topk(const double* rewards, double* values, double* baselines,
                                int* topk_idx, double* topk_val, int G, int C, int k, int grpo,
                                void* stream);

/* ---- NF4 base weights (reference: load_in_4bit=True, distributed_actor.py:16-17, :58-66) ---- */
int b200rl_nf4_quantize(const void* w_bf16, void* packed, float* absmax, long long n, void* stream);
int b200rl_nf4_dequant(const void* packed, const float* absmax, void* out_bf16, int rows, int cols,
                       int transpose, void* stream);

/* ---- G8: (P2P reduce +) Adam/AdamW over the flat LoRA buffer
 *      (distributed_actor.py:283-294 export, :302-333 merge+step, :209-211 optimizer) ----------- */
int b200rl_lora_reduce_adamw(float* p, float* m, float* v, const float* const* grads_host,
                             float* const* params_peer_host, int world, int rank, long long n,
                             int step, float lr, float beta1, float beta2, float eps,
                             float weight_decay, int zero_local_grad, void* stream);
int b200rl_p2p_barrier(unsigned int* const* flags_peer_host, int world, int rank, unsigned int epoch,
                       void* stream);
/* same with an explicit timeout (seconds; <= 0 = env B200RL_P2P_TIMEOUT_S, default 600).  A peer that does not arrive
 * does not trap the context: the waiter records it in a host-visible status word, later reduce kernels become no-ops,
 * and b200rl_p2p_status() returns B200RL_ERR_STATE (reference equivalent: ray.get(..., timeout=240),
 * distributed_trainer.py:200, :333). */
int b200rl_p2p_barrier_timeout(unsigned int* const* flags_peer_host, int world, int rank, unsigned int epoch,
                               double timeout_s, void* stream);
int b200rl_p2p_status(int reset);
int b200rl_p2p_alloc(long long bytes, void** ptr, void* handle64);
int b200rl_p2p_open(const void* handle64, void** ptr);
int b200rl_p2p_close(void* ptr);
int b200rl_p2p_free(void* ptr);
int b200rl_p2p_enable_peer_access(int peer_device); /* same-process learners on different devices (no IPC handle) */
int b200rl_lora_pack(const float* flat, void* arena_bf16, const void* descs_dev, int n_desc,
                     int max_elems, void* stream);
int b200rl_lora_grad_accum(float* flat, const void* descs_dev, int n_desc, int max_elems,
                           void* stream);
int b200rl_sizeof_pack_desc(void);
int b200rl_sizeof_unpack_desc(void);

/* ---- full learner (C++ host driver: 28-layer forward/backward over the kernels above) -------
 *      reference: BaseLearner.compute_current_policy_probs (:215-261), Learner.compute_loss
 *      (:349-395), GRPOLearner.compute_loss (:440-493), loss.backward() (:385, :483) ----------- */
typedef struct b200rl_model_config {
  int vocab, hidden, inter, n_layers, n_q_heads, n_kv_heads, head_dim;
  int lora_r;
  float lora_scale; /* alpha / r */
  float rms_eps;
  float rope_theta;
  int max_tokens; /* largest B*L of a micro-batch the workspace is sized for */
  int max_batch;  /* largest micro-batch (sequences) */
  int max_seq;    /* largest L */
  int max_score_rows; /* largest B*T (rows that reach lm_head) */
} b200rl_model_config;

/* per-layer device pointers (all frozen tensors owned by the caller) */
typedef struct b200rl_layer_weights {
  const void* qkv_packed;  const float* qkv_absmax;   /* NF4 [ (nq+2nkv)*hd, hidden ] */
  const void* o_packed;    const float* o_absmax;     /* NF4 [ hidden, nq*hd ] */
  const void* gu_packed;   const float* gu_absmax;    /* NF4 [ 2*inter, hidden ] (gate rows then up rows) */
  const void* down_packed; const float* down_absmax;  /* NF4 [ hidden, inter ] */
  const void* qkv_bias;                               /* bf16 [ (nq+2nkv)*hd ] */
  const void* ln1_w; const void* ln2_w;               /* bf16 [ hidden ] */
} b200rl_layer_weights;

typedef struct b200rl_model b200rl_model;

long long b200rl_model_workspace_bytes(const b200rl_model_config* cfg);
long long b200rl_model_lora_numel(const b200rl_model_config* cfg);
int b200rl_model_create(const b200rl_model_config* cfg, const b200rl_layer_weights* layers_host,
                        const void* embed, const void* final_norm_w, const void* lm_head,
                        float* lora_flat, float* lora_grad_flat,
                        void* workspace, long long workspace_bytes, b200rl_model** out);
int b200rl_model_destroy(b200rl_model* m);
/* Optional resident bf16 copy of the dequantised NF4 base weights (filled lazily, never invalidated: the base is frozen,
 * bitsandbytes Linear4bit in the reference, distributed_actor.py:125-139). buf = NULL detaches. Results are bit-identical
 * with and without the cache (same dequant kernel, same GEMM operands). */
long long b200rl_model_weight_cache_bytes(const b200rl_model_config* cfg);
int b200rl_model_set_weight_cache(b200rl_model* m, void* buf, long long bytes);
/* bit 0: fuse SwiGLU into the gate|up and down-dX GEMM epilogues (default 1; bit-identical results) */
/* no weight cache attached: 1 = NF4 base weights are dequantised inside the GEMM mainloop (b200rl_gemm_nf4), 0 (default)
 * = into a scratch right before each GEMM.  Measured trade-off: DESIGN.md section 5. */
int b200rl_model_set_nf4_inkernel(b200rl_model* m, int enable);
int b200rl_model_set_fusion(b200rl_model* m, int flags);
/* refresh the bf16 operand copies of the LoRA tensors after an optimizer step */
int b200rl_model_sync_lora(b200rl_model* m, void* stream);
/* one micro-batch: scores B sequences of length L = P+T, accumulates LoRA grads.
 * ids [B,L] int32, attn_mask [B,L] int32 (1 = real token), answer_mask [B,T] int32, adv [B] f64,
 * lp_out [B,T] f32 (per-token log-probs), loss_accum (device f64, += loss_m), nb = number of
 * micro-batches of the step (1/nb scaling, distributed_actor.py:382/:479). backward=0 scores only. */
/* device pointer of a named activation buffer (parity bisection in tests; NULL if unknown) */
void* b200rl_model_debug_ptr(b200rl_model* m, const char* name, int layer);
int b200rl_model_microbatch(b200rl_model* m, const int* ids, const int* attn_mask,
                            const int* answer_mask, const double* adv, float* lp_out,
                            double* loss_accum, int B, int P, int T, int nb, int grpo, int backward,
                            void* stream);

/* extended form: lora_off=1 runs the adapter-disabled forward (reference policy pi_ref, scoring only);
 * ref_lp [B,T] + kl_beta add the KL term to the loss and its gradient. */
int b200rl_model_microbatch_ex(b200rl_model* m, const int* ids, const int* attn_mask,
                               const int* answer_mask, const double* adv, float* lp_out,
                               double* loss_accum, int B, int P, int T, int nb, int grpo, int backward,
                               int lora_off, const float* ref_lp, double kl_beta, void* stream);

/* packed ("shared-prompt") micro-batch: all arrays are device int32 built by distrl_llm_b200/packing.py */
typedef struct b200rl_packed_batch {
  int rows;        /* G*P + B*T packed token rows */
  int B, T;        /* sequences, scored positions per sequence */
  int max_pos;     /* P + T (RoPE table length) */
  int n_qblocks, n_kblocks;
  int part_rows;   /* rows of the fp32 dK/dV partial buffer */
  const int* ids;          /* [rows] */
  const int* pos;          /* [rows] position of the token in its original sequence */
  const int* key_mask;     /* [rows] 1 = real token */
  const int* score_src;    /* [n_score] packed row whose hidden state predicts completion token (i, t) */
  const int* targets;      /* [n_score] completion token ids */
  const int* answer_mask;  /* [B*T] */
  const int* sc_start;     /* [rows+1] CSR: scored rows fed by each packed row */
  const int* sc_list;
  const b200rl_attn_qblock* qblocks;
  const b200rl_attn_kblock* kblocks;
  const int* red_start;    /* [rows+1] CSR: dK/dV partial rows of each packed row */
  const int* red_list;
  /* live scored rows only (distributed_actor.py:245-260 scores all T positions and masks afterwards; positions with
   * answer_mask 0 carry no loss and no gradient, so the final norm / lm_head / log-softmax / lm_head dX run on the
   * n_score <= B*T live ones): score_slot[n_score] = i*T + t of each scored row.  n_score 0 / score_slot NULL = all
   * B*T positions in slot order.  Log-probs of the positions left out are reported as 0. */
  int n_score;
  const int* score_slot;
} b200rl_packed_batch;
/* same contract as b200rl_model_microbatch_ex on the packed layout (head_dim 128 only) */
int b200rl_model_microbatch_packed(b200rl_model* m, const b200rl_packed_batch* pb, const double* adv, float* lp_out,
                                   double* loss_accum, int nb, int grpo, int backward, int lora_off,
                                   const float* ref_lp, double kl_beta, void* stream);

/* General form of the two calls above: every optional term of the loss in one argument block.
 *   lora_off   adapter-disabled scoring pass (pi_ref); forward only
 *   ref_lp / kl_beta     KL(pi || pi_ref) term, k3 estimator (north_star; absent from the reference)
 *   old_lp / clip_eps    clipped-ratio surrogate against the generating policy's log-probs (SURVEY.md 8(f) N4)
 * ref_lp / old_lp are [B*T] f32 device arrays or NULL.  All zero / NULL = exactly the reference's loss
 * (distributed_actor.py:375, :467-470). */
typedef struct b200rl_loss_args {
  int nb, grpo, backward, lora_off;
  const float* ref_lp;
  double kl_beta;
  const float* old_lp;
  double clip_eps;
} b200rl_loss_args;
int b200rl_model_pass(b200rl_model* m, const int* ids, const int* attn_mask, const int* answer_mask, const double* adv,
                      float* lp_out, double* loss_accum, int B, int P, int T, const b200rl_loss_args* args, void* stream);
int b200rl_model_pass_packed(b200rl_model* m, const b200rl_packed_batch* pb, const double* adv, float* lp_out,
                             double* loss_accum, const b200rl_loss_args* args, void* stream);
/* Entropy of the policy and entropy bonus (reference: compute_entropy_bonus, distributed_actor.py:266-281; call sites
 * commented out at :377-379 and :472-480; config key commented out at :437).
 *   alpha      bonus weight: loss -= alpha * mean_i( sum_t mask H / len_i ) per micro-batch; > 0 rewards entropy
 *   ent_out    [B*T] f32 device: per-token entropy in nats (0 for positions left out of compact scoring); required
 *              whenever alpha != 0 or ent_accum is set
 *   ent_accum  device f64[2] or NULL: += {sum mask*H, sum mask} of the pass (passes that compute a loss value only)
 * args NULL in the calls below = b200rl_model_pass / b200rl_model_pass_packed. */
typedef struct b200rl_entropy_args {
  double alpha;
  float* ent_out;
  double* ent_accum;
} b200rl_entropy_args;
int b200rl_model_pass_ent(b200rl_model* m, const int* ids, const int* attn_mask, const int* answer_mask,
                          const double* adv, float* lp_out, double* loss_accum, int B, int P, int T,
                          const b200rl_loss_args* args, const b200rl_entropy_args* ent, void* stream);
int b200rl_model_pass_packed_ent(b200rl_model* m, const b200rl_packed_batch* pb, const double* adv, float* lp_out,
                                 double* loss_accum, const b200rl_loss_args* args, const b200rl_entropy_args* ent,
                                 void* stream);

/* per-op CUDA-event profiling of the driver (categories: 0 gemm, 1 skinny LoRA gemm, 2 dW gemm, 3 nf4
 * dequant, 4 attn fwd, 5 attn bwd, 6 row kernels, 7 logprob, 8 misc); read() returns sums since the last
 * read: ms[9], work[9] (algorithmic flops or bytes), count[9]. */
int b200rl_model_profile(b200rl_model* m, int enable);
int b200rl_model_profile_read(b200rl_model* m, double* ms, double* work, long long* count);
long long b200rl_launch_count(void); /* kernels launched by the library so far */
/* 1 (default; env B200RL_PDL=0): hot-path kernels are launched with programmatic dependent launch, so that each
 * kernel's prologue overlaps the previous kernel's tail (csrc/common.cuh). Results are unaffected. */
int b200rl_set_pdl(int enable);

#ifdef __cplusplus
}
#endif
#endif /* B200RL_H */
