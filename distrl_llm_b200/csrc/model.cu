// C++ host driver of the learner hot path: Qwen2-style causal LM (NF4 base + LoRA on
// q,k,v,o,gate,up,down) forward -> per-token log-probs -> PG/GRPO loss -> backward into the flat
// fp32 LoRA gradient buffer.  One call = one pass over k micro-batches of the reference's hot loop, in the classic
// [B, P+T] layout (b200rl_model_microbatch) or the packed shared-prompt / ragged layout built by
// distrl_llm_b200/packing.py (b200rl_model_microbatch_packed).
//
// Reference being replaced (file:line in /root/reference):
//   BaseLearner.compute_current_policy_probs   distributed_actor.py:215-261
//     :233-239  full_inputs / full_attention_mask  -> ids [B,L], attn_mask [B,L] (L = P+T)
//     :241-243  policy(...).logits                 -> layer loop below (lm_head only at the T scored rows)
//     :245-249  shift / slice                      -> rows P-1..L-2 predict tokens P..L-1
//     :252-260  log_softmax + gather               -> b200rl logprob kernel (G7)
//   Learner.compute_loss :375 / GRPOLearner.compute_loss :467-470, :382/:479 (1/num_batches),
//   loss.backward() :385/:483                      -> analytic backward below (store, no recompute)
//   LoRA spec helper.py:25-45 (7 target modules, bias none, dropout 0)
//
// LoRA math per projection: y = x W^T + s (x A^T) B^T, s = alpha/r.  Fused groups (qkv, o, gate|up,
// down) use block-structured operand copies so one GEMM mainloop covers base + LoRA:
//   Acat [K2, Kin] (A_j stacked, zero padded to K2 = roundup(nproj*r, 64)),  Bcat [Nout, K2]
//   (block diagonal).  Backward GEMMs read W / Acat / Bcat as stored through MN-major UMMA descriptors
//   (no transposed copies, no transposed dequant).
#include <stdlib.h>
#include "gemm_common.cuh"
#include "b200rl.h"
#include <vector>
#include <string.h>
#include <new>

namespace b200rl {

// from the other translation units (GemmArgs / gemm_fuse_supported: gemm_common.cuh)
int gemm_dispatch(const GemmArgs& a, cudaStream_t stream);
int dw_grouped_splits(int total_m_blocks, int kb_total);
int dw_grouped_dispatch(int nprob, const void* const* Y, const long long* ldy, const int* rows, const void* const* U,
                        const long long* ldu, float* const* C, const long long* split_stride, int tokens, int splits,
                        cudaStream_t stream);

}  // namespace b200rl

using namespace b200rl;

extern "C" {
int b200rl_embed(const int*, const void*, void*, int, int, int, void*);
int b200rl_rmsnorm_fwd(const void*, const void*, void*, float*, int, int, float, void*);
int b200rl_rmsnorm_bwd(const void*, const void*, const void*, const float*, const void*, void*, int, int, void*);
int b200rl_rope_table(float*, int, int, float, void*);
int b200rl_rope(void*, const float*, int, int, long long, int, int, int, void*);
int b200rl_swiglu_fwd(const void*, void*, int, int, void*);
int b200rl_swiglu_bwd(const void*, const void*, void*, int, int, void*);
int b200rl_gather_rows(const void*, void*, int, int, int, int, int, void*);
int b200rl_scatter_rows(const void*, void*, int, int, int, int, int, void*);
int b200rl_attn_fwd(const void*, const int*, void*, float*, int, int, int, int, int, float, void*);
int b200rl_attn_bwd(const void*, const int*, const void*, const void*, const float*, float*, void*, int, int, int, int, int, float, void*);
int b200rl_logprob(void*, long long, const int*, const float*, float*, int, int, int, void*);
int b200rl_loss_coef(const int*, const double*, float*, int*, int, int, int, void*);
int b200rl_loss_value(const float*, const int*, const double*, double*, int, int, int, void*);
int b200rl_logprob_kl(void*, long long, const int*, const float*, const float*, const float*, float*, int, int, int, void*);
int b200rl_logprob_clip(void*, long long, const int*, const float*, const float*, const float*, const float*, double, float*, int, int, int, void*);
int b200rl_loss_value_clip(const float*, const int*, const double*, const float*, double, const float*, double, double*, int, int, int, void*);
int b200rl_loss_coef_kl(const int*, const double*, float*, float*, double, int*, int, int, int, void*);
int b200rl_loss_value_kl(const float*, const int*, const double*, const float*, double, double*, int, int, int, void*);
int b200rl_logprob_entropy(void*, long long, const int*, const float*, const float*, const float*, const float*, double, float*,
                           int, int, int, const int*, const int*, const int*, int, int, int, double, float*, void*);
int b200rl_loss_value_entropy(const float*, const int*, const double*, const float*, double, const float*, double, double*, int,
                              int, int, const float*, double, double*, void*);
int b200rl_nf4_dequant(const void*, const float*, void*, int, int, int, void*);
int b200rl_lora_pack(const float*, void*, const void*, int, int, void*);
int b200rl_rope_pos(void*, const float*, const int*, int, long long, int, int, int, void*);
int b200rl_gather_rows_idx(const void*, const int*, void*, int, int, void*);
int b200rl_scatter_add_rows(const void*, const int*, const int*, void*, int, int, void*);
}

namespace {

struct PackDescH {  // must match PackDesc in optim.cu
  long long src_off;
  int rows, cols;
  long long dst_off;
  int dst_ld;
  int transpose;
};

struct AccumBlock {
  long long dst_off;  // into the flat grad buffer
  int rows, cols;     // destination tensor shape
  int row_off, col_off;
  int transpose;
};
struct AccumArgs {
  AccumBlock blk[3];
  int nblk;
  const float* slabs;
  long long slab_stride;
  int splits;
  int ld;
};
// grouped variant: every block names its own slab set (one launch for all dA / dB blocks of a layer)
struct AccumBlockG {
  AccumBlock b;
  const float* slabs;
  long long slab_stride;
};
struct AccumArgsG {
  AccumBlockG blk[16];
  int nblk;
  int splits;
  int ld;
};

__global__ void grad_accum_kernel(float* __restrict__ flat, const AccumArgs a) {
  pdl_enter();
  const AccumBlock d = a.blk[blockIdx.y];
  const long long n = (long long)d.rows * d.cols;
  for (long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x; idx < n;
       idx += (long long)gridDim.x * blockDim.x) {
    const int i = (int)(idx / d.cols), j = (int)(idx % d.cols);
    const long long o = d.transpose ? (long long)(d.row_off + j) * a.ld + d.col_off + i
                                    : (long long)(d.row_off + i) * a.ld + d.col_off + j;
    float acc = 0.f;
    for (int s = 0; s < a.splits; ++s) acc += a.slabs[(long long)s * a.slab_stride + o];  // fixed order
    flat[d.dst_off + idx] += acc;
  }
}

__global__ void grad_accum_grouped_kernel(float* __restrict__ flat, const AccumArgsG a) {
  pdl_enter();
  const AccumBlock d = a.blk[blockIdx.y].b;
  const float* __restrict__ slabs = a.blk[blockIdx.y].slabs;
  const long long stride = a.blk[blockIdx.y].slab_stride;
  const long long n = (long long)d.rows * d.cols;
  for (long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x; idx < n;
       idx += (long long)gridDim.x * blockDim.x) {
    const int i = (int)(idx / d.cols), j = (int)(idx % d.cols);
    const long long o = d.transpose ? (long long)(d.row_off + j) * a.ld + d.col_off + i
                                    : (long long)(d.row_off + i) * a.ld + d.col_off + j;
    float acc = 0.f;
    for (int s = 0; s < a.splits; ++s) acc += slabs[(long long)s * stride + o];  // fixed order
    flat[d.dst_off + idx] += acc;
  }
}

// out[i] = bf16(sum_s slabs[s][i])  (fixed order; alpha was applied per slab by the GEMM epilogue)
__global__ void reduce_slabs_bf16_kernel(const float* __restrict__ slabs, long long slab_stride, int splits,
                                         bf16* __restrict__ out, long long n8) {
  pdl_enter();
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n8) return;
  float acc[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
  for (int s = 0; s < splits; ++s) {
    const float4 a = *reinterpret_cast<const float4*>(slabs + (long long)s * slab_stride + i * 8);
    const float4 b = *reinterpret_cast<const float4*>(slabs + (long long)s * slab_stride + i * 8 + 4);
    acc[0] += a.x; acc[1] += a.y; acc[2] += a.z; acc[3] += a.w;
    acc[4] += b.x; acc[5] += b.y; acc[6] += b.z; acc[7] += b.w;
  }
  reinterpret_cast<bf16x8*>(out)[i] = pack8(acc);
}

__global__ void targets_kernel(const int* __restrict__ ids, int* __restrict__ targets, int L, int P,
                               int T, int n) {
  pdl_enter();
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int b = i / T, t = i % T;
  targets[i] = ids[(long long)b * L + P + t];
}

inline long long align_up(long long x, long long a) { return (x + a - 1) / a * a; }

// one fused projection group
struct Group {
  int Kin, Nout, nproj, K2;
  int out_dims[3];       // per projection output rows
  // offsets (elements) into the bf16 LoRA operand arena of the layer
  long long acat, bcat;
  // flat fp32 offsets of A_j / B_j
  long long a_off[3], b_off[3];
};

}  // namespace

struct b200rl_model {
  b200rl_model_config cfg;
  std::vector<b200rl_layer_weights> layers;
  const bf16 *embed, *final_norm, *lm_head;
  float *lora_flat, *lora_grad;
  long long lora_numel;
  int QKV, QD;  // qkv row width, q width
  std::vector<Group> groups;  // 4 per layer: qkv, o, gu, down
  long long arena_per_layer;
  int K2max;
  // workspace pointers
  uint8_t* ws;
  long long ws_bytes;
  bf16* arena;          // bf16 LoRA operand copies, all layers
  void* pack_descs;     // device PackDescH[n_pack]
  int n_pack, pack_max_elems;
  bf16* X;              // [(n_layers+1)][Mt][H]
  struct LayerAct {
    bf16 *h1, *qkv, *attn_o, *x_mid, *h2, *gu, *act, *u_qkv, *u_o, *u_gu, *u_d;
    float *rstd1, *rstd2, *lse;
  };
  std::vector<LayerAct> act;
  bf16 *wbuf, *xsel, *hsel, *logits, *dhsel, *dx, *dx2, *dh, *dact, *dgu, *dattn, *dqkv, *du;  // du: 4 x [Mt][K2max]
  float* gslabs;            // grouped dW slabs
  long long gslab_elems;
  bool grouped_dw = !(getenv("B200RL_GROUPED_DW") && getenv("B200RL_GROUPED_DW")[0] == '0');
  float *rstd_f, *lp, *coef, *klw, *delta, *slabs, *rope_cs, *kvpart;
  long long kvpart_rows;
  int *targets, *lens;
  long long slab_elems;
  int rope_L;
  // optional resident bf16 copy of the dequantised base weights (b200rl_model_set_weight_cache): 15 GB for a 7B
  // model, 8 % of a B200's HBM, and it removes 2 x n_layers x 4 dequant passes per micro-batch
  bool fuse_swiglu = !(getenv("B200RL_FUSE_SWIGLU") && getenv("B200RL_FUSE_SWIGLU")[0] == '0');  // b200rl_model_set_fusion
  bf16* wcache = nullptr;
  long long wcache_per_layer = 0;
  // without a cache: 0 = dequantise each matrix into the scratch right before its GEMM, 1 = hand the NF4 storage to the GEMM,
  // whose producer warps dequantise it inside the mainloop (b200rl_model_set_nf4_inkernel; env B200RL_NF4_INKERNEL=1)
  bool nf4_inkernel = getenv("B200RL_NF4_INKERNEL") && getenv("B200RL_NF4_INKERNEL")[0] == '1';
  const void* next_q = nullptr;      // set by base_weight(), consumed by the next gemm_l()
  const float* next_am = nullptr;
  std::vector<uint8_t> wcache_valid;  // [n_layers*4]
  // optional per-op CUDA-event profiling (bench.py roofline / DESIGN.md breakdown)
  bool prof_on = false;
  std::vector<cudaEvent_t> prof_ev;
  std::vector<int> prof_cat;
  std::vector<double> prof_work;
  int prof_n = 0;
};

enum { CAT_GEMM = 0, CAT_GEMM_SKINNY = 1, CAT_GEMM_DW = 2, CAT_DEQUANT = 3, CAT_ATTN_FWD = 4, CAT_ATTN_BWD = 5,
       CAT_ROW = 6, CAT_LOGPROB = 7, CAT_MISC = 8, CAT_END = -1, NCAT = 9 };

static inline void prof_mark(b200rl_model* m, cudaStream_t st, int cat, double work) {
  if (!m->prof_on || m->prof_n >= (int)m->prof_ev.size()) return;
  cudaEventRecord(m->prof_ev[m->prof_n], st);
  m->prof_cat[m->prof_n] = cat;
  m->prof_work[m->prof_n] = work;
  ++m->prof_n;
}
#define PM(cat, work) prof_mark(m, st, (cat), (double)(work))

static void build_groups(b200rl_model* m) {
  const b200rl_model_config& c = m->cfg;
  const int H = c.hidden, I = c.inter, r = c.lora_r;
  const int QD = c.n_q_heads * c.head_dim, KD = c.n_kv_heads * c.head_dim;
  m->QD = QD;
  m->QKV = QD + 2 * KD;
  long long flat = 0;
  m->groups.clear();
  m->K2max = 64;
  long long arena_layer = 0;
  for (int l = 0; l < c.n_layers; ++l) {
    long long arena = 0;
    auto add = [&](int Kin, int nproj, const int* outs) {
      Group g;
      g.Kin = Kin;
      g.nproj = nproj;
      g.Nout = 0;
      for (int j = 0; j < nproj; ++j) {
        g.out_dims[j] = outs[j];
        g.Nout += outs[j];
      }
      g.K2 = (int)align_up((long long)nproj * r, 64);
      if (g.K2 > m->K2max) m->K2max = g.K2;
      // flat layout: per projection A [r, Kin] then B [out, r] (PEFT lora_A.weight / lora_B.weight)
      for (int j = 0; j < nproj; ++j) {
        g.a_off[j] = flat;
        flat += (long long)r * Kin;
        g.b_off[j] = flat;
        flat += (long long)outs[j] * r;
      }
      g.acat = arena;   arena += (long long)g.K2 * Kin;
      g.bcat = arena;   arena += (long long)g.Nout * g.K2;
      arena = align_up(arena, 64);
      m->groups.push_back(g);
    };
    const int o_qkv[3] = {QD, KD, KD};
    const int o_o[1] = {H};
    const int o_gu[2] = {I, I};
    const int o_d[1] = {H};
    add(H, 3, o_qkv);
    add(QD, 1, o_o);
    add(H, 2, o_gu);
    add(I, 1, o_d);
    arena_layer = arena;
  }
  m->arena_per_layer = arena_layer;
  m->lora_numel = align_up(flat, 4);
}

static int dw_splits(int tokens, int Ny, int bn_cols) {
  // enough (tile, split) work units to cover the SMs; the GEMM clamps to the k-block count
  const int tiles = ((Ny + 127) / 128) * ((bn_cols + 63) / 64 > 1 ? (bn_cols + 127) / 128 : 1);
  int s = (num_sms() + tiles - 1) / tiles;
  const int kb = (tokens + 63) / 64;
  if (s > kb) s = kb;
  if (s < 1) s = 1;
  if (s > 16) s = 16;
  const int per = (kb + s - 1) / s;
  return (kb + per - 1) / per;
}

struct WsPlan {
  long long total;
  long long off_arena, off_pack, off_X, off_wbuf, off_xsel, off_hsel, off_logits, off_dhsel, off_dx,
      off_dh, off_dx2, off_gslabs, off_dact, off_dgu, off_dattn, off_dqkv, off_du, off_rstd_f, off_lp, off_coef, off_klw, off_delta, off_kvpart,
      off_slabs, off_rope, off_targets, off_lens, off_layers;
  long long per_layer;
  long long slab_elems, gslab_elems;
};

static WsPlan plan_ws(const b200rl_model* m) {
  const b200rl_model_config& c = m->cfg;
  const long long Mt = c.max_tokens, H = c.hidden, I = c.inter, V = c.vocab;
  const long long R = c.max_score_rows;
  const long long QKV = m->QKV, QD = m->QD;
  WsPlan p;
  long long o = 0;
  auto take = [&](long long bytes) {
    long long at = o;
    o = align_up(o + bytes, 1024);
    return at;
  };
  p.off_arena = take(m->arena_per_layer * c.n_layers * 2);
  p.off_pack = take((long long)sizeof(PackDescH) * 28 * c.n_layers);
  p.off_X = take((long long)(c.n_layers + 1) * Mt * H * 2);
  long long wmax = std::max(std::max(QKV * H, QD * H), std::max(2 * I * H, I * H));
  p.off_wbuf = take(wmax * 2);
  p.off_xsel = take(R * H * 2);
  p.off_hsel = take(R * H * 2);
  p.off_logits = take(R * V * 2);
  p.off_dhsel = take(R * H * 2);
  p.off_dx = take(Mt * H * 2);
  p.off_dh = take(Mt * H * 2);
  p.off_dx2 = take(Mt * H * 2);
  // grouped dW: <= 4 K-ranges of [rows, 64] fp32 for the 8 problems of a layer (dB rows = out dims, dA rows = in dims)
  p.gslab_elems = 4 * (QKV + H + 2 * I + H + H + QD + H + I) * 64;
  p.off_gslabs = take(p.gslab_elems * 4);
  p.off_dact = take(Mt * I * 2);
  p.off_dgu = take(Mt * 2 * I * 2);
  p.off_dattn = take(Mt * QD * 2);
  p.off_dqkv = take(Mt * QKV * 2);
  p.off_du = take(4 * Mt * m->K2max * 2);
  p.off_rstd_f = take(R * 4);
  p.off_lp = take(R * 4);
  p.off_coef = take(R * 4);
  p.off_klw = take(R * 4);
  p.off_delta = take((long long)c.max_batch * c.n_q_heads * c.max_seq * 4);
  // fp32 dK/dV partial slabs of the packed (shared-prompt) attention backward: <= 2*max_tokens rows
  p.off_kvpart = take(c.head_dim == 128 ? 2 * Mt * 2 * c.n_kv_heads * c.head_dim * 4 : 0);
  long long nmax = std::max(std::max(QKV, 2 * I), std::max(H, I));
  p.slab_elems = 16 * std::max(nmax, (long long)128) * m->K2max;  // generous: <=16 splits
  // tighter: splits * Ny is bounded by ~ (num_sms/tiles+1) * Ny <= 2*128*num_sms for Ny < 128*sms
  long long bound = (long long)(2 * 128 * 160 + nmax) * m->K2max;
  if (p.slab_elems > bound) p.slab_elems = bound;
  p.off_slabs = take(p.slab_elems * 4);
  p.off_rope = take((long long)c.max_seq * c.head_dim * 4);
  p.off_targets = take(R * 4);
  p.off_lens = take((long long)c.max_batch * 4);
  p.off_layers = o;
  long long lo = 0;
  auto ltake = [&](long long bytes) { lo = align_up(lo + bytes, 1024); };
  ltake(Mt * H * 2);        // h1
  ltake(Mt * QKV * 2);      // qkv
  ltake(Mt * QD * 2);       // attn_o
  ltake(Mt * H * 2);        // x_mid
  ltake(Mt * H * 2);        // h2
  ltake(Mt * 2 * I * 2);    // gu
  ltake(Mt * I * 2);        // act
  for (int j = 0; j < 4; ++j) ltake(Mt * m->K2max * 2);  // u_*
  ltake(Mt * 4);            // rstd1
  ltake(Mt * 4);            // rstd2
  ltake((long long)c.max_batch * c.n_q_heads * c.max_seq * 4);  // lse
  p.per_layer = lo;
  p.total = p.off_layers + lo * c.n_layers;
  return p;
}

static int validate_cfg(const b200rl_model_config* c) {
  B200RL_REQUIRE(c != nullptr, "model: null config");
  B200RL_REQUIRE(c->vocab > 0 && c->vocab % 8 == 0, "model: vocab must be a multiple of 8");
  B200RL_REQUIRE(c->hidden % 64 == 0 && c->inter % 64 == 0, "model: hidden and inter must be multiples of 64 (NF4 blocks)");
  B200RL_REQUIRE(c->head_dim == 32 || c->head_dim == 64 || c->head_dim == 128, "model: head_dim must be 32/64/128");
  B200RL_REQUIRE(c->n_kv_heads > 0 && c->n_q_heads % c->n_kv_heads == 0, "model: bad head counts");
  B200RL_REQUIRE((c->n_q_heads * c->head_dim) % 64 == 0 && (c->n_kv_heads * c->head_dim) % 64 == 0,
                 "model: head widths must be multiples of 64");
  B200RL_REQUIRE(c->lora_r > 0 && c->lora_r % 8 == 0, "model: lora_r must be a positive multiple of 8");
  B200RL_REQUIRE(c->n_layers > 0 && c->max_tokens > 0 && c->max_batch > 0 && c->max_seq > 0 &&
                     c->max_score_rows > 0, "model: bad sizes");
  return 0;
}

extern "C" long long b200rl_model_lora_numel(const b200rl_model_config* cfg) {
  if (validate_cfg(cfg)) return -1;
  b200rl_model m;
  m.cfg = *cfg;
  build_groups(&m);
  return m.lora_numel;
}

extern "C" long long b200rl_model_workspace_bytes(const b200rl_model_config* cfg) {
  if (validate_cfg(cfg)) return -1;
  b200rl_model m;
  m.cfg = *cfg;
  build_groups(&m);
  return plan_ws(&m).total;
}

extern "C" int b200rl_model_create(const b200rl_model_config* cfg, const b200rl_layer_weights* layers_host,
                                   const void* embed, const void* final_norm_w, const void* lm_head,
                                   float* lora_flat, float* lora_grad_flat,
                                   void* workspace, long long workspace_bytes, b200rl_model** out) {
  int rc = validate_cfg(cfg);
  if (rc) return rc;
  B200RL_REQUIRE(layers_host && embed && final_norm_w && lm_head && lora_flat &&
                     lora_grad_flat && workspace && out, "model_create: null pointer");
  b200rl_model* m = new (std::nothrow) b200rl_model();
  B200RL_REQUIRE(m != nullptr, "model_create: out of host memory");
  m->cfg = *cfg;
  m->layers.assign(layers_host, layers_host + cfg->n_layers);
  m->embed = (const bf16*)embed;
  m->final_norm = (const bf16*)final_norm_w;
  m->lm_head = (const bf16*)lm_head;
  m->lora_flat = lora_flat;
  m->lora_grad = lora_grad_flat;
  build_groups(m);
  WsPlan p = plan_ws(m);
  if (workspace_bytes < p.total) {
    delete m;
    return set_error(B200RL_ERR_ARG, "model_create: workspace too small (%lld < %lld)", workspace_bytes, p.total);
  }
  if ((reinterpret_cast<uintptr_t>(workspace) & 1023u) != 0) {
    delete m;
    return set_error(B200RL_ERR_ARG, "model_create: workspace must be 1024-byte aligned");
  }
  uint8_t* w = (uint8_t*)workspace;
  m->ws = w;
  m->ws_bytes = p.total;
  m->arena = (bf16*)(w + p.off_arena);
  m->pack_descs = w + p.off_pack;
  m->X = (bf16*)(w + p.off_X);
  m->wbuf = (bf16*)(w + p.off_wbuf);
  m->dx2 = (bf16*)(w + p.off_dx2);
  m->gslabs = (float*)(w + p.off_gslabs);
  m->gslab_elems = p.gslab_elems;
  m->xsel = (bf16*)(w + p.off_xsel);
  m->hsel = (bf16*)(w + p.off_hsel);
  m->logits = (bf16*)(w + p.off_logits);
  m->dhsel = (bf16*)(w + p.off_dhsel);
  m->dx = (bf16*)(w + p.off_dx);
  m->dh = (bf16*)(w + p.off_dh);
  m->dact = (bf16*)(w + p.off_dact);
  m->dgu = (bf16*)(w + p.off_dgu);
  m->dattn = (bf16*)(w + p.off_dattn);
  m->dqkv = (bf16*)(w + p.off_dqkv);
  m->du = (bf16*)(w + p.off_du);
  m->rstd_f = (float*)(w + p.off_rstd_f);
  m->lp = (float*)(w + p.off_lp);
  m->coef = (float*)(w + p.off_coef);
  m->klw = (float*)(w + p.off_klw);
  m->delta = (float*)(w + p.off_delta);
  m->kvpart = (float*)(w + p.off_kvpart);
  m->kvpart_rows = cfg->head_dim == 128 ? 2LL * cfg->max_tokens : 0;
  m->slabs = (float*)(w + p.off_slabs);
  m->slab_elems = p.slab_elems;
  m->rope_cs = (float*)(w + p.off_rope);
  m->targets = (int*)(w + p.off_targets);
  m->lens = (int*)(w + p.off_lens);
  m->rope_L = 0;
  const b200rl_model_config& c = m->cfg;
  const long long Mt = c.max_tokens, H = c.hidden, I = c.inter;
  m->act.resize(c.n_layers);
  for (int l = 0; l < c.n_layers; ++l) {
    uint8_t* b = w + p.off_layers + p.per_layer * l;
    long long lo = 0;
    auto ltake = [&](long long bytes) {
      uint8_t* at = b + lo;
      lo = align_up(lo + bytes, 1024);
      return at;
    };
    b200rl_model::LayerAct& a = m->act[l];
    a.h1 = (bf16*)ltake(Mt * H * 2);
    a.qkv = (bf16*)ltake(Mt * m->QKV * 2);
    a.attn_o = (bf16*)ltake(Mt * m->QD * 2);
    a.x_mid = (bf16*)ltake(Mt * H * 2);
    a.h2 = (bf16*)ltake(Mt * H * 2);
    a.gu = (bf16*)ltake(Mt * 2 * I * 2);
    a.act = (bf16*)ltake(Mt * I * 2);
    a.u_qkv = (bf16*)ltake(Mt * m->K2max * 2);
    a.u_o = (bf16*)ltake(Mt * m->K2max * 2);
    a.u_gu = (bf16*)ltake(Mt * m->K2max * 2);
    a.u_d = (bf16*)ltake(Mt * m->K2max * 2);
    a.rstd1 = (float*)ltake(Mt * 4);
    a.rstd2 = (float*)ltake(Mt * 4);
    a.lse = (float*)ltake((long long)c.max_batch * c.n_q_heads * c.max_seq * 4);
  }
  // pack descriptors (fp32 master -> 4 bf16 operand layouts per projection)
  std::vector<PackDescH> descs;
  int max_elems = 0;
  const int r = c.lora_r;
  for (int l = 0; l < c.n_layers; ++l) {
    const long long base = m->arena_per_layer * l;
    for (int gi = 0; gi < 4; ++gi) {
      const Group& g = m->groups[l * 4 + gi];
      int row_off = 0;
      for (int j = 0; j < g.nproj; ++j) {
        // A_j [r, Kin] -> Acat rows j*r.. (ld Kin)
        descs.push_back({g.a_off[j], r, g.Kin, base + g.acat + (long long)j * r * g.Kin, g.Kin, 0});
        // B_j [out_j, r] -> Bcat rows row_off.., cols j*r.. (ld K2)
        descs.push_back({g.b_off[j], g.out_dims[j], r, base + g.bcat + (long long)row_off * g.K2 + j * r, g.K2, 0});
        max_elems = std::max(max_elems, std::max(r * g.Kin, g.out_dims[j] * r));
        row_off += g.out_dims[j];
      }
    }
  }
  m->n_pack = (int)descs.size();
  m->pack_max_elems = max_elems;
  cudaError_t e = cudaMemcpy(m->pack_descs, descs.data(), descs.size() * sizeof(PackDescH), cudaMemcpyHostToDevice);
  if (e == cudaSuccess) e = cudaMemset(m->arena, 0, (size_t)(m->arena_per_layer * c.n_layers * 2));
  if (e != cudaSuccess) {
    delete m;
    return set_error(B200RL_ERR_CUDA, "model_create: %s", cudaGetErrorString(e));
  }
  *out = m;
  return 0;
}

extern "C" int b200rl_model_destroy(b200rl_model* m) {
  delete m;
  return 0;
}

extern "C" int b200rl_model_sync_lora(b200rl_model* m, void* stream) {
  B200RL_REQUIRE(m != nullptr, "model_sync_lora: null model");
  return b200rl_lora_pack(m->lora_flat, m->arena, m->pack_descs, m->n_pack, m->pack_max_elems, stream);
}

// named buffer lookup for parity bisection (tests only)
extern "C" void* b200rl_model_debug_ptr(b200rl_model* m, const char* name, int layer) {
  if (!m || !name) return nullptr;
  const long long Mt = m->cfg.max_tokens, H = m->cfg.hidden;
  if (!strcmp(name, "x")) return m->X + (long long)layer * Mt * H;
  if (!strcmp(name, "logits")) return m->logits;
  if (!strcmp(name, "hsel")) return m->hsel;
  if (!strcmp(name, "dx")) return m->dx;
  if (!strcmp(name, "dqkv")) return m->dqkv;
  if (!strcmp(name, "wbuf")) return m->wbuf;
  if (layer < 0 || layer >= m->cfg.n_layers) return nullptr;
  b200rl_model::LayerAct& a = m->act[layer];
  if (!strcmp(name, "h1")) return a.h1;
  if (!strcmp(name, "qkv")) return a.qkv;
  if (!strcmp(name, "attn_o")) return a.attn_o;
  if (!strcmp(name, "x_mid")) return a.x_mid;
  if (!strcmp(name, "h2")) return a.h2;
  if (!strcmp(name, "gu")) return a.gu;
  if (!strcmp(name, "act")) return a.act;
  if (!strcmp(name, "u_qkv")) return a.u_qkv;
  return nullptr;
}

#define RC(expr)              \
  do {                        \
    int _rc = (expr);         \
    if (_rc) return _rc;      \
  } while (0)

namespace {

int gemm_l(b200rl_model* m, int cat, int layout, cudaStream_t st, const bf16* A1, long long lda1, const bf16* B1, long long ldb1, int K1,
            const bf16* A2, long long lda2, const bf16* B2, long long ldb2, int K2, bf16* C,
            long long ldc, const bf16* bias, const bf16* residual, long long ldr, float alpha, int M,
            int N, int fuse = 0, void* aux = nullptr, long long ld_aux = 0, const bf16* extB = nullptr,
            long long ld_ext = 0, float ext_alpha = 1.f) {
  GemmArgs a;
  a.A1 = A1; a.B1 = B1; a.A2 = A2; a.B2 = B2;
  a.lda1 = lda1; a.ldb1 = ldb1; a.lda2 = lda2; a.ldb2 = ldb2;
  a.K1 = K1; a.K2 = K2; a.C = C; a.ldc = ldc; a.c_fp32 = 0;
  a.bias = bias; a.residual = residual; a.ldr = ldr; a.alpha = alpha;
  a.M = M; a.N = N; a.mn_major = layout; a.splits = 1; a.c_split_stride = 0;
  a.force_bn = 0; a.max_ctas = 0;
  a.fuse = fuse; a.aux = aux; a.ld_aux = ld_aux;
  a.ext_B = extB; a.ld_ext_b = ld_ext; a.ext_alpha = ext_alpha;   // LoRA intermediate A2 produced inside this launch
  if (m->next_q) {   // base_weight() chose the in-kernel dequant for this GEMM: B1 is NF4 storage
    a.nf4_packed = m->next_q; a.nf4_absmax = m->next_am;
    m->next_q = nullptr; m->next_am = nullptr;
  }
  PM(cat, 2.0 * M * N * K1 + (K2 ? 2.0 * M * N * m->cfg.lora_r : 0.0) + (extB ? 2.0 * M * K2 * (double)K1 : 0.0));
  if (cat == CAT_GEMM_SKINNY) {
    // rank-r LoRA intermediates (N = K2 <= 192): only ceil(M/128) output tiles, so split K across CTAs
    // into fp32 slabs (deterministic order) and reduce to bf16 in a second, tiny kernel
    const int tiles = ((M + 127) / 128) * ((N + 127) / 128 > 1 ? (N + 127) / 128 : 1);
    const int kb = (K1 + 63) / 64;
    const int sms = num_sms();
    int best_s = 1;
    double best = 1e30;
    for (int sp = 1; sp <= 8 && sp <= kb; ++sp) {
      const double t = (double)((tiles * sp + sms - 1) / sms) / sp;
      if (t < best - 1e-9) {
        best = t;
        best_s = sp;
      }
    }
    const int per = (kb + best_s - 1) / best_s;
    const int splits = (kb + per - 1) / per;
    const long long stride = (long long)M * N;
    if (splits > 1 && K2 == 0 && ldc == N && splits * stride <= m->slab_elems) {
      a.C = m->slabs; a.c_fp32 = 1; a.splits = splits; a.c_split_stride = stride;
      int rc = gemm_dispatch(a, st);
      if (rc) return rc;
      const long long n8 = stride / 8;
      B200RL_CUDA_OK(launch_pdl(reduce_slabs_bf16_kernel, dim3((unsigned)((n8 + 255) / 256)), dim3(256), 0, st, m->slabs, stride, splits, C, n8));
      B200RL_LAUNCH_OK();
      return 0;
    }
  }
  return gemm_dispatch(a, st);
}

// LoRA weight gradients of one group from (dY, u') and (x, du):
//   dBcat = dY^T . u'  -> B_j blocks ; dAcat^T = x^T . du -> A_j blocks (transposed unpack)
int lora_dw(b200rl_model* m, cudaStream_t st, const Group& g, const bf16* dY, long long ld_dy,
            const bf16* u, const bf16* x, long long ld_x, const bf16* du, int M) {
  for (int pass = 0; pass < 2; ++pass) {
    const bf16* Y = pass == 0 ? dY : x;
    const long long ldy = pass == 0 ? ld_dy : ld_x;
    const int Ny = pass == 0 ? g.Nout : g.Kin;
    const bf16* U = pass == 0 ? u : du;
    const int splits = dw_splits(M, Ny, g.K2);
    const long long stride = (long long)Ny * g.K2;
    if ((long long)splits * stride > m->slab_elems)
      return set_error(B200RL_ERR_STATE, "lora_dw: slab scratch too small (%lld > %lld)", (long long)splits * stride, m->slab_elems);
    GemmArgs a;
    memset(&a, 0, sizeof(a));
    a.A1 = Y; a.lda1 = ldy; a.B1 = U; a.ldb1 = g.K2; a.K1 = M; a.K2 = 0;
    a.C = m->slabs; a.ldc = g.K2; a.c_fp32 = 1; a.alpha = 1.f;
    a.M = Ny; a.N = g.K2; a.mn_major = 3; a.splits = splits; a.c_split_stride = stride;
    PM(CAT_GEMM_DW, 2.0 * M * Ny * m->cfg.lora_r * g.nproj);
    RC(gemm_dispatch(a, st));
    PM(CAT_MISC, 0);
    AccumArgs acc;
    memset(&acc, 0, sizeof(acc));
    acc.nblk = g.nproj;
    acc.slabs = m->slabs;
    acc.slab_stride = stride;
    acc.splits = splits;
    acc.ld = g.K2;
    int row_off = 0, max_elems = 0;
    const int r = m->cfg.lora_r;
    for (int j = 0; j < g.nproj; ++j) {
      AccumBlock& b = acc.blk[j];
      if (pass == 0) {  // dB_j [out_j, r] = slab[row_off + i][j*r + jj]
        b.dst_off = g.b_off[j]; b.rows = g.out_dims[j]; b.cols = r;
        b.row_off = row_off; b.col_off = j * r; b.transpose = 0;
      } else {          // dA_j [r, Kin]: dA_j[i][k] = slab[k][j*r + i]
        b.dst_off = g.a_off[j]; b.rows = r; b.cols = g.Kin;
        b.row_off = 0; b.col_off = j * r; b.transpose = 1;
      }
      max_elems = std::max(max_elems, b.rows * b.cols);
      row_off += g.out_dims[j];
    }
    int bx = (max_elems + 255) / 256;
    if (bx > 128) bx = 128;
    dim3 grid(bx, g.nproj);
    B200RL_CUDA_OK(launch_pdl(grad_accum_kernel, dim3(grid), dim3(256), 0, st, m->lora_grad, acc));
    B200RL_LAUNCH_OK();
  }
  return 0;
}

// Grouped form of lora_dw for one layer (all K2 == 64): problems 2g = dBcat_g = dY_g^T . u_g, 2g+1 = dAcat_g^T = x_g^T . du_g.
int lora_dw_grouped(b200rl_model* m, cudaStream_t st, const Group* const* gs, const bf16* const* dYs, const long long* ldYs,
                    const bf16* const* us, const bf16* const* xs, const long long* ldXs, const bf16* const* dus, int M) {
  const void* Y[8];
  const void* U[8];
  long long ldy[8], ldu[8], stride[8];
  int rows[8];
  float* C[8];
  int total_blocks = 0;
  double flops = 0;
  for (int g = 0; g < 4; ++g) {
    Y[2 * g] = dYs[g]; ldy[2 * g] = ldYs[g]; rows[2 * g] = gs[g]->Nout; U[2 * g] = us[g]; ldu[2 * g] = 64;
    Y[2 * g + 1] = xs[g]; ldy[2 * g + 1] = ldXs[g]; rows[2 * g + 1] = gs[g]->Kin; U[2 * g + 1] = dus[g]; ldu[2 * g + 1] = 64;
    total_blocks += (gs[g]->Nout + 127) / 128 + (gs[g]->Kin + 127) / 128;
    flops += 2.0 * M * (gs[g]->Nout + gs[g]->Kin) * m->cfg.lora_r * gs[g]->nproj;
  }
  const int splits = dw_grouped_splits(total_blocks, (M + 63) / 64);
  long long off = 0;
  for (int i = 0; i < 8; ++i) {
    stride[i] = (long long)rows[i] * 64;
    C[i] = m->gslabs + off;
    off += stride[i] * splits;
  }
  if (off > m->gslab_elems) return set_error(B200RL_ERR_STATE, "lora_dw_grouped: slab scratch too small (%lld > %lld)", off, m->gslab_elems);
  PM(CAT_GEMM_DW, flops);
  const int used = dw_grouped_dispatch(8, Y, ldy, rows, U, ldu, C, stride, M, splits, st);
  if (used <= 0) return used < 0 ? used : set_error(B200RL_ERR_STATE, "lora_dw_grouped: dispatch returned 0");
  PM(CAT_MISC, 0);
  AccumArgsG acc;
  memset(&acc, 0, sizeof(acc));
  acc.splits = used;
  acc.ld = 64;
  const int r = m->cfg.lora_r;
  int nb = 0, max_elems = 0;
  for (int g = 0; g < 4; ++g) {
    const Group& G = *gs[g];
    int row_off = 0;
    for (int j = 0; j < G.nproj; ++j) {
      AccumBlockG& b = acc.blk[nb++];   // dB_j [out_j, r] = slab[row_off + i][j*r + jj]
      b.slabs = C[2 * g]; b.slab_stride = stride[2 * g];
      b.b.dst_off = G.b_off[j]; b.b.rows = G.out_dims[j]; b.b.cols = r;
      b.b.row_off = row_off; b.b.col_off = j * r; b.b.transpose = 0;
      max_elems = std::max(max_elems, b.b.rows * b.b.cols);
      row_off += G.out_dims[j];
    }
    for (int j = 0; j < G.nproj; ++j) {
      AccumBlockG& b = acc.blk[nb++];   // dA_j [r, Kin]: dA_j[i][k] = slab[k][j*r + i]
      b.slabs = C[2 * g + 1]; b.slab_stride = stride[2 * g + 1];
      b.b.dst_off = G.a_off[j]; b.b.rows = r; b.b.cols = G.Kin;
      b.b.row_off = 0; b.b.col_off = j * r; b.b.transpose = 1;
      max_elems = std::max(max_elems, b.b.rows * b.b.cols);
    }
  }
  acc.nblk = nb;
  int bx = (max_elems + 255) / 256;
  if (bx > 64) bx = 64;
  B200RL_CUDA_OK(launch_pdl(grad_accum_grouped_kernel, dim3(bx, nb), dim3(256), 0, st, m->lora_grad, acc));
  B200RL_LAUNCH_OK();
  return 0;
}

}  // namespace

namespace {
// token layout of one micro-batch: classic [B, L] padded batch, or the packed shared-prompt layout
struct Layout {
  int M, B, T, L, P;
  const int* ids;
  const int* key_mask;      // classic: attention_mask [B, L]; packed: [rows]
  const int* answer_mask;
  const b200rl_packed_batch* pb;  // nullptr = classic
};
}  // namespace

// Dequantised base weight of projection `which` (0 qkv, 1 o, 2 gate|up, 3 down) of layer l: from the resident cache
// when one is attached (filled on first use), else NF4 -> bf16 into the shared scratch right before the GEMM.
static int base_weight(b200rl_model* m, cudaStream_t st, int l, int which, const bf16** out, int M = 0, int N = 0, int K1 = 0) {
  const b200rl_model_config& c = m->cfg;
  const b200rl_layer_weights& w = m->layers[l];
  const int H = c.hidden, I = c.inter, QKV = m->QKV, QD = m->QD;
  const void* packed[4] = {w.qkv_packed, w.o_packed, w.gu_packed, w.down_packed};
  const float* absmax[4] = {(const float*)w.qkv_absmax, (const float*)w.o_absmax, (const float*)w.gu_absmax, (const float*)w.down_absmax};
  const int rows[4] = {QKV, H, 2 * I, H}, cols[4] = {H, QD, H, I};
  bf16* dst = m->wbuf;
  if (!m->wcache && m->nf4_inkernel && gemm_nf4_supported(M, N, K1)) {
    // in-kernel dequant: the GEMM that follows (M x N output, reduction depth K1) reads the packed codes itself
    m->next_q = packed[which];
    m->next_am = absmax[which];
    *out = nullptr;
    return 0;
  }
  if (m->wcache) {
    long long off = 0;
    for (int i = 0; i < which; ++i) off += (long long)rows[i] * cols[i];
    dst = m->wcache + m->wcache_per_layer * l + off;
    *out = dst;
    if (m->wcache_valid[l * 4 + which]) return 0;
    m->wcache_valid[l * 4 + which] = 1;
  }
  *out = dst;
  PM(CAT_DEQUANT, 2.5625 * rows[which] * (double)cols[which]);
  RC(b200rl_nf4_dequant(packed[which], absmax[which], dst, rows[which], cols[which], 0, (void*)st));
  return 0;
}

static int run_microbatch(b200rl_model* m, const Layout& lay, const double* adv, float* lp_out, double* loss_accum,
                          int nb, int grpo, int backward, int lora_off, const float* ref_lp, double kl_beta,
                          const float* old_lp, double clip_eps, const b200rl_entropy_args* ent, void* stream) {
  const b200rl_model_config& c = m->cfg;
  const b200rl_packed_batch* pb = lay.pb;
  const int M = lay.M, B = lay.B, T = lay.T, L = lay.L, P = lay.P;
  const int* score_slot = (lay.pb && lay.pb->n_score > 0) ? lay.pb->score_slot : nullptr;
  const int R = score_slot ? lay.pb->n_score : B * T;   // scored rows: all B*T positions, or the live ones only
  const int* ids = lay.ids;
  const int* attn_mask = lay.key_mask;
  const int* answer_mask = lay.answer_mask;
  B200RL_REQUIRE(!backward || (adv && nb >= 1), "model_microbatch: backward needs adv and nb");
  B200RL_REQUIRE(!(backward && lora_off), "model_microbatch: the adapter-off (reference policy) pass is forward only");
  B200RL_REQUIRE(kl_beta == 0.0 || ref_lp, "model_microbatch: kl_beta != 0 needs ref_lp");
  const bool use_kl = backward && kl_beta != 0.0 && ref_lp;
  B200RL_REQUIRE(clip_eps >= 0.0, "model_microbatch: clip_eps must be >= 0");
  const bool use_clip = old_lp && clip_eps > 0.0;
  // entropy (b200rl_entropy_args): per-token H whenever ent_out is given, the bonus term when alpha != 0
  const bool use_ent = ent && (ent->ent_out || ent->alpha != 0.0 || ent->ent_accum);
  B200RL_REQUIRE(!use_ent || ent->ent_out, "model_microbatch: entropy_alpha != 0 or ent_accum needs ent_out");
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  const int H = c.hidden, I = c.inter, QKV = m->QKV, QD = m->QD, V = c.vocab;
  const long long Mt = c.max_tokens;
  const float s = c.lora_scale;
  const float attn_scale = 1.0f / sqrtf((float)c.head_dim);

  if (m->rope_L != L) {
    RC(b200rl_rope_table(m->rope_cs, L, c.head_dim, c.rope_theta, stream));
    m->rope_L = L;
  }
  // ---------------- forward ----------------
  const bf16* Wd = nullptr;
  const bool fuse_swiglu = m->fuse_swiglu && gemm_fuse_supported(M, I);
  const bool lora = !lora_off;  // adapter-disabled pass = reference policy pi_ref (KL term)
  PM(CAT_ROW, 2.0 * M * H * 2);
  RC(b200rl_embed(ids, m->embed, m->X, M, H, V, stream));
  for (int l = 0; l < c.n_layers; ++l) {
    const b200rl_layer_weights& w = m->layers[l];
    b200rl_model::LayerAct& a = m->act[l];
    const bf16* ar = m->arena + m->arena_per_layer * l;
    const Group& gq = m->groups[l * 4 + 0];
    const Group& go = m->groups[l * 4 + 1];
    const Group& gg = m->groups[l * 4 + 2];
    const Group& gd = m->groups[l * 4 + 3];
    bf16* x = m->X + (long long)l * Mt * H;
    bf16* xn = m->X + (long long)(l + 1) * Mt * H;
    PM(CAT_ROW, 2.0 * M * H * 2);
    RC(b200rl_rmsnorm_fwd(x, w.ln1_w, a.h1, a.rstd1, M, H, c.rms_eps, stream));
    // LoRA intermediates u = s x A^T: produced by the "ext units" of the big GEMM itself when the CTA-pair kernel runs it
    // (gemm2_tcgen05.cu), else by a separate split-K skinny GEMM
    const bool xq = lora && gemm_ext_supported(M, QKV, gq.K2), xo = lora && gemm_ext_supported(M, H, go.K2);
    const bool xg = lora && gemm_ext_supported(M, 2 * I, gg.K2), xd = lora && gemm_ext_supported(M, H, gd.K2);
    if (lora && !xq) RC(gemm_l(m, CAT_GEMM_SKINNY, 0, st, a.h1, H, ar + gq.acat, H, H, nullptr, 0, nullptr, 0, 0, a.u_qkv, gq.K2, nullptr, nullptr, 0, s, M, gq.K2));
    RC(base_weight(m, st, l, 0, &Wd, M, QKV, H));
    RC(gemm_l(m, CAT_GEMM, 0, st, a.h1, H, Wd, H, H, a.u_qkv, gq.K2, ar + gq.bcat, gq.K2, lora ? gq.K2 : 0, a.qkv, QKV,
               (const bf16*)w.qkv_bias, nullptr, 0, 1.f, M, QKV, 0, nullptr, 0, xq ? ar + gq.acat : nullptr, H, s));
    PM(CAT_ROW, 2.0 * M * (c.n_q_heads + c.n_kv_heads) * c.head_dim * 2);
    if (pb) RC(b200rl_rope_pos(a.qkv, m->rope_cs, pb->pos, M, QKV, c.n_q_heads + c.n_kv_heads, c.head_dim, 0, stream));
    else RC(b200rl_rope(a.qkv, m->rope_cs, M, L, QKV, c.n_q_heads + c.n_kv_heads, c.head_dim, 0, stream));
    PM(CAT_ATTN_FWD, 2.0 * B * c.n_q_heads * (double)L * L * c.head_dim);
    if (pb) RC(b200rl_attn_seg_fwd(a.qkv, attn_mask, a.attn_o, a.lse, M, c.n_q_heads, c.n_kv_heads, attn_scale, pb->qblocks, pb->n_qblocks, stream));
    else RC(b200rl_attn_fwd(a.qkv, attn_mask, a.attn_o, a.lse, B, L, c.n_q_heads, c.n_kv_heads, c.head_dim, attn_scale, stream));
    if (lora && !xo) RC(gemm_l(m, CAT_GEMM_SKINNY, 0, st, a.attn_o, QD, ar + go.acat, QD, QD, nullptr, 0, nullptr, 0, 0, a.u_o, go.K2, nullptr, nullptr, 0, s, M, go.K2));
    RC(base_weight(m, st, l, 1, &Wd, M, H, QD));
    RC(gemm_l(m, CAT_GEMM, 0, st, a.attn_o, QD, Wd, QD, QD, a.u_o, go.K2, ar + go.bcat, go.K2, lora ? go.K2 : 0, a.x_mid, H,
               nullptr, x, H, 1.f, M, H, 0, nullptr, 0, xo ? ar + go.acat : nullptr, QD, s));
    PM(CAT_ROW, 2.0 * M * H * 2);
    RC(b200rl_rmsnorm_fwd(a.x_mid, w.ln2_w, a.h2, a.rstd2, M, H, c.rms_eps, stream));
    if (lora && !xg) RC(gemm_l(m, CAT_GEMM_SKINNY, 0, st, a.h2, H, ar + gg.acat, H, H, nullptr, 0, nullptr, 0, 0, a.u_gu, gg.K2, nullptr, nullptr, 0, s, M, gg.K2));
    RC(base_weight(m, st, l, 2, &Wd, M, 2 * I, H));
    if (fuse_swiglu) {  // gate|up GEMM whose epilogue also writes act = silu(gate)*up
      RC(gemm_l(m, CAT_GEMM, 0, st, a.h2, H, Wd, H, H, a.u_gu, gg.K2, ar + gg.bcat, gg.K2, lora ? gg.K2 : 0, a.gu, 2 * I,
                 nullptr, nullptr, 0, 1.f, M, 2 * I, 1, a.act, I, xg ? ar + gg.acat : nullptr, H, s));
    } else {
      RC(gemm_l(m, CAT_GEMM, 0, st, a.h2, H, Wd, H, H, a.u_gu, gg.K2, ar + gg.bcat, gg.K2, lora ? gg.K2 : 0, a.gu, 2 * I,
                 nullptr, nullptr, 0, 1.f, M, 2 * I, 0, nullptr, 0, xg ? ar + gg.acat : nullptr, H, s));
      PM(CAT_ROW, 3.0 * M * I * 2);
      RC(b200rl_swiglu_fwd(a.gu, a.act, M, I, stream));
    }
    if (lora && !xd) RC(gemm_l(m, CAT_GEMM_SKINNY, 0, st, a.act, I, ar + gd.acat, I, I, nullptr, 0, nullptr, 0, 0, a.u_d, gd.K2, nullptr, nullptr, 0, s, M, gd.K2));
    RC(base_weight(m, st, l, 3, &Wd, M, H, I));
    RC(gemm_l(m, CAT_GEMM, 0, st, a.act, I, Wd, I, I, a.u_d, gd.K2, ar + gd.bcat, gd.K2, lora ? gd.K2 : 0, xn, H, nullptr,
               a.x_mid, H, 1.f, M, H, 0, nullptr, 0, xd ? ar + gd.acat : nullptr, I, s));
  }
  // head: only the T scored positions (rows P-1 .. L-2) go through the final norm and lm_head
  bf16* xf = m->X + (long long)c.n_layers * Mt * H;
  PM(CAT_ROW, 2.0 * R * H * 2);
  if (pb) RC(b200rl_gather_rows_idx(xf, pb->score_src, m->xsel, R, H, stream));
  else RC(b200rl_gather_rows(xf, m->xsel, B, L, T, P - 1, H, stream));
  PM(CAT_ROW, 2.0 * R * H * 2);
  RC(b200rl_rmsnorm_fwd(m->xsel, m->final_norm, m->hsel, m->rstd_f, R, H, c.rms_eps, stream));
  RC(gemm_l(m, CAT_GEMM, 0, st, m->hsel, H, m->lm_head, H, H, nullptr, 0, nullptr, 0, 0, m->logits, V, nullptr, nullptr, 0, 1.f, R, V));
  PM(CAT_MISC, 0);
  const int* targets = pb ? pb->targets : m->targets;
  if (!pb) {
    B200RL_CUDA_OK(launch_pdl(targets_kernel, dim3((R + 255) / 256), dim3(256), 0, st, ids, m->targets, L, P, T, R));
    B200RL_LAUNCH_OK();
  }
  PM(CAT_MISC, 0);
  if (backward) RC(b200rl_loss_coef_kl(answer_mask, adv, m->coef, use_kl ? m->klw : nullptr, kl_beta, m->lens, B, T, nb, stream));
  float* lp = lp_out ? lp_out : m->lp;
  if (score_slot) B200RL_CUDA_OK(cudaMemsetAsync(lp, 0, sizeof(float) * (size_t)B * T, st));  // positions left out report 0
  if (score_slot && use_ent) B200RL_CUDA_OK(cudaMemsetAsync(ent->ent_out, 0, sizeof(float) * (size_t)B * T, st));
  PM(CAT_LOGPROB, (backward ? 2.0 : 1.0) * R * V * 2);
  if (use_ent)
    RC(b200rl_logprob_entropy(m->logits, V, targets, backward ? m->coef : nullptr, use_kl ? m->klw : nullptr,
                              use_kl ? ref_lp : nullptr, use_clip ? old_lp : nullptr, use_clip ? clip_eps : 0.0, lp, R, V,
                              backward ? 1 : 0, score_slot, answer_mask, backward ? m->lens : nullptr, B, T, nb,
                              backward ? ent->alpha : 0.0, ent->ent_out, stream));
  else
    RC(b200rl_logprob_slots(m->logits, V, targets, backward ? m->coef : nullptr, use_kl ? m->klw : nullptr,
                            use_kl ? ref_lp : nullptr, use_clip ? old_lp : nullptr, use_clip ? clip_eps : 0.0, lp, R, V,
                            backward ? 1 : 0, score_slot, stream));
  PM(CAT_MISC, 0);
  if (loss_accum && adv) {
    if (use_ent)
      RC(b200rl_loss_value_entropy(lp, answer_mask, adv, use_kl ? ref_lp : nullptr, use_kl ? kl_beta : 0.0,
                                   use_clip ? old_lp : nullptr, use_clip ? clip_eps : 0.0, loss_accum, B, T, grpo,
                                   ent->ent_out, ent->alpha, ent->ent_accum, stream));
    else
      RC(b200rl_loss_value_clip(lp, answer_mask, adv, use_kl ? ref_lp : nullptr, use_kl ? kl_beta : 0.0,
                                use_clip ? old_lp : nullptr, use_clip ? clip_eps : 0.0, loss_accum, B, T, grpo, stream));
  }
  if (!backward) {
    PM(CAT_END, 0);
    return 0;
  }

  // ---------------- backward ----------------
  RC(gemm_l(m, CAT_GEMM, 2, st, m->logits, V, m->lm_head, H, V, nullptr, 0, nullptr, 0, 0, m->dhsel, H, nullptr, nullptr, 0, 1.f, R, H));
  PM(CAT_ROW, 3.0 * R * H * 2);
  RC(b200rl_rmsnorm_bwd(m->dhsel, m->xsel, m->final_norm, m->rstd_f, nullptr, m->dhsel, R, H, stream));
  PM(CAT_ROW, 1.0 * (R + M) * H * 2);
  if (pb) RC(b200rl_scatter_add_rows(m->dhsel, pb->sc_start, pb->sc_list, m->dx, M, H, stream));
  else RC(b200rl_scatter_rows(m->dhsel, m->dx, B, L, T, P - 1, H, stream));
  for (int l = c.n_layers - 1; l >= 0; --l) {
    const b200rl_layer_weights& w = m->layers[l];
    b200rl_model::LayerAct& a = m->act[l];
    const bf16* ar = m->arena + m->arena_per_layer * l;
    const Group& gq = m->groups[l * 4 + 0];
    const Group& go = m->groups[l * 4 + 1];
    const Group& gg = m->groups[l * 4 + 2];
    const Group& gd = m->groups[l * 4 + 3];
    bf16* x = m->X + (long long)l * Mt * H;
    // Backward GEMMs read W (and the LoRA operands) exactly as stored: B operand MN-major (layout 2).
    // Every group keeps its own du; dx / dx2 alternate as the residual-stream gradient so that all (dY, u, x, du) of
    // the layer are still alive when the grouped dW launch runs (before the layer's last rmsnorm_bwd overwrites dx).
    const bool grouped = m->grouped_dw && gq.K2 == 64 && go.K2 == 64 && gg.K2 == 64 && gd.K2 == 64;
    bf16* du_d = m->du;
    bf16* du_g = m->du + 1 * Mt * m->K2max;
    bf16* du_o = m->du + 2 * Mt * m->K2max;
    bf16* du_q = m->du + 3 * Mt * m->K2max;
    // ---- down projection:  X[l+1] = x_mid + act.Wd^T + u_d.Bd^T
    // du = s dY B: inside the dX GEMM (ext units) when it runs on the CTA-pair kernel and the grouped dW launch (which is
    // the only other consumer of du) comes after it; else the separate skinny GEMM
    const bool yd = grouped && gemm_ext_supported(M, I, gd.K2), yg = grouped && gemm_ext_supported(M, H, gg.K2);
    const bool yo = grouped && gemm_ext_supported(M, QD, go.K2), yq = grouped && l > 0 && gemm_ext_supported(M, H, gq.K2);
    if (!yd) RC(gemm_l(m, CAT_GEMM_SKINNY, 2, st, m->dx, H, ar + gd.bcat, gd.K2, H, nullptr, 0, nullptr, 0, 0, du_d, gd.K2, nullptr, nullptr, 0, s, M, gd.K2));
    if (!grouped) RC(lora_dw(m, st, gd, m->dx, H, a.u_d, a.act, I, du_d, M));
    RC(base_weight(m, st, l, 3, &Wd, M, I, H));
    if (fuse_swiglu) {  // dact never reaches HBM: the epilogue turns it into dgate|dup
      RC(gemm_l(m, CAT_GEMM, 2, st, m->dx, H, Wd, I, H, du_d, gd.K2, ar + gd.acat, I, gd.K2, m->dgu, 2 * I, nullptr, nullptr, 0, 1.f, M, I,
                 2, a.gu, 2 * I, yd ? ar + gd.bcat : nullptr, gd.K2, s));
    } else {
      RC(gemm_l(m, CAT_GEMM, 2, st, m->dx, H, Wd, I, H, du_d, gd.K2, ar + gd.acat, I, gd.K2, m->dact, I, nullptr, nullptr, 0, 1.f, M, I,
                 0, nullptr, 0, yd ? ar + gd.bcat : nullptr, gd.K2, s));
      PM(CAT_ROW, 5.0 * M * I * 2);
      RC(b200rl_swiglu_bwd(a.gu, m->dact, m->dgu, M, I, stream));
    }
    // ---- gate|up:  gu = h2.Wgu^T + u_gu.Bgu^T
    if (!yg) RC(gemm_l(m, CAT_GEMM_SKINNY, 2, st, m->dgu, 2 * I, ar + gg.bcat, gg.K2, 2 * I, nullptr, 0, nullptr, 0, 0, du_g, gg.K2, nullptr, nullptr, 0, s, M, gg.K2));
    if (!grouped) RC(lora_dw(m, st, gg, m->dgu, 2 * I, a.u_gu, a.h2, H, du_g, M));
    RC(base_weight(m, st, l, 2, &Wd, M, H, 2 * I));
    RC(gemm_l(m, CAT_GEMM, 2, st, m->dgu, 2 * I, Wd, H, 2 * I, du_g, gg.K2, ar + gg.acat, H, gg.K2, m->dh, H, nullptr, nullptr, 0, 1.f, M, H,
               0, nullptr, 0, yg ? ar + gg.bcat : nullptr, gg.K2, s));
    PM(CAT_ROW, 4.0 * M * H * 2);
    RC(b200rl_rmsnorm_bwd(m->dh, a.x_mid, w.ln2_w, a.rstd2, m->dx, m->dx2, M, H, stream));
    // ---- o projection:  x_mid = x + attn_o.Wo^T + u_o.Bo^T
    if (!yo) RC(gemm_l(m, CAT_GEMM_SKINNY, 2, st, m->dx2, H, ar + go.bcat, go.K2, H, nullptr, 0, nullptr, 0, 0, du_o, go.K2, nullptr, nullptr, 0, s, M, go.K2));
    if (!grouped) RC(lora_dw(m, st, go, m->dx2, H, a.u_o, a.attn_o, QD, du_o, M));
    RC(base_weight(m, st, l, 1, &Wd, M, QD, H));
    RC(gemm_l(m, CAT_GEMM, 2, st, m->dx2, H, Wd, QD, H, du_o, go.K2, ar + go.acat, QD, go.K2, m->dattn, QD, nullptr, nullptr, 0, 1.f, M, QD,
               0, nullptr, 0, yo ? ar + go.bcat : nullptr, go.K2, s));
    // ---- attention + rope
    PM(CAT_ATTN_BWD, 4.0 * B * c.n_q_heads * (double)L * L * c.head_dim);
    if (pb) RC(b200rl_attn_seg_bwd(a.qkv, attn_mask, a.attn_o, m->dattn, a.lse, m->delta, m->dqkv, m->kvpart, M, c.n_q_heads, c.n_kv_heads, attn_scale,
                                   pb->qblocks, pb->n_qblocks, pb->kblocks, pb->n_kblocks, pb->red_start, pb->red_list, stream));
    else RC(b200rl_attn_bwd(a.qkv, attn_mask, a.attn_o, m->dattn, a.lse, m->delta, m->dqkv, B, L, c.n_q_heads, c.n_kv_heads, c.head_dim, attn_scale, stream));
    PM(CAT_ROW, 2.0 * M * (c.n_q_heads + c.n_kv_heads) * c.head_dim * 2);
    if (pb) RC(b200rl_rope_pos(m->dqkv, m->rope_cs, pb->pos, M, QKV, c.n_q_heads + c.n_kv_heads, c.head_dim, 1, stream));
    else RC(b200rl_rope(m->dqkv, m->rope_cs, M, L, QKV, c.n_q_heads + c.n_kv_heads, c.head_dim, 1, stream));
    // ---- qkv projection:  qkv = h1.Wqkv^T + u_qkv.Bqkv^T + bias
    if (!yq) RC(gemm_l(m, CAT_GEMM_SKINNY, 2, st, m->dqkv, QKV, ar + gq.bcat, gq.K2, QKV, nullptr, 0, nullptr, 0, 0, du_q, gq.K2, nullptr, nullptr, 0, s, M, gq.K2));
    if (!grouped) RC(lora_dw(m, st, gq, m->dqkv, QKV, a.u_qkv, a.h1, H, du_q, M));
    if (yq) {   // the qkv dX GEMM produces du_q: it has to run before the grouped dW launch that consumes it
      RC(base_weight(m, st, l, 0, &Wd, M, H, QKV));
      RC(gemm_l(m, CAT_GEMM, 2, st, m->dqkv, QKV, Wd, H, QKV, du_q, gq.K2, ar + gq.acat, H, gq.K2, m->dh, H, nullptr, nullptr, 0, 1.f, M, H,
                 0, nullptr, 0, ar + gq.bcat, gq.K2, s));
    }
    if (grouped) {
      // all eight dB / dA GEMMs of the layer in one launch, all their blocks accumulated by one more
      const Group* gs[4] = {&gd, &gg, &go, &gq};
      const bf16* dYs[4] = {m->dx, m->dgu, m->dx2, m->dqkv};
      const long long ldYs[4] = {H, 2 * I, H, QKV};
      const bf16* us[4] = {a.u_d, a.u_gu, a.u_o, a.u_qkv};
      const bf16* xs[4] = {a.act, a.h2, a.attn_o, a.h1};
      const long long ldXs[4] = {I, H, QD, H};
      const bf16* dus[4] = {du_d, du_g, du_o, du_q};
      RC(lora_dw_grouped(m, st, gs, dYs, ldYs, us, xs, ldXs, dus, M));
    }
    if (l > 0) {  // embeddings are frozen: layer 0 needs no input gradient
      if (!yq) {
        RC(base_weight(m, st, l, 0, &Wd, M, H, QKV));
        RC(gemm_l(m, CAT_GEMM, 2, st, m->dqkv, QKV, Wd, H, QKV, du_q, gq.K2, ar + gq.acat, H, gq.K2, m->dh, H, nullptr, nullptr, 0, 1.f, M, H));
      }
      PM(CAT_ROW, 4.0 * M * H * 2);
      RC(b200rl_rmsnorm_bwd(m->dh, x, w.ln1_w, a.rstd1, m->dx2, m->dx, M, H, stream));
    }
  }
  PM(CAT_END, 0);
  return 0;
}

// ---- resident dequantised-weight cache ---------------------------------------------------------------
extern "C" long long b200rl_model_weight_cache_bytes(const b200rl_model_config* c) {
  if (!c) return -1;
  const long long QKV = (long long)(c->n_q_heads + 2 * c->n_kv_heads) * c->head_dim, QD = (long long)c->n_q_heads * c->head_dim;
  const long long per = QKV * c->hidden + c->hidden * QD + 2LL * c->inter * c->hidden + (long long)c->hidden * c->inter;
  return per * 2 * c->n_layers;
}
extern "C" int b200rl_model_set_weight_cache(b200rl_model* m, void* buf, long long bytes) {
  B200RL_REQUIRE(m != nullptr, "model_set_weight_cache: null model");
  if (!buf) { m->wcache = nullptr; return 0; }
  const long long need = b200rl_model_weight_cache_bytes(&m->cfg);
  B200RL_REQUIRE(bytes >= need, "model_set_weight_cache: buffer too small");
  B200RL_REQUIRE((reinterpret_cast<uintptr_t>(buf) & 1023) == 0, "model_set_weight_cache: buffer must be 1024-byte aligned");
  m->wcache = (bf16*)buf;
  m->wcache_per_layer = need / 2 / m->cfg.n_layers;
  m->wcache_valid.assign((size_t)m->cfg.n_layers * 4, 0);
  return 0;
}

// Without a weight cache: 1 = the GEMMs dequantise the NF4 base inside their mainloop (north_star), 0 = each matrix is
// dequantised into the shared scratch right before its GEMM.  Same bits either way (tests/test_gpu_learner.py).
extern "C" int b200rl_model_set_nf4_inkernel(b200rl_model* m, int enable) {
  B200RL_REQUIRE(m != nullptr, "model_set_nf4_inkernel: null model");
  m->nf4_inkernel = enable != 0;
  return 0;
}

// bit 0: SwiGLU fused into the gate|up / down-dX GEMM epilogues (default on; results are bit-identical either way)
extern "C" int b200rl_model_set_fusion(b200rl_model* m, int flags) {
  B200RL_REQUIRE(m != nullptr, "model_set_fusion: null model");
  m->fuse_swiglu = (flags & 1) != 0;
  return 0;
}

// ---- profiling API (bench.py) ---------------------------------------------------------------------
extern "C" int b200rl_model_profile(b200rl_model* m, int enable) {
  B200RL_REQUIRE(m != nullptr, "model_profile: null model");
  if (enable && m->prof_ev.empty()) {
    const int cap = 1 << 16;
    m->prof_ev.resize(cap);
    m->prof_cat.resize(cap);
    m->prof_work.resize(cap);
    for (int i = 0; i < cap; ++i) B200RL_CUDA_OK(cudaEventCreate(&m->prof_ev[i]));
  }
  m->prof_on = enable != 0;
  m->prof_n = 0;
  return 0;
}

// Sums per category since the last read: ms[NCAT], work[NCAT] (flops or bytes), count[NCAT]. Synchronises.
extern "C" int b200rl_model_profile_read(b200rl_model* m, double* ms, double* work, long long* count) {
  B200RL_REQUIRE(m && ms && work && count, "model_profile_read: null pointer");
  for (int i = 0; i < NCAT; ++i) { ms[i] = 0; work[i] = 0; count[i] = 0; }
  if (m->prof_n > 0) B200RL_CUDA_OK(cudaEventSynchronize(m->prof_ev[m->prof_n - 1]));
  for (int i = 0; i + 1 < m->prof_n; ++i) {
    const int c = m->prof_cat[i];
    if (c < 0) continue;
    float t = 0.f;
    B200RL_CUDA_OK(cudaEventElapsedTime(&t, m->prof_ev[i], m->prof_ev[i + 1]));
    ms[c] += t; work[c] += m->prof_work[i]; count[c] += 1;
  }
  m->prof_n = 0;
  return 0;
}

static int classic_pass(b200rl_model* m, const int* ids, const int* attn_mask, const int* answer_mask, const double* adv,
                        float* lp_out, double* loss_accum, int B, int P, int T, int nb, int grpo, int backward,
                        int lora_off, const float* ref_lp, double kl_beta, const float* old_lp, double clip_eps,
                        const b200rl_entropy_args* ent, void* stream) {
  B200RL_REQUIRE(m && ids && attn_mask && answer_mask, "model_microbatch: null pointer");
  const b200rl_model_config& c = m->cfg;
  const int L = P + T;
  B200RL_REQUIRE(B > 0 && P >= 1 && T >= 1, "model_microbatch: need B>0, P>=1, T>=1 (B=%d P=%d T=%d)", B, P, T);
  B200RL_REQUIRE(B * L <= c.max_tokens && B <= c.max_batch && L <= c.max_seq && B * T <= c.max_score_rows,
                 "model_microbatch: batch exceeds the workspace (B=%d L=%d)", B, L);
  Layout lay;
  lay.M = B * L; lay.B = B; lay.T = T; lay.L = L; lay.P = P;
  lay.ids = ids; lay.key_mask = attn_mask; lay.answer_mask = answer_mask; lay.pb = nullptr;
  return run_microbatch(m, lay, adv, lp_out, loss_accum, nb, grpo, backward, lora_off, ref_lp, kl_beta, old_lp, clip_eps, ent,
                        stream);
}

extern "C" int b200rl_model_microbatch_ex(b200rl_model* m, const int* ids, const int* attn_mask,
                                          const int* answer_mask, const double* adv, float* lp_out,
                                          double* loss_accum, int B, int P, int T, int nb, int grpo,
                                          int backward, int lora_off, const float* ref_lp, double kl_beta,
                                          void* stream) {
  return classic_pass(m, ids, attn_mask, answer_mask, adv, lp_out, loss_accum, B, P, T, nb, grpo, backward, lora_off, ref_lp,
                      kl_beta, nullptr, 0.0, nullptr, stream);
}

extern "C" int b200rl_model_microbatch(b200rl_model* m, const int* ids, const int* attn_mask,
                                       const int* answer_mask, const double* adv, float* lp_out,
                                       double* loss_accum, int B, int P, int T, int nb, int grpo,
                                       int backward, void* stream) {
  return b200rl_model_microbatch_ex(m, ids, attn_mask, answer_mask, adv, lp_out, loss_accum, B, P, T, nb, grpo,
                                    backward, 0, nullptr, 0.0, stream);
}

static int packed_pass(b200rl_model* m, const b200rl_packed_batch* pb, const double* adv, float* lp_out,
                       double* loss_accum, int nb, int grpo, int backward, int lora_off, const float* ref_lp,
                       double kl_beta, const float* old_lp, double clip_eps, const b200rl_entropy_args* ent,
                       void* stream) {
  B200RL_REQUIRE(m && pb, "model_microbatch_packed: null pointer");
  const b200rl_model_config& c = m->cfg;
  B200RL_REQUIRE(c.head_dim == 128, "model_microbatch_packed: the packed layout needs head_dim 128 (tcgen05 attention)");
  B200RL_REQUIRE(pb->ids && pb->pos && pb->key_mask && pb->score_src && pb->targets && pb->answer_mask &&
                     pb->sc_start && pb->sc_list && pb->qblocks && pb->kblocks && pb->red_start && pb->red_list,
                 "model_microbatch_packed: null array");
  B200RL_REQUIRE(pb->rows > 0 && pb->rows <= c.max_tokens && pb->B > 0 && pb->B <= c.max_batch && pb->T >= 1 &&
                     pb->B * pb->T <= c.max_score_rows && pb->max_pos >= 1 && pb->max_pos <= c.max_seq,
                 "model_microbatch_packed: batch exceeds the workspace (rows=%d B=%d T=%d)", pb->rows, pb->B, pb->T);
  B200RL_REQUIRE(pb->n_score >= 0 && pb->n_score <= pb->B * pb->T && (pb->n_score == 0 || pb->score_slot),
                 "model_microbatch_packed: n_score=%d outside [0, B*T=%d] or score_slot missing", pb->n_score, pb->B * pb->T);
  B200RL_REQUIRE(pb->part_rows <= m->kvpart_rows, "model_microbatch_packed: %d dK/dV partial rows > capacity %lld",
                 pb->part_rows, m->kvpart_rows);
  Layout lay;
  lay.M = pb->rows; lay.B = pb->B; lay.T = pb->T; lay.L = pb->max_pos; lay.P = 0;
  lay.ids = pb->ids; lay.key_mask = pb->key_mask; lay.answer_mask = pb->answer_mask; lay.pb = pb;
  return run_microbatch(m, lay, adv, lp_out, loss_accum, nb, grpo, backward, lora_off, ref_lp, kl_beta, old_lp, clip_eps, ent,
                        stream);
}

extern "C" int b200rl_model_microbatch_packed(b200rl_model* m, const b200rl_packed_batch* pb, const double* adv,
                                              float* lp_out, double* loss_accum, int nb, int grpo, int backward,
                                              int lora_off, const float* ref_lp, double kl_beta, void* stream) {
  return packed_pass(m, pb, adv, lp_out, loss_accum, nb, grpo, backward, lora_off, ref_lp, kl_beta, nullptr, 0.0, nullptr,
                     stream);
}

// general forms: the loss terms in one argument block (include/b200rl.h b200rl_loss_args)
extern "C" int b200rl_model_pass(b200rl_model* m, const int* ids, const int* attn_mask, const int* answer_mask,
                                 const double* adv, float* lp_out, double* loss_accum, int B, int P, int T,
                                 const b200rl_loss_args* a, void* stream) {
  return b200rl_model_pass_ent(m, ids, attn_mask, answer_mask, adv, lp_out, loss_accum, B, P, T, a, nullptr, stream);
}
extern "C" int b200rl_model_pass_packed(b200rl_model* m, const b200rl_packed_batch* pb, const double* adv, float* lp_out,
                                        double* loss_accum, const b200rl_loss_args* a, void* stream) {
  return b200rl_model_pass_packed_ent(m, pb, adv, lp_out, loss_accum, a, nullptr, stream);
}

// with the per-token entropy / entropy bonus (reference: compute_entropy_bonus, distributed_actor.py:266-281; call sites
// commented out at :377-379 and :472-480).  ent NULL = b200rl_model_pass / b200rl_model_pass_packed.
extern "C" int b200rl_model_pass_ent(b200rl_model* m, const int* ids, const int* attn_mask, const int* answer_mask,
                                     const double* adv, float* lp_out, double* loss_accum, int B, int P, int T,
                                     const b200rl_loss_args* a, const b200rl_entropy_args* ent, void* stream) {
  B200RL_REQUIRE(a != nullptr, "model_pass: null args");
  return classic_pass(m, ids, attn_mask, answer_mask, adv, lp_out, loss_accum, B, P, T, a->nb, a->grpo, a->backward,
                      a->lora_off, a->ref_lp, a->kl_beta, a->old_lp, a->clip_eps, ent, stream);
}
extern "C" int b200rl_model_pass_packed_ent(b200rl_model* m, const b200rl_packed_batch* pb, const double* adv,
                                            float* lp_out, double* loss_accum, const b200rl_loss_args* a,
                                            const b200rl_entropy_args* ent, void* stream) {
  B200RL_REQUIRE(a != nullptr, "model_pass_packed: null args");
  return packed_pass(m, pb, adv, lp_out, loss_accum, a->nb, a->grpo, a->backward, a->lora_off, a->ref_lp, a->kl_beta,
                     a->old_lp, a->clip_eps, ent, stream);
}
