// G7: token-gather / log-softmax / advantage-scale in ONE coalesced pass over the logits.
//
// Reference: BaseLearner.compute_current_policy_probs per-row log_softmax + gather
// (distributed_actor.py:252-260), PG loss (:375), GRPO loss (:467-470), 1/num_batches scaling
// (:382, :479) and the autograd backward of all of it (:385, :483).
//
// Because the loss is linear in the per-token log-probs with coefficients that depend only on
// (advantage, answer mask, length, batch sizes),
//     d loss / d lp[i,t] = coef[i,t] = -A_i * mask[i,t] / (len_i * B_m * nb),
// forward and backward fuse: pass 1 streams a logits row once (online max / sum-exp, fp32 like the
// reference's autocast log_softmax), pass 2 re-reads the row (L2-resident: 304 KB per row at
// V=152064) and overwrites it in place with dlogits = coef * (onehot(y) - softmax(z)).
// HBM traffic = read T*V*2 + write T*V*2 bytes; the reference saves an fp32 [T,V] log-prob tensor
// per row for autograd instead.
#include "common.cuh"

namespace b200rl {

static constexpr float LOG2E = 1.4426950408889634f;
static constexpr float LN2 = 0.6931471805599453f;

// Optional per-token entropy (ENT = true; reference helper BaseLearner.compute_entropy_bonus, distributed_actor.py:266-281,
// whose call sites are commented out at :377-379 and :472-480):
//   H = -sum_v p_v ln p_v,  p = softmax(z) at temperature 1, fp32.
// Pass 1 carries a third running quantity next to (m, s) in the log2 domain, shifted by the running max m:
//   u = sum_v 2^(y_v - m) (y_v - m),  y = z log2(e);  when m moves to m' > m:  u' = 2^(m - m') (u + s (m - m')).
// Then H = ln2 (log2 s - u / s), which stays accurate on peaked rows (lse - E[z] cancels there).
// Pass 2 adds the gradient of the bonus term -e * H, e = alpha * mask / (len * Bm * nb):
//   d(-e H)/dz_v = e p_v (ln p_v + H),  ln p_v = (y_v - lse2) ln2 (no extra exp / log).
// merge (om, os, ou) into (m, s, u); nm = max(m, om).  A side with s == 0 (m == -inf) contributes nothing.
__device__ __forceinline__ void ent_combine(float m, float s, float& u, float om, float os, float ou, float nm) {
  const float a = s > 0.f ? exp2f(m - nm) * (u + s * (m - nm)) : 0.f;
  const float b = os > 0.f ? exp2f(om - nm) * (ou + os * (om - nm)) : 0.f;
  u = a + b;
}

struct EntArgs {
  const int* mask;   // [Bm*T] answer mask; e = 0 where it is 0
  const int* lens;   // [Bm] answer lengths (loss_coef); NULL = e = 0 (scoring only)
  int T, Bm, nb;
  double alpha;
  float* ent_out;    // [Bm*T] per-token H (through slot)
};

// one CTA per row
template <bool ENT>
__device__ __forceinline__ void logprob_row(bf16* __restrict__ logits, long long ld, const int* __restrict__ targets,
                                            const float* __restrict__ coef, const float* __restrict__ klw,
                                            const float* __restrict__ ref_lp, const float* __restrict__ old_lp,
                                            float clip_eps, float* __restrict__ lp_out, int V, int write_grad,
                                            const int* __restrict__ slot, const EntArgs& ea) {
  __shared__ float red_m[32], red_s[32], red_u[32];
  __shared__ float s_lse2, s_max2, s_ent;
  const size_t row = blockIdx.x;
  bf16* z = logits + row * ld;
  const bf16x8* zv = reinterpret_cast<const bf16x8*>(z);
  const int nvec = V / 8;  // V % 8 == 0 checked on host
  // ---- pass 1: online softmax statistics in the log2 domain ----
  float m = -INFINITY, s = 0.f, u = 0.f;
  for (int i = threadIdx.x; i < nvec; i += blockDim.x) {
    float f[8];
    unpack8(zv[i], f);
    float lm = f[0];
#pragma unroll
    for (int j = 1; j < 8; ++j) lm = fmaxf(lm, f[j]);
    lm *= LOG2E;
    if (lm > m) {
      if constexpr (ENT) {
        const float sc = exp2f(m - lm);
        u = s > 0.f ? sc * (u + s * (m - lm)) : 0.f;
        s *= sc;
      } else {
        s *= exp2f(m - lm);
      }
      m = lm;
    }
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      if constexpr (ENT) {
        const float d = f[j] * LOG2E - m;
        const float ex = exp2f(d);
        s += ex;
        u += ex * d;
      } else {
        s += exp2f(f[j] * LOG2E - m);
      }
    }
  }
  // warp then block combine of (m, s[, u])
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const float om = __shfl_xor_sync(0xffffffffu, m, o);
    const float os = __shfl_xor_sync(0xffffffffu, s, o);
    const float nm = fmaxf(m, om);
    if constexpr (ENT) {
      const float ou = __shfl_xor_sync(0xffffffffu, u, o);
      ent_combine(m, s, u, om, os, ou, nm);
    }
    s = (nm == -INFINITY) ? 0.f : s * exp2f(m - nm) + os * exp2f(om - nm);
    m = nm;
  }
  const int w = threadIdx.x >> 5, l = threadIdx.x & 31;
  if (l == 0) {
    red_m[w] = m;
    red_s[w] = s;
    if constexpr (ENT) red_u[w] = u;
  }
  __syncthreads();
  if (w == 0) {
    const int nw = blockDim.x >> 5;
    m = l < nw ? red_m[l] : -INFINITY;
    s = l < nw ? red_s[l] : 0.f;
    if constexpr (ENT) u = l < nw ? red_u[l] : 0.f;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      const float om = __shfl_xor_sync(0xffffffffu, m, o);
      const float os = __shfl_xor_sync(0xffffffffu, s, o);
      const float nm = fmaxf(m, om);
      if constexpr (ENT) {
        const float ou = __shfl_xor_sync(0xffffffffu, u, o);
        ent_combine(m, s, u, om, os, ou, nm);
      }
      s = (nm == -INFINITY) ? 0.f : s * exp2f(m - nm) + os * exp2f(om - nm);
      m = nm;
    }
    if (l == 0) {
      s_max2 = m;
      s_lse2 = m + log2f(s);  // log2-sum-exp2
      if constexpr (ENT) s_ent = LN2 * (log2f(s) - u / s);
    }
  }
  __syncthreads();
  const float lse2 = s_lse2;
  // compacted scoring (packed layout, live rows only): logits / targets are per compacted row, the per-token arrays
  // (coef, klw, ref_lp, old_lp, lp_out) stay [B*T] and are addressed through the row's slot
  const size_t sl = slot ? (size_t)slot[row] : row;
  const int y = targets[row];
  const float zy = (y >= 0 && y < V) ? __bfloat162float(z[y]) : 0.f;
  const float lp = (y >= 0 && y < V) ? (zy * LOG2E - lse2) * LN2 : 0.f;
  float c = coef ? coef[sl] : 0.f;
  // optional clipped-ratio surrogate (not in the reference, whose ratio exp(lp - lp.detach()) is identically 1,
  // distributed_actor.py:467): loss_t = -min(rho A, clip(rho, 1-eps, 1+eps) A) with rho = exp(lp - old_lp), so
  // d loss_t / d lp = -A rho while the unclipped branch is the active minimum and 0 once rho has left the trust region in
  // the direction the advantage pushes.  coef carries -A mask / (len Bm nb): its sign is that of -A.
  if (old_lp && clip_eps > 0.f && c != 0.f) {
    const float rho = __expf(lp - old_lp[sl]);
    const bool active = c < 0.f ? rho <= 1.f + clip_eps : rho >= 1.f - clip_eps;
    c = active ? c * rho : 0.f;
  }
  // optional KL(pi || pi_ref) term, k3 estimator exp(q-p) - (q-p) - 1 per token:
  // d k3 / d lp = 1 - exp(q - p); klw carries beta * mask / (len * Bm * nb)   (not in the reference: beta = 0)
  if (klw && ref_lp && klw[sl] != 0.f) c += klw[sl] * (1.f - __expf(ref_lp[sl] - lp));
  if (threadIdx.x == 0 && lp_out) lp_out[sl] = lp;
  float H = 0.f, e = 0.f;
  if constexpr (ENT) {
    H = s_ent;
    if (threadIdx.x == 0) ea.ent_out[sl] = H;
    const int len = ea.lens ? ea.lens[sl / ea.T] : 0;
    if (len > 0 && ea.mask[sl] != 0 && ea.alpha != 0.0)
      e = (float)(ea.alpha / ((double)len * (double)ea.Bm * (double)ea.nb));
  }
  if (!write_grad) return;
  __syncthreads();  // z[y] read above must precede the in-place overwrite
  // ---- pass 2: dz = coef * (onehot - softmax) [+ e p (ln p + H)], in place ----
  bf16x8* zw = reinterpret_cast<bf16x8*>(z);
  if (c == 0.f && (!ENT || e == 0.f)) {
    bf16x8 zero;
    zero.u = make_uint4(0u, 0u, 0u, 0u);
    for (int i = threadIdx.x; i < nvec; i += blockDim.x) zw[i] = zero;
    return;
  }
  for (int i = threadIdx.x; i < nvec; i += blockDim.x) {
    float f[8];
    unpack8(zv[i], f);
    const int base = i * 8;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      if constexpr (ENT) {
        const float t = f[j] * LOG2E - lse2;   // log2 p
        const float p = exp2f(t);
        f[j] = c * (((base + j) == y ? 1.f : 0.f) - p) + e * p * (t * LN2 + H);
      } else {
        const float p = exp2f(f[j] * LOG2E - lse2);
        f[j] = c * (((base + j) == y ? 1.f : 0.f) - p);
      }
    }
    zw[i] = pack8(f);
  }
}

__global__ void __launch_bounds__(1024)
logprob_kernel(bf16* __restrict__ logits, long long ld, const int* __restrict__ targets,
               const float* __restrict__ coef, const float* __restrict__ klw,
               const float* __restrict__ ref_lp, const float* __restrict__ old_lp, float clip_eps,
               float* __restrict__ lp_out, int V, int write_grad, const int* __restrict__ slot) {
  logprob_row<false>(logits, ld, targets, coef, klw, ref_lp, old_lp, clip_eps, lp_out, V, write_grad, slot, EntArgs{});
}

__global__ void __launch_bounds__(1024)
logprob_entropy_kernel(bf16* __restrict__ logits, long long ld, const int* __restrict__ targets,
                       const float* __restrict__ coef, const float* __restrict__ klw,
                       const float* __restrict__ ref_lp, const float* __restrict__ old_lp, float clip_eps,
                       float* __restrict__ lp_out, int V, int write_grad, const int* __restrict__ slot, EntArgs ea) {
  logprob_row<true>(logits, ld, targets, coef, klw, ref_lp, old_lp, clip_eps, lp_out, V, write_grad, slot, ea);
}

// ------------------------------------------------------------------------------------------
// loss coefficients (reference :375 / :470 with :382 / :479 scaling), fp64 like the reference's
// float64 rewards tensor (:350, :441), emitted as fp32 per scored token:
//   len_i = sum_t mask[i,t];  coef[i,t] = -A_i * mask[i,t] / (len_i * Bm * nb)   (0 when len_i = 0)
// ------------------------------------------------------------------------------------------
__global__ void loss_coef_kernel(const int* __restrict__ mask, const double* __restrict__ adv,
                                 float* __restrict__ coef, float* __restrict__ klw, double beta,
                                 int* __restrict__ lens, int T, int Bm, int nb) {
  __shared__ int red[32];
  const int i = blockIdx.x;
  int cnt = 0;
  for (int t = threadIdx.x; t < T; t += blockDim.x) cnt += mask[(size_t)i * T + t] != 0;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = cnt;
  __syncthreads();
  if (threadIdx.x < 32) {
    int t = threadIdx.x < (blockDim.x >> 5) ? red[threadIdx.x] : 0;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) t += __shfl_xor_sync(0xffffffffu, t, o);
    if (threadIdx.x == 0) red[0] = t;
  }
  __syncthreads();
  const int len = red[0];
  if (threadIdx.x == 0 && lens) lens[i] = len;
  const double base = len > 0 ? -adv[i] / ((double)len * (double)Bm * (double)nb) : 0.0;
  const double kbase = len > 0 ? beta / ((double)len * (double)Bm * (double)nb) : 0.0;
  for (int t = threadIdx.x; t < T; t += blockDim.x) {
    const bool on = mask[(size_t)i * T + t] != 0;
    coef[(size_t)i * T + t] = on ? (float)base : 0.f;
    if (klw) klw[(size_t)i * T + t] = on ? (float)kbase : 0.f;
  }
}

// loss value of one micro-batch, accumulated on the device (no per-micro-batch .item() sync):
//   PG   (:375): loss_m = -(1/Bm) sum_i A_i * (sum_t mask*lp) / len_i
//   GRPO (:467-470): importance = exp(lp - lp.detach()) == 1  =>  loss_m = -(1/Bm) sum_i A_i * [len_i>0]
// The reference's returned scalar is the SUM of loss_m over micro-batches (quirk Q2) -> *accum += loss_m.
// ENT: also L_H = -alpha (1/Bm) sum_i [len_i>0] (sum_t mask H) / len_i, and ent_accum[0] += sum mask*H,
// ent_accum[1] += sum mask (single CTA, fixed order: deterministic).
template <bool ENT>
__device__ __forceinline__ void loss_value_body(const float* __restrict__ lp, const int* __restrict__ mask,
                                                const double* __restrict__ adv, const float* __restrict__ ref_lp,
                                                double beta, const float* __restrict__ old_lp, double clip_eps,
                                                double* __restrict__ accum, int Bm, int T, int grpo,
                                                const float* __restrict__ ent, double alpha,
                                                double* __restrict__ ent_accum) {
  __shared__ double red[32];
  __shared__ double rede[32];
  double total = 0.0, ent_sum = 0.0, ent_n = 0.0;
  for (int i = 0; i < Bm; ++i) {
    double s = 0.0, kl = 0.0, hs = 0.0;
    int cnt = 0;
    for (int t = threadIdx.x; t < T; t += blockDim.x) {
      if (mask[(size_t)i * T + t] != 0) {
        if constexpr (ENT) hs += (double)ent[(size_t)i * T + t];
        const double p = (double)lp[(size_t)i * T + t];
        if (old_lp && clip_eps > 0.0) {   // clipped surrogate: s accumulates min(rho A, clip(rho) A) instead of lp
          const double rho = exp(p - (double)old_lp[(size_t)i * T + t]);
          const double a = adv[i];
          const double cl = fmin(fmax(rho, 1.0 - clip_eps), 1.0 + clip_eps);
          s += fmin(rho * a, cl * a);
        } else {
          s += p;
        }
        cnt += 1;
        if (ref_lp) {
          const double d = (double)ref_lp[(size_t)i * T + t] - p;
          kl += exp(d) - d - 1.0;
        }
      }
    }
    s = warp_sum_d(s);
    kl = warp_sum_d(kl);
    if constexpr (ENT) hs = warp_sum_d(hs);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
    __syncthreads();
    __shared__ double redk[32];
    if ((threadIdx.x & 31) == 0) {
      red[threadIdx.x >> 5] = s;
      redk[threadIdx.x >> 5] = kl;
      if constexpr (ENT) rede[threadIdx.x >> 5] = hs;
    }
    __shared__ int redc[32];
    if ((threadIdx.x & 31) == 0) redc[threadIdx.x >> 5] = cnt;
    __syncthreads();
    if (threadIdx.x == 0) {
      double ss = 0.0, kk = 0.0, hh = 0.0;
      int cc = 0;
      for (int w = 0; w < (blockDim.x >> 5); ++w) {
        ss += red[w];
        kk += redk[w];
        cc += redc[w];
        if constexpr (ENT) hh += rede[w];
      }
      const bool clipped = old_lp && clip_eps > 0.0;
      if (cc > 0) total += (clipped ? ss / (double)cc : (grpo ? adv[i] : adv[i] * (ss / (double)cc))) - beta * (kk / (double)cc);
      if constexpr (ENT) {
        if (cc > 0 && alpha != 0.0) total += alpha * (hh / (double)cc);
        ent_sum += hh;
        ent_n += (double)cc;
      }
    }
    __syncthreads();
  }
  if (threadIdx.x == 0) *accum += -total / (double)Bm;
  if constexpr (ENT) {
    if (threadIdx.x == 0 && ent_accum) {
      ent_accum[0] += ent_sum;
      ent_accum[1] += ent_n;
    }
  }
}

__global__ void loss_value_kernel(const float* __restrict__ lp, const int* __restrict__ mask,
                                  const double* __restrict__ adv, const float* __restrict__ ref_lp,
                                  double beta, const float* __restrict__ old_lp, double clip_eps,
                                  double* __restrict__ accum, int Bm, int T, int grpo) {
  loss_value_body<false>(lp, mask, adv, ref_lp, beta, old_lp, clip_eps, accum, Bm, T, grpo, nullptr, 0.0, nullptr);
}

__global__ void loss_value_entropy_kernel(const float* __restrict__ lp, const int* __restrict__ mask,
                                          const double* __restrict__ adv, const float* __restrict__ ref_lp,
                                          double beta, const float* __restrict__ old_lp, double clip_eps,
                                          double* __restrict__ accum, int Bm, int T, int grpo,
                                          const float* __restrict__ ent, double alpha, double* __restrict__ ent_accum) {
  loss_value_body<true>(lp, mask, adv, ref_lp, beta, old_lp, clip_eps, accum, Bm, T, grpo, ent, alpha, ent_accum);
}

}  // namespace b200rl

using namespace b200rl;
#define STREAM reinterpret_cast<cudaStream_t>(stream)

extern "C" int b200rl_logprob_kl(void* logits, long long ld, const int* targets, const float* coef,
                                 const float* klw, const float* ref_lp, float* lp_out, int rows, int V,
                                 int write_grad, void* stream) {
  B200RL_REQUIRE(logits && targets && rows > 0 && V > 0 && V % 8 == 0 && ld % 8 == 0,
                 "logprob: bad args (rows=%d V=%d ld=%lld)", rows, V, ld);
  B200RL_REQUIRE(!write_grad || coef, "logprob: write_grad needs coef");
  const int threads = V >= 8192 ? 1024 : 256;
  logprob_kernel<<<rows, threads, 0, STREAM>>>((bf16*)logits, ld, targets, coef, klw, ref_lp, nullptr, 0.f, lp_out, V,
                                               write_grad, nullptr);
  B200RL_LAUNCH_OK();
  return 0;
}

extern "C" int b200rl_logprob(void* logits, long long ld, const int* targets, const float* coef,
                              float* lp_out, int rows, int V, int write_grad, void* stream) {
  B200RL_REQUIRE(logits && targets && rows > 0 && V > 0 && V % 8 == 0 && ld % 8 == 0,
                 "logprob: bad args (rows=%d V=%d ld=%lld)", rows, V, ld);
  B200RL_REQUIRE(!write_grad || coef, "logprob: write_grad needs coef");
  const int threads = V >= 8192 ? 1024 : 256;
  logprob_kernel<<<rows, threads, 0, STREAM>>>((bf16*)logits, ld, targets, coef, nullptr, nullptr, nullptr, 0.f, lp_out,
                                               V, write_grad, nullptr);
  B200RL_LAUNCH_OK();
  return 0;
}

extern "C" int b200rl_loss_coef_kl(const int* mask, const double* adv, float* coef, float* klw, double beta,
                                   int* lens, int Bm, int T, int nb, void* stream) {
  B200RL_REQUIRE(mask && adv && coef && Bm > 0 && T > 0 && nb > 0, "loss_coef: bad args");
  loss_coef_kernel<<<Bm, 256, 0, STREAM>>>(mask, adv, coef, klw, beta, lens, T, Bm, nb);
  B200RL_LAUNCH_OK();
  return 0;
}

extern "C" int b200rl_loss_coef(const int* mask, const double* adv, float* coef, int* lens, int Bm,
                                int T, int nb, void* stream) {
  B200RL_REQUIRE(mask && adv && coef && Bm > 0 && T > 0 && nb > 0, "loss_coef: bad args");
  loss_coef_kernel<<<Bm, 256, 0, STREAM>>>(mask, adv, coef, nullptr, 0.0, lens, T, Bm, nb);
  B200RL_LAUNCH_OK();
  return 0;
}

extern "C" int b200rl_loss_value_kl(const float* lp, const int* mask, const double* adv, const float* ref_lp,
                                    double beta, double* accum, int Bm, int T, int grpo, void* stream) {
  B200RL_REQUIRE(lp && mask && adv && accum && Bm > 0 && T > 0, "loss_value: bad args");
  loss_value_kernel<<<1, 256, 0, STREAM>>>(lp, mask, adv, ref_lp, beta, nullptr, 0.0, accum, Bm, T, grpo);
  B200RL_LAUNCH_OK();
  return 0;
}

extern "C" int b200rl_loss_value(const float* lp, const int* mask, const double* adv, double* accum,
                                 int Bm, int T, int grpo, void* stream) {
  B200RL_REQUIRE(lp && mask && adv && accum && Bm > 0 && T > 0, "loss_value: bad args");
  loss_value_kernel<<<1, 256, 0, STREAM>>>(lp, mask, adv, nullptr, 0.0, nullptr, 0.0, accum, Bm, T, grpo);
  B200RL_LAUNCH_OK();
  return 0;
}

// Clipped-ratio variants (SURVEY.md 8(f) N4; not in the reference): old_lp [rows] = log-probs of the policy that
// generated the batch, clip_eps = trust-region half width.  old_lp == NULL or clip_eps == 0 is the plain form above.
extern "C" int b200rl_logprob_slots(void* logits, long long ld, const int* targets, const float* coef, const float* klw,
                                    const float* ref_lp, const float* old_lp, double clip_eps, float* lp_out, int rows,
                                    int V, int write_grad, const int* slot, void* stream) {
  B200RL_REQUIRE(logits && targets && rows > 0 && V > 0 && V % 8 == 0 && ld % 8 == 0,
                 "logprob: bad args (rows=%d V=%d ld=%lld)", rows, V, ld);
  B200RL_REQUIRE(!write_grad || coef, "logprob: write_grad needs coef");
  B200RL_REQUIRE(clip_eps >= 0.0, "logprob: clip_eps must be >= 0");
  const int threads = V >= 8192 ? 1024 : 256;
  logprob_kernel<<<rows, threads, 0, STREAM>>>((bf16*)logits, ld, targets, coef, klw, ref_lp, old_lp, (float)clip_eps,
                                               lp_out, V, write_grad, slot);
  B200RL_LAUNCH_OK();
  return 0;
}

extern "C" int b200rl_logprob_clip(void* logits, long long ld, const int* targets, const float* coef, const float* klw,
                                   const float* ref_lp, const float* old_lp, double clip_eps, float* lp_out, int rows,
                                   int V, int write_grad, void* stream) {
  return b200rl_logprob_slots(logits, ld, targets, coef, klw, ref_lp, old_lp, clip_eps, lp_out, rows, V, write_grad,
                              nullptr, stream);
}

extern "C" int b200rl_loss_value_clip(const float* lp, const int* mask, const double* adv, const float* ref_lp,
                                      double beta, const float* old_lp, double clip_eps, double* accum, int Bm, int T,
                                      int grpo, void* stream) {
  B200RL_REQUIRE(lp && mask && adv && accum && Bm > 0 && T > 0, "loss_value: bad args");
  loss_value_kernel<<<1, 256, 0, STREAM>>>(lp, mask, adv, ref_lp, beta, old_lp, clip_eps, accum, Bm, T, grpo);
  B200RL_LAUNCH_OK();
  return 0;
}

// Per-token policy entropy and entropy bonus (reference: BaseLearner.compute_entropy_bonus, distributed_actor.py:266-281,
// call sites commented out in the PG loss :377-379 and the GRPO loss :472-480).  Same arguments as b200rl_logprob_slots
// plus: ent_out [Bm*T] f32 per-token H (required; addressed through slot), and the bonus weight
// e = alpha * mask / (len * Bm * nb) derived from mask [Bm*T] and lens [Bm] (lens NULL or alpha 0: no bonus gradient).
extern "C" int b200rl_logprob_entropy(void* logits, long long ld, const int* targets, const float* coef, const float* klw,
                                      const float* ref_lp, const float* old_lp, double clip_eps, float* lp_out, int rows,
                                      int V, int write_grad, const int* slot, const int* mask, const int* lens, int Bm,
                                      int T, int nb, double alpha, float* ent_out, void* stream) {
  B200RL_REQUIRE(logits && targets && rows > 0 && V > 0 && V % 8 == 0 && ld % 8 == 0,
                 "logprob_entropy: bad args (rows=%d V=%d ld=%lld)", rows, V, ld);
  B200RL_REQUIRE(!write_grad || coef, "logprob_entropy: write_grad needs coef");
  B200RL_REQUIRE(clip_eps >= 0.0, "logprob_entropy: clip_eps must be >= 0");
  B200RL_REQUIRE(ent_out && T > 0, "logprob_entropy: needs ent_out and T > 0");
  B200RL_REQUIRE(alpha == 0.0 || !lens || (mask && Bm > 0 && nb > 0),
                 "logprob_entropy: alpha != 0 with lens needs mask, Bm > 0 and nb > 0");
  const int threads = V >= 8192 ? 1024 : 256;
  EntArgs ea{mask, alpha != 0.0 ? lens : nullptr, T, Bm, nb, alpha, ent_out};
  logprob_entropy_kernel<<<rows, threads, 0, STREAM>>>((bf16*)logits, ld, targets, coef, klw, ref_lp, old_lp,
                                                       (float)clip_eps, lp_out, V, write_grad, slot, ea);
  B200RL_LAUNCH_OK();
  return 0;
}

// loss value with the entropy term (see loss_value_body); ent [Bm*T] = ent_out of b200rl_logprob_entropy,
// ent_accum (device f64[2], optional) += {sum mask*H, sum mask}.
extern "C" int b200rl_loss_value_entropy(const float* lp, const int* mask, const double* adv, const float* ref_lp,
                                         double beta, const float* old_lp, double clip_eps, double* accum, int Bm, int T,
                                         int grpo, const float* ent, double alpha, double* ent_accum, void* stream) {
  B200RL_REQUIRE(lp && mask && adv && accum && Bm > 0 && T > 0, "loss_value_entropy: bad args");
  B200RL_REQUIRE(ent, "loss_value_entropy: needs the per-token entropy");
  loss_value_entropy_kernel<<<1, 256, 0, STREAM>>>(lp, mask, adv, ref_lp, beta, old_lp, clip_eps, accum, Bm, T, grpo, ent,
                                                   alpha, ent_accum);
  B200RL_LAUNCH_OK();
  return 0;
}
