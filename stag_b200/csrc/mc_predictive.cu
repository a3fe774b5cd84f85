// Monte-Carlo predictive statistics in bounded memory: per-node predictive entropy, expected entropy and mutual
// information of S sample outputs, accumulated over any number of calls without an [S,N,C] stack.
//
// The reference keeps the [S,N,C] outputs of its sequential passes and takes their mean (stag/models.py:46-55); the
// uncertainty a user wants from a stochastic GNN is, per node and with p_s the output of sample s,
//   mean          = (1/S) sum_s p_s
//   pred_entropy  = H(mean)                  (total)
//   exp_entropy   = (1/S) sum_s H(p_s)       (aleatoric)
//   mutual_info   = pred_entropy - exp_entropy   (epistemic)
// with H the entropy torch.distributions gives for Categorical(probs=.) / Bernoulli(probs=.) -- the probability
// semantics of nll.cu: renormalise (Categorical), clamp to [eps, 1-eps] before the log, a row that sums to zero or
// holds a NaN gives NaN, an out-of-range label gives NaN.
//
// stag_mc_accumulate adds a chunk of samples into two float64 accumulators (sum of p_s, sum of H(p_s)); one warp owns
// one node row, holds its accumulator row in registers and adds the samples in sample order, so a sequence of calls
// over consecutive chunks yields the same bits whatever the chunk sizes.  No atomics, each probability read once.
// stag_mc_finalize turns the accumulators into the statistics (and the log-likelihood of labels under the mean).
#include "common.cuh"

namespace stag {

constexpr int MC_THREADS = 256, MC_WARPS = MC_THREADS / 32;
constexpr int MC_MAX_C = 1024;                          // 32 slots per lane: the accumulator row stays in registers
constexpr double kMcEps = 1.1920928955078125e-07;       // torch.finfo(float32).eps, as kProbEps in nll.cu

struct McAccParams {
  const float* probs;
  int64_t ld, ss, N;
  int C, S;
  double* acc_sum;  // [N, C] contiguous
  double* acc_ent;  // [N]
};

struct McStatsParams {
  const double* acc_sum;
  const double* acc_ent;
  int64_t N, S;
  int C;
  const int64_t* y_idx;  // categorical: [N]
  const float* y_val;    // bernoulli: [N, C], row stride ldy
  int64_t ldy;
  float *mean, *pred, *expd, *mi, *loglik;
};

__device__ __forceinline__ double mc_warp_sum(double v) {
  // butterfly: every lane ends with the same bits (each step adds the same two values in either order)
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// torch's clamp_probs; a NaN stays NaN (fmin / fmax alone would turn it into a finite value)
__device__ __forceinline__ double mc_clamp(double q) { return q != q ? q : fmin(fmax(q, kMcEps), 1.0 - kMcEps); }

// Categorical(probs=q).entropy() term of one class of a renormalised row: -q log(clamp(q))
__device__ __forceinline__ double cat_term(double q) { return -q * log(mc_clamp(q)); }

// Bernoulli(probs=p).entropy() of one label: binary_cross_entropy_with_logits(logit(clamp(p)), p)
//   = -(p log pc + (1 - p) log(1 - pc))
__device__ __forceinline__ double bern_entropy(double p) {
  const double pc = mc_clamp(p);
  return -(p * log(pc) + (1.0 - p) * log1p(-pc));
}

// the same two terms for the per-sample entropies of the accumulator, in fp32 as torch evaluates them for fp32 outputs:
// a float64 log per read probability made the accumulator compute-bound (0.53 TB/s at the arxiv shape, NVIDIA B200 at 1000 W)
__device__ __forceinline__ float mc_clampf(float q) { return q != q ? q : fminf(fmaxf(q, (float)kMcEps), 1.0f - (float)kMcEps); }
__device__ __forceinline__ float cat_termf(float q) { return -q * logf(mc_clampf(q)); }
__device__ __forceinline__ float bern_entropyf(float p) {
  const float pc = mc_clampf(p);
  return -(p * logf(pc) + (1.0f - p) * log1pf(-pc));
}

// K: slots per lane (C <= 32 K); U: samples whose loads are issued together
template <int KIND, int K, int U>
__global__ void __launch_bounds__(MC_THREADS) mc_accumulate_kernel(const McAccParams p) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int64_t nwarps = (int64_t)gridDim.x * MC_WARPS;
  for (int64_t v = (int64_t)blockIdx.x * MC_WARPS + warp; v < p.N; v += nwarps) {
    double* arow = p.acc_sum + v * p.C;
    const float* row0 = p.probs + v * p.ld;
    double acc[K];
#pragma unroll
    for (int k = 0; k < K; ++k) {
      const int c = lane + 32 * k;
      acc[k] = c < p.C ? arow[c] : 0.0;
    }
    double ent = p.acc_ent[v];
    for (int s0 = 0; s0 < p.S; s0 += U) {
      float x[U][K];
#pragma unroll
      for (int u = 0; u < U; ++u)
#pragma unroll
        for (int k = 0; k < K; ++k) {
          const int c = lane + 32 * k;
          x[u][k] = (s0 + u < p.S && c < p.C) ? __ldg(row0 + (int64_t)(s0 + u) * p.ss + c) : 0.f;
        }
#pragma unroll
      for (int u = 0; u < U; ++u) {
        if (s0 + u >= p.S) break;
        double h = 0.0;
        if (KIND == 0) {
          double sum = 0.0;
#pragma unroll
          for (int k = 0; k < K; ++k) sum += (double)x[u][k];
          const float inv = (float)(1.0 / mc_warp_sum(sum));  // 0 -> inf: q = 0 * inf = NaN, as torch's 0 / 0
#pragma unroll
          for (int k = 0; k < K; ++k)
            if (lane + 32 * k < p.C) h += (double)cat_termf(x[u][k] * inv);
        } else {
#pragma unroll
          for (int k = 0; k < K; ++k)
            if (lane + 32 * k < p.C) h += (double)bern_entropyf(x[u][k]);
        }
        ent += mc_warp_sum(h);
#pragma unroll
        for (int k = 0; k < K; ++k) acc[k] += (double)x[u][k];
      }
    }
#pragma unroll
    for (int k = 0; k < K; ++k) {
      const int c = lane + 32 * k;
      if (c < p.C) arow[c] = acc[k];
    }
    if (lane == 0) p.acc_ent[v] = ent;
  }
}

template <int KIND>
__global__ void __launch_bounds__(MC_THREADS) mc_stats_kernel(const McStatsParams p) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int64_t nwarps = (int64_t)gridDim.x * MC_WARPS;
  const double S = (double)p.S;
  for (int64_t v = (int64_t)blockIdx.x * MC_WARPS + warp; v < p.N; v += nwarps) {
    const double* arow = p.acc_sum + v * p.C;
    float* mrow = p.mean + v * p.C;
    double h = 0.0, ll = 0.0;
    if (KIND == 0) {
      double sum = 0.0;
      for (int c = lane; c < p.C; c += 32) {
        const double m = arow[c] / S;
        mrow[c] = (float)m;
        sum += m;
      }
      const double inv = 1.0 / mc_warp_sum(sum);
      for (int c = lane; c < p.C; c += 32) h += cat_term(arow[c] / S * inv);
      if (p.loglik && lane == 0) {
        const int64_t yv = p.y_idx[v];
        ll = (yv < 0 || yv >= p.C) ? __longlong_as_double(0x7ff8000000000000ULL) : log(mc_clamp(arow[yv] / S * inv));
      }
    } else {
      const float* yrow = p.y_val ? p.y_val + v * p.ldy : nullptr;
      for (int c = lane; c < p.C; c += 32) {
        const double m = arow[c] / S;
        mrow[c] = (float)m;
        h += bern_entropy(m);
        if (yrow) {
          // Bernoulli(probs=m).log_prob(y) = -binary_cross_entropy_with_logits(logit(clamp(m)), y)
          const double pc = mc_clamp(m), yy = (double)yrow[c];
          ll += yy * log(pc) + (1.0 - yy) * log1p(-pc);
        }
      }
      ll = mc_warp_sum(ll);
    }
    h = mc_warp_sum(h);
    if (lane == 0) {
      const double e = p.acc_ent[v] / S;
      p.pred[v] = (float)h;
      p.expd[v] = (float)e;
      p.mi[v] = (float)(h - e);
      if (p.loglik) p.loglik[v] = (float)ll;
    }
  }
}

static int mc_grid(int64_t N) {
  const int64_t want = (N + MC_WARPS - 1) / MC_WARPS;
  const int64_t cap = (int64_t)1 << 20;
  return (int)(want < 1 ? 1 : (want < cap ? want : cap));
}

template <int KIND>
static void launch_accumulate(const McAccParams& p, int grid, cudaStream_t stream) {
  // U x K float loads in flight per lane: enough bytes in flight per warp to cover the latency at small C
  if (p.C <= 32) mc_accumulate_kernel<KIND, 1, 6><<<grid, MC_THREADS, 0, stream>>>(p);
  else if (p.C <= 64) mc_accumulate_kernel<KIND, 2, 4><<<grid, MC_THREADS, 0, stream>>>(p);
  else if (p.C <= 128) mc_accumulate_kernel<KIND, 4, 4><<<grid, MC_THREADS, 0, stream>>>(p);
  else if (p.C <= 256) mc_accumulate_kernel<KIND, 8, 1><<<grid, MC_THREADS, 0, stream>>>(p);
  else if (p.C <= 512) mc_accumulate_kernel<KIND, 16, 1><<<grid, MC_THREADS, 0, stream>>>(p);
  else mc_accumulate_kernel<KIND, 32, 1><<<grid, MC_THREADS, 0, stream>>>(p);
}

}  // namespace stag

using namespace stag;

extern "C" int stag_mc_accumulate(const float* probs, int64_t ld, int64_t sample_stride, int64_t N, int32_t C,
                                  int32_t S, int kind, double* acc_sum, double* acc_ent, void* stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  STAG_CHECK_ARG(N >= 0 && C > 0 && S >= 0, "stag_mc_accumulate: bad sizes N=%lld C=%d S=%d", (long long)N, C, S);
  STAG_CHECK_ARG(kind == 0 || kind == 1, "stag_mc_accumulate: kind must be 0 (categorical) or 1 (bernoulli)");
  STAG_CHECK_ARG(ld >= C, "stag_mc_accumulate: row stride %lld smaller than C=%d", (long long)ld, C);
  if (C > MC_MAX_C) {
    set_error("stag_mc_accumulate: C=%d above the supported %d classes", C, MC_MAX_C);
    return STAG_EUNSUPPORTED;
  }
  if (N == 0 || S == 0) return STAG_OK;
  STAG_CHECK_ARG(probs && acc_sum && acc_ent, "stag_mc_accumulate: null pointer");
  McAccParams p;
  p.probs = probs; p.ld = ld; p.ss = sample_stride; p.N = N; p.C = C; p.S = S;
  p.acc_sum = acc_sum; p.acc_ent = acc_ent;
  const int grid = mc_grid(N);
  if (kind == 0) launch_accumulate<0>(p, grid, stream);
  else launch_accumulate<1>(p, grid, stream);
  STAG_LAUNCH_CHECK();
  return STAG_OK;
}

extern "C" int stag_mc_finalize(const double* acc_sum, const double* acc_ent, int64_t N, int32_t C, int64_t S_total,
                                int kind, const void* y, int64_t ldy, float* mean, float* pred_entropy,
                                float* exp_entropy, float* mutual_info, float* loglik, void* stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  STAG_CHECK_ARG(N >= 0 && C > 0 && S_total > 0, "stag_mc_finalize: bad sizes N=%lld C=%d S_total=%lld",
                 (long long)N, C, (long long)S_total);
  STAG_CHECK_ARG(kind == 0 || kind == 1, "stag_mc_finalize: kind must be 0 (categorical) or 1 (bernoulli)");
  STAG_CHECK_ARG((y == nullptr) == (loglik == nullptr), "stag_mc_finalize: y and loglik go together");
  STAG_CHECK_ARG(kind == 0 || y == nullptr || ldy >= C, "stag_mc_finalize: label row stride smaller than C");
  if (N == 0) return STAG_OK;
  STAG_CHECK_ARG(acc_sum && acc_ent && mean && pred_entropy && exp_entropy && mutual_info,
                 "stag_mc_finalize: null pointer");
  McStatsParams p;
  p.acc_sum = acc_sum; p.acc_ent = acc_ent; p.N = N; p.S = S_total; p.C = C;
  p.y_idx = kind == 0 ? (const int64_t*)y : nullptr;
  p.y_val = kind == 1 ? (const float*)y : nullptr;
  p.ldy = ldy;
  p.mean = mean; p.pred = pred_entropy; p.expd = exp_entropy; p.mi = mutual_info; p.loglik = loglik;
  const int grid = mc_grid(N);
  if (kind == 0) mc_stats_kernel<0><<<grid, MC_THREADS, 0, stream>>>(p);
  else mc_stats_kernel<1><<<grid, MC_THREADS, 0, stream>>>(p);
  STAG_LAUNCH_CHECK();
  return STAG_OK;
}
