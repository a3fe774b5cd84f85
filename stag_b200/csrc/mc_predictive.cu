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
// stag_calibration bins [N,C] probabilities (the mean, say) into an integer calibration table against labels.
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

// ---- calibration tables (stag_calibration) ----------------------------------------------------------------------------
// One warp per row, as mc_stats_kernel: the Categorical row sum s is taken in its order (lane l adds classes l, l+32, ...,
// then the xor butterfly), so the oracle can restate it.  Every table term is an integer (a count or fx(x) = rint(x 2^32))
// and every sum an integer sum, so the table does not depend on the order of the additions: a CTA adds its rows into a
// shared copy of its part of the table and flushes each non-zero entry with one 64-bit global atomic.
//
// The per-class table has 3 C B entries (1.5 MB at C = 1024, B = 64).  Where it does not fit in CAL_SMEM_BUDGET the
// classes are cut into J slices of 32 ks classes and a CTA owns one (row group, slice) pair: every slice reads the whole
// row (validity and s need it) but adds only its own classes.  The J CTAs of a row group are adjacent in launch order
// and walk the same rows, so the re-reads come from L2.
constexpr int CAL_HEAD = 6;                 // n, n_invalid, n_correct | tp, 0 | fp, 0 | fn, brier
constexpr int CAL_MAX_BINS = 64;
constexpr int CAL_SMEM_BUDGET = 110 * 1024; // two CTAs per SM at the largest slice
constexpr double kCalOne = 4294967296.0;    // STAG_CAL_ONE

struct CalParams {
  const float* probs;
  int64_t ld, N;
  int C, B;
  const int64_t* y_idx;  // categorical: [N]
  const float* y_val;    // bernoulli: [N, C], row stride ldy
  int64_t ldy;
  const uint8_t* mask;   // [N] or NULL
  unsigned long long* table;
  int J, ks, Cs;         // class slices, 32-class slots per slice, classes per slice (stride of the shared table)
  int64_t R;             // row groups: CTA b takes slice b % J of the rows b / J + R k
};

// rint(x a) for x a in [0, 2^52): adding 2^52 rounds to an integer (ties to even) that is the low word of the double,
// without a conversion instruction (the conversions were the longest part of a row's chain)
__device__ __forceinline__ long long cal_rint(double x, double a) {
  return __double_as_longlong(__fma_rn(x, a, 4503599627370496.0)) - 0x4330000000000000LL;
}
__device__ __forceinline__ long long cal_fx(double x) { return cal_rint(x, kCalOne); }  // x in [0, 1]

// bins are (lo, hi] with interior edges edge[i] = i * (1.0 / B), as np.linspace(0, 1, B + 1) makes them: bin(x) = the
// number of interior edges strictly below x (np.searchsorted), x in [0, 1].  rint(x B) is within one of it.
__device__ __forceinline__ int cal_bin(double x, int B, double Bd, const double* edge) {
  int b = min((int)cal_rint(x, Bd), B - 1);
  while (b > 0 && !(edge[b] < x)) --b;
  while (b < B - 1 && edge[b + 1] < x) ++b;
  return b;
}

// shared entry e holds lo[e] + 2^32 hi[e].  A 64-bit shared atomic add compiles to a CAS loop on sm_100a; two 32-bit
// adds do not, and the thread whose add wraps the low word carries into the high one.
__device__ __forceinline__ void cal_add(unsigned* lo, unsigned* hi, int e, unsigned long long v) {
  if (!v) return;
  const unsigned l = (unsigned)v;
  const unsigned old = atomicAdd(lo + e, l);
  const unsigned h = (unsigned)(v >> 32) + (old + l < old ? 1u : 0u);
  if (h) atomicAdd(hi + e, h);
}
// counts stay below the rows of one call (< 2^31): the low word never wraps
__device__ __forceinline__ void cal_count(unsigned* lo, int e) { atomicAdd(lo + e, 1u); }

template <int KIND, int K>
struct CalRow {
  float x[K], t[K];  // probabilities; Bernoulli labels
  int64_t y;         // Categorical label
  bool on;           // inside [0, N) and not masked out
};

template <int KIND, int K>
__device__ __forceinline__ void cal_load(const CalParams& p, int64_t v, int lane, CalRow<KIND, K>& r) {
  r.on = v < p.N && (!p.mask || __ldg(p.mask + v));
  const float* row = p.probs + (r.on ? v : 0) * p.ld;
#pragma unroll
  for (int k = 0; k < K; ++k) {
    const int c = lane + 32 * k;
    r.x[k] = (r.on && c < p.C) ? __ldg(row + c) : 0.f;
  }
  if (KIND == 0) {
    r.y = r.on ? __ldg(p.y_idx + v) : 0;
  } else {
    const float* yrow = p.y_val + (r.on ? v : 0) * p.ldy;
#pragma unroll
    for (int k = 0; k < K; ++k) {
      const int c = lane + 32 * k;
      r.t[k] = (r.on && c < p.C) ? __ldg(yrow + c) : 0.f;
    }
  }
}

template <int KIND, int K>
__device__ __forceinline__ void cal_row(const CalParams& p, const CalRow<KIND, K>& r, int lane, int j, int k0, int k1,
                                        const double* edge, unsigned* lo, unsigned* hi,
                                        long long (&hdr)[CAL_HEAD]) {
  const double Bd = (double)p.B;
  const int B = p.B, BC = p.B * p.Cs, top = CAL_HEAD, cls = CAL_HEAD + 3 * p.B, c0 = 32 * k0;
  bool bad = false;
  if (KIND == 0) {
    double s = 0.0;
    float best = -1.f;
    int bi = 0x7fffffff;
#pragma unroll
    for (int k = 0; k < K; ++k) {
      const int c = lane + 32 * k;
      if (c < p.C) {
        const float m = r.x[k];
        bad |= !(m >= 0.f) || isinf(m);
        s += (double)m;
        if (m > best) { best = m; bi = c; }  // strict: the first of equal values in a lane's increasing classes
      }
    }
    bad = __any_sync(0xffffffffu, bad);
    s = mc_warp_sum(s);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {  // argmax, ties to the lower class (torch.argmax)
      const float ob = __shfl_xor_sync(0xffffffffu, best, o);
      const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
      if (ob > best || (ob == best && oi < bi)) { best = ob; bi = oi; }
    }
    if (bad || s == 0.0 || r.y < 0 || r.y >= p.C) {
      if (j == 0 && lane == 0) ++hdr[1];
      return;
    }
    if (j == 0 && lane == 0) ++hdr[0];
#pragma unroll
    for (int k = 0; k < K; ++k) {
      const int c = lane + 32 * k;
      if (k >= k0 && k < k1 && c < p.C) {
        const double q = (double)r.x[k] / s;
        const bool is_y = c == r.y;
        const double d = q - (is_y ? 1.0 : 0.0);
        hdr[5] += cal_fx(d * d);
        const int b = cal_bin(q, B, Bd, edge);
        const long long fq = cal_fx(q);
        const int e = cls + b * p.Cs + (c - c0);  // shared per-class table [3][B][Cs]: the lanes of a bin hit
        cal_count(lo, e);                         // consecutive words
        cal_add(lo, hi, e + BC, fq);
        if (is_y) cal_count(lo, e + 2 * BC);
        if (c == bi) {                            // the lane of the argmax class: conf = q_k, top-label bin(conf)
          hdr[2] += is_y;
          cal_count(lo, top + b);
          cal_add(lo, hi, top + B + b, fq);
          if (is_y) cal_count(lo, top + 2 * B + b);
        }
      }
    }
  } else {
#pragma unroll
    for (int k = 0; k < K; ++k) {
      const int c = lane + 32 * k;
      if (c < p.C) bad |= !(r.x[k] >= 0.f && r.x[k] <= 1.f) || !(r.t[k] >= 0.f && r.t[k] <= 1.f);
    }
    bad = __any_sync(0xffffffffu, bad);
    if (bad) {
      if (j == 0 && lane == 0) ++hdr[1];
      return;
    }
    if (j == 0 && lane == 0) ++hdr[0];
#pragma unroll
    for (int k = 0; k < K; ++k) {
      const int c = lane + 32 * k;
      if (k >= k0 && k < k1 && c < p.C) {
        const bool pos = r.x[k] > 0.5f, tru = r.t[k] > 0.5f;
        hdr[2] += pos && tru;
        hdr[3] += pos && !tru;
        hdr[4] += !pos && tru;
        const double pd = (double)r.x[k], td = (double)r.t[k], d = pd - td;
        hdr[5] += cal_fx(d * d);
        const int e = cls + cal_bin(pd, B, Bd, edge) * p.Cs + (c - c0);
        cal_count(lo, e);
        cal_add(lo, hi, e + BC, cal_fx(pd));
        cal_add(lo, hi, e + 2 * BC, cal_fx(td));
      }
    }
  }
}

template <int KIND, int K>
__global__ void __launch_bounds__(MC_THREADS, 1) calib_kernel(const CalParams p) {
  extern __shared__ unsigned cal_smem[];
  const int E = CAL_HEAD + 3 * p.B + 3 * p.Cs * p.B;
  unsigned *lo = cal_smem, *hi = cal_smem + E;
  for (int e = threadIdx.x; e < 2 * E; e += MC_THREADS) cal_smem[e] = 0u;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int j = blockIdx.x % p.J;
  const int k0 = j * p.ks, k1 = k0 + p.ks;
  __shared__ double edge[CAL_MAX_BINS];
  if (threadIdx.x < p.B) edge[threadIdx.x] = (double)threadIdx.x * (1.0 / p.B);
  long long hdr[CAL_HEAD] = {0, 0, 0, 0, 0, 0};
  __syncthreads();
  // small rows: the next row's loads are issued before this row is processed
  constexpr bool kPrefetch = K <= 8;
  const int64_t step = p.R * MC_WARPS;
  int64_t v = (int64_t)(blockIdx.x / p.J) * MC_WARPS + warp;
  CalRow<KIND, K> next;
  if (kPrefetch) cal_load(p, v, lane, next);
  for (; v < p.N; v += step) {
    CalRow<KIND, K> r;
    if (kPrefetch) {
      r = next;
      cal_load(p, v + step, lane, next);
    } else {
      cal_load(p, v, lane, r);
    }
    if (r.on) cal_row(p, r, lane, j, k0, k1, edge, lo, hi, hdr);
  }
#pragma unroll
  for (int i = 0; i < CAL_HEAD; ++i) {
    long long s = hdr[i];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    if (lane == 0) cal_add(lo, hi, i, (unsigned long long)s);
  }
  __syncthreads();
  const int head = CAL_HEAD + 3 * p.B, BC = p.B * p.Cs;
  for (int e = threadIdx.x; e < E; e += MC_THREADS) {
    const unsigned long long val = (unsigned long long)lo[e] | ((unsigned long long)hi[e] << 32);
    if (!val) continue;
    int64_t g = e;
    if (e >= head) {  // [3][B][Cs] slice -> [3][C][B]
      const int r = e - head, tab = r / BC, b = (r % BC) / p.Cs, c = 32 * k0 + r % p.Cs;
      g = head + ((int64_t)tab * p.C + c) * p.B + b;
    }
    atomicAdd(p.table + g, val);
  }
}

template <int KIND, int K>
static int launch_calib_k(CalParams p, size_t smem, cudaStream_t stream) {
  auto kern = calib_kernel<KIND, K>;
  // the attribute and the occupancy query of the last (device, shared size) of this instantiation: the query costs more
  // host time than the kernel takes at the arxiv shape
  static thread_local int last_dev = -1, per_sm = 0;
  static thread_local size_t last_smem = 0;
  int dev = 0;
  STAG_CUDA(cudaGetDevice(&dev));
  if (dev != last_dev || smem != last_smem) {
    if (smem > 48 * 1024)
      STAG_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    STAG_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, MC_THREADS, smem));
    last_dev = dev;
    last_smem = smem;
  }
  // one resident wave: every CTA flushes its table once, so more CTAs than fit cost flushes and gain nothing
  const int64_t groups = ((int64_t)(per_sm > 0 ? per_sm : 1) * num_sms()) / p.J;
  const int64_t need = (p.N + MC_WARPS - 1) / MC_WARPS;
  p.R = groups < 1 ? 1 : (groups < need ? groups : need);
  kern<<<(unsigned)(p.R * p.J), MC_THREADS, smem, stream>>>(p);
  STAG_LAUNCH_CHECK();
  return STAG_OK;
}

template <int KIND>
static int launch_calib(const CalParams& p, size_t smem, cudaStream_t stream) {
  if (p.C <= 32) return launch_calib_k<KIND, 1>(p, smem, stream);
  if (p.C <= 64) return launch_calib_k<KIND, 2>(p, smem, stream);
  if (p.C <= 128) return launch_calib_k<KIND, 4>(p, smem, stream);
  if (p.C <= 256) return launch_calib_k<KIND, 8>(p, smem, stream);
  if (p.C <= 512) return launch_calib_k<KIND, 16>(p, smem, stream);
  return launch_calib_k<KIND, 32>(p, smem, stream);
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

extern "C" int64_t stag_calibration_table_len(int32_t C, int32_t n_bins) {
  if (C < 1 || n_bins < 1 || n_bins > CAL_MAX_BINS) return STAG_EINVAL;
  return CAL_HEAD + 3 * (int64_t)n_bins + 3 * (int64_t)C * n_bins;
}

extern "C" int stag_calibration(const float* probs, int64_t ld, int64_t N, int32_t C, int kind, const void* y,
                                int64_t ldy, const uint8_t* mask, int32_t n_bins, int64_t* table, void* stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  STAG_CHECK_ARG(N >= 0 && C > 0, "stag_calibration: bad sizes N=%lld C=%d", (long long)N, C);
  STAG_CHECK_ARG(kind == 0 || kind == 1, "stag_calibration: kind must be 0 (categorical) or 1 (bernoulli)");
  STAG_CHECK_ARG(n_bins >= 1 && n_bins <= CAL_MAX_BINS, "stag_calibration: n_bins=%d outside [1, %d]", n_bins,
                 CAL_MAX_BINS);
  STAG_CHECK_ARG(ld >= C && (kind == 0 || ldy >= C), "stag_calibration: row strides smaller than C=%d", C);
  if (C > MC_MAX_C) {
    set_error("stag_calibration: C=%d above the supported %d classes", C, MC_MAX_C);
    return STAG_EUNSUPPORTED;
  }
  if (N == 0) return STAG_OK;
  STAG_CHECK_ARG(probs && y && table, "stag_calibration: null pointer");
  // every term is at most STAG_CAL_ONE: 2^31 terms per entry keep a zeroed table below 2^63
  STAG_CHECK_ARG(N <= (((int64_t)1 << 31) - 1) / C, "stag_calibration: N*C = %lld terms in one call, above 2^31 - 1",
                 (long long)N * C);
  CalParams p;
  p.probs = probs; p.ld = ld; p.N = N; p.C = C; p.B = n_bins;
  p.y_idx = kind == 0 ? (const int64_t*)y : nullptr;
  p.y_val = kind == 1 ? (const float*)y : nullptr;
  p.ldy = ldy; p.mask = mask; p.table = (unsigned long long*)table;
  // 8 bytes of shared memory per table entry: the header and top-label table, and 3 B entries per class of a slice
  const int slots = (C + 31) / 32;
  const int64_t fixed = 8 * (int64_t)(CAL_HEAD + 3 * n_bins), per_slot = 8 * 3 * 32 * (int64_t)n_bins;
  const int64_t fit = (CAL_SMEM_BUDGET - fixed) / per_slot;
  p.ks = fit < 1 ? 1 : (fit < slots ? (int)fit : slots);
  p.J = (slots + p.ks - 1) / p.ks;
  p.Cs = C < 32 * p.ks ? C : 32 * p.ks;
  p.R = 1;
  const size_t smem = 8 * (size_t)(CAL_HEAD + 3 * n_bins + 3 * p.Cs * n_bins);
  return kind == 0 ? launch_calib<0>(p, smem, stream) : launch_calib<1>(p, smem, stream);
}
