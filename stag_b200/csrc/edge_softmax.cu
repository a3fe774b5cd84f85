// Segmented softmax over the in-edges of every destination node (dgl.nn.edge_softmax as the reference's GAT uses it,
// stag/zoo/gat.py:122:  a = edge_softmax(graph, e),  e [E,H] = noise * leaky_relu(el[u] + er[v])), forward and backward.
// Replaces the scatter-amax / gather / exp / index_add / gather / divide chain (and its autograd graph) by one pass
// per direction over the CSC rows: one warp per destination, a lane per (in-edge, head) pair, per-head max / sum by
// shuffles between the lanes that hold the same head.  logits and outputs are in ORIGINAL edge order ([E,H], like every
// per-edge tensor of the reference); the row's edges are reached through the CSC edge ids.  Deterministic.
#include "common.cuh"
#include "noise.cuh"
#include "param_finalize.cuh"

namespace stag {

constexpr int SM_THREADS = 256, SM_WARPS = SM_THREADS / 32;

struct SoftmaxParams {
  const int32_t* indptr;
  const int32_t* eid;
  int64_t N;
  int H;
  const float* in0;  // forward: logits;  backward: a
  const float* in1;  // backward: da
  float* out;        // forward: a;       backward: dlogits
};

// combine `v` over the lanes that hold the same head (lane % H, H a power of two <= 32)
template <bool MAX>
__device__ __forceinline__ float head_reduce(float v, int H) {
  for (int o = 16; o >= H; o >>= 1) {
    const float w = __shfl_xor_sync(0xffffffffu, v, o);
    v = MAX ? fmaxf(v, w) : v + w;
  }
  return v;
}

// H divides 32: element t = lane + 32 k of a row's (edge, head) pairs has head lane % H for every k
template <bool BWD>
__global__ void __launch_bounds__(SM_THREADS) edge_softmax_pow2_kernel(const SoftmaxParams p) {
  const int lane = threadIdx.x & 31;
  const int64_t nwarps = (int64_t)gridDim.x * SM_WARPS;
  const int H = p.H, hsh = __ffs(H) - 1, h = lane & (H - 1);
  for (int64_t v = (int64_t)blockIdx.x * SM_WARPS + (threadIdx.x >> 5); v < p.N; v += nwarps) {
    const int e0 = __ldg(p.indptr + v), e1 = __ldg(p.indptr + v + 1);
    const int total = (e1 - e0) << hsh;
    if (total == 0) continue;
    if (!BWD) {
      float m = -INFINITY;
      for (int t = lane; t < total; t += 32)
        m = fmaxf(m, __ldg(p.in0 + (int64_t)__ldg(p.eid + e0 + (t >> hsh)) * H + h));
      m = head_reduce<true>(m, H);
      float s = 0.f;
      for (int t = lane; t < total; t += 32)
        s += expf(__ldg(p.in0 + (int64_t)__ldg(p.eid + e0 + (t >> hsh)) * H + h) - m);
      s = head_reduce<false>(s, H);
      for (int t = lane; t < total; t += 32) {
        const int64_t o = (int64_t)__ldg(p.eid + e0 + (t >> hsh)) * H + h;
        p.out[o] = expf(__ldg(p.in0 + o) - m) / s;
      }
    } else {
      float d = 0.f;  // sum_e a_e da_e of this head
      for (int t = lane; t < total; t += 32) {
        const int64_t o = (int64_t)__ldg(p.eid + e0 + (t >> hsh)) * H + h;
        d = fmaf(__ldg(p.in0 + o), __ldg(p.in1 + o), d);
      }
      d = head_reduce<false>(d, H);
      for (int t = lane; t < total; t += 32) {
        const int64_t o = (int64_t)__ldg(p.eid + e0 + (t >> hsh)) * H + h;
        p.out[o] = __ldg(p.in0 + o) * (__ldg(p.in1 + o) - d);
      }
    }
  }
}

// any H: one head at a time, lanes over the edges of the row
template <bool BWD>
__global__ void __launch_bounds__(SM_THREADS) edge_softmax_any_kernel(const SoftmaxParams p) {
  const int lane = threadIdx.x & 31;
  const int64_t nwarps = (int64_t)gridDim.x * SM_WARPS;
  const int H = p.H;
  for (int64_t v = (int64_t)blockIdx.x * SM_WARPS + (threadIdx.x >> 5); v < p.N; v += nwarps) {
    const int e0 = __ldg(p.indptr + v), e1 = __ldg(p.indptr + v + 1);
    for (int h = 0; h < H && e1 > e0; ++h) {
      if (!BWD) {
        float m = -INFINITY;
        for (int j = e0 + lane; j < e1; j += 32) m = fmaxf(m, __ldg(p.in0 + (int64_t)__ldg(p.eid + j) * H + h));
        m = head_reduce<true>(m, 1);
        float s = 0.f;
        for (int j = e0 + lane; j < e1; j += 32) s += expf(__ldg(p.in0 + (int64_t)__ldg(p.eid + j) * H + h) - m);
        s = head_reduce<false>(s, 1);
        for (int j = e0 + lane; j < e1; j += 32) {
          const int64_t o = (int64_t)__ldg(p.eid + j) * H + h;
          p.out[o] = expf(__ldg(p.in0 + o) - m) / s;
        }
      } else {
        float d = 0.f;
        for (int j = e0 + lane; j < e1; j += 32) {
          const int64_t o = (int64_t)__ldg(p.eid + j) * H + h;
          d = fmaf(__ldg(p.in0 + o), __ldg(p.in1 + o), d);
        }
        d = head_reduce<false>(d, 1);
        for (int j = e0 + lane; j < e1; j += 32) {
          const int64_t o = (int64_t)__ldg(p.eid + j) * H + h;
          p.out[o] = __ldg(p.in0 + o) * (__ldg(p.in1 + o) - d);
        }
      }
    }
  }
}

static int softmax_launch(const StagGraph* g, const float* in0, const float* in1, int H, float* out, bool bwd,
                          cudaStream_t stream, const char* who) {
  STAG_CHECK_ARG(g != nullptr && g->indptr != nullptr, "%s: null graph", who);
  STAG_CHECK_ARG(H > 0, "%s: H=%d must be positive", who, H);
  if (g->num_rows == 0 || g->num_edges == 0) return STAG_OK;
  STAG_CHECK_ARG(g->eid && in0 && out && (!bwd || in1), "%s: null argument", who);
  SoftmaxParams p;
  p.indptr = g->indptr; p.eid = g->eid; p.N = g->num_rows; p.H = H; p.in0 = in0; p.in1 = in1; p.out = out;
  const int64_t want = (g->num_rows + SM_WARPS - 1) / SM_WARPS;
  const int grid = (int)(want < (int64_t)num_sms() * 16 ? want : (int64_t)num_sms() * 16);
  const bool pow2 = H <= 32 && (H & (H - 1)) == 0;
  if (pow2) {
    if (bwd) edge_softmax_pow2_kernel<true><<<grid, SM_THREADS, 0, stream>>>(p);
    else edge_softmax_pow2_kernel<false><<<grid, SM_THREADS, 0, stream>>>(p);
  } else {
    if (bwd) edge_softmax_any_kernel<true><<<grid, SM_THREADS, 0, stream>>>(p);
    else edge_softmax_any_kernel<false><<<grid, SM_THREADS, 0, stream>>>(p);
  }
  STAG_LAUNCH_CHECK();
  return STAG_OK;
}

// ---- attention logits fused in (stag/zoo/gat.py:113-122) -----------------------------------------------------------
//   logit[s,e,h] = w_s[e,h] * leaky_relu(el[s,u_e,h] + er[s,v_e,h]),   a[s,e,h] = softmax over the in-edges of v
// The [E,H] logits (two gathers, an add, the leaky relu, the noise product: five torch launches and their autograd
// graph) never exist: the forward recomputes them per pass over the row (el rows come from L1 / L2), the backward emits
//   dw[e,h] = dlogit * leaky(pre),   t[e,h] = dlogit * w * leaky'(pre)  (= d pre, summed per SOURCE by the caller on the CSR),
//   d_er[v,h] = sum over the row of t   -- no atomics anywhere: deterministic, unlike index_add of the gather's autograd.
// The noise w is none (1), read from an external [S,E,H] tensor, or drawn in the kernel (KIND = Normal / Uniform /
// Bernoulli, K == H): the variate of (edge e, head h, sample s) is the one stag_noise_emit writes for channel h -- slot
// h%4 + 4*((h%64)/32) of Philox block 8*(h/64) + (h%32)/4, sample index sample_base + s -- so the fused attention equals
// the attention over the materialised tensor bit for bit.  The backward regenerates it and reduces the parameter
// gradients: SCALAR / CHANNEL through per-warp shared-memory rows, per-CTA partials and param_finalize_kernel (fixed
// order), EDGE / EDGE_CHANNEL by the one warp that owns the edge's destination row.  One warp per destination row, the
// S samples as a loop inside the row: every output element has a single writer.
struct AttnParams {
  const int32_t* indptr;
  const int32_t* indices;
  const int32_t* eid;
  int64_t N, E;
  int H, S;
  const float* el;   // [S?][num_cols, H]
  int64_t el_ss;     // sample stride of el (0: shared)
  const float* er;   // [S?][N, H]
  int64_t er_ss;
  // noise
  int pshape, relu, sample_base;
  const float* p0;
  const float* p1;
  const float* ext;  // EXTERNAL: [S, E, H] in original edge order
  PhiloxKey key;
  const uint32_t* ctr;  // optional device-side addend to key.c3
  float slope;
  float* a;          // [S, E, H] forward: out;  backward: in
  const float* da;   // backward
  float* dw;         // backward, EXTERNAL only, may be null
  float* t;          // backward: d(el[u] + er[v]) per edge
  float* d_er;       // backward: [S, N, H]
  float* dp0;        // backward, parameter gradients (Normal / Uniform): EDGE shapes accumulate here
  float* dp1;
  float* dp_partial; // backward, SCALAR / CHANNEL: [gridDim.x][2][H]
};

// raw variate (standard normal / U[0,1)) of head h: the value raw_oct writes to channel h (noise.cuh)
template <int KIND>
__device__ __forceinline__ float raw_head(uint32_t e, int h, uint32_t sample, const PhiloxKey& key) {
  const uint32_t q = 8u * (uint32_t)(h >> 6) + (uint32_t)((h & 31) >> 2);
  const int j = (h & 3) + 4 * ((h >> 5) & 1);
  const uint4 r = philox4x32<kPhiloxRounds>(q, e, sample, key.c3, key.k0, key.k1);
  const int i = j >> 1;
  const uint32_t w = i == 0 ? r.x : (i == 1 ? r.y : (i == 2 ? r.z : r.w));
  if (KIND == STAG_NOISE_NORMAL) {
    float rad, c, s;
    bm_parts(w, rad, c, s);
    return (j & 1) ? rad * s : rad * c;
  }
  return (j & 1) ? half_uniform<true>(w) : half_uniform<false>(w);
}

// noise w of (edge e, head h, sample s); `raw` / `pos` (generated kinds) feed the parameter gradients
template <int KIND>
__device__ __forceinline__ float attn_noise(const AttnParams& p, const PhiloxKey& key, int64_t e, int h, int s, float& raw,
                                            bool& pos) {
  if (KIND == STAG_NOISE_NONE) return 1.0f;
  if (KIND == STAG_NOISE_EXTERNAL) return __ldg(p.ext + ((int64_t)s * p.E + e) * p.H + h);
  raw = raw_head<KIND>((uint32_t)e, h, (uint32_t)(p.sample_base + s), key);
  const int64_t pi = p.pshape == STAG_PARAM_SCALAR ? 0
                     : (p.pshape == STAG_PARAM_CHANNEL ? h : (p.pshape == STAG_PARAM_EDGE ? e : e * p.H + h));
  const float w = transform<KIND>(raw, __ldg(p.p0 + pi), p.p1 ? __ldg(p.p1 + pi) : 0.f);
  pos = w > 0.f;
  return p.relu ? fmaxf(w, 0.f) : w;
}

template <bool POW2, bool BWD, int KIND>
__global__ void __launch_bounds__(SM_THREADS) attention_softmax_kernel(const AttnParams p) {
  extern __shared__ float sdp[];  // BWD, SCALAR / CHANNEL parameter gradients: [SM_WARPS][2][H]
  constexpr bool PG = BWD && (KIND == STAG_NOISE_NORMAL || KIND == STAG_NOISE_UNIFORM);
  const int lane = threadIdx.x & 31;
  const int64_t nwarps = (int64_t)gridDim.x * SM_WARPS;
  const int H = p.H, hsh = POW2 ? __ffs(H) - 1 : 0;
  PhiloxKey key = p.key;
  if (KIND >= STAG_NOISE_NORMAL && p.ctr) key.c3 += __ldg(p.ctr);
  const bool cta_dp = PG && p.dp_partial != nullptr;
  const bool edge_dp = PG && p.dp0 != nullptr && p.dp_partial == nullptr;
  float* wdp = sdp + (threadIdx.x >> 5) * 2 * H;
  if (cta_dp) {
    for (int i = threadIdx.x; i < SM_WARPS * 2 * H; i += SM_THREADS) sdp[i] = 0.f;
    __syncthreads();
  }
  float g0 = 0.f, g1 = 0.f;  // POW2: this lane's head's share of the SCALAR / CHANNEL gradients
  for (int64_t v = (int64_t)blockIdx.x * SM_WARPS + (threadIdx.x >> 5); v < p.N; v += nwarps) {
    const int e0 = __ldg(p.indptr + v), e1 = __ldg(p.indptr + v + 1);
    if (e1 == e0) {
      if (BWD)
        for (int s = 0; s < p.S; ++s)
          for (int h = lane; h < H; h += 32) p.d_er[((int64_t)s * p.N + v) * H + h] = 0.f;
      continue;
    }
    // POW2: lanes over the (edge, head) pairs of the row, head = lane % H, one pass;  else: head by head, lanes over the edges
    const int nh = POW2 ? 1 : H;
    for (int hh = 0; hh < nh; ++hh) {
      const int h = POW2 ? (lane & (H - 1)) : hh;
      const int total = POW2 ? (e1 - e0) << hsh : (e1 - e0);
      const int red = POW2 ? H : 1;
      for (int s = 0; s < p.S; ++s) {
        const float* el = p.el + s * p.el_ss;
        const float erv = __ldg(p.er + s * p.er_ss + v * H + h);
        const int64_t so = (int64_t)s * p.E * H;  // sample offset of a / da / dw / t
        auto edge_of = [&](int t) { return e0 + (POW2 ? (t >> hsh) : t); };
        auto pre_of = [&](int j) { return __ldg(el + (int64_t)__ldg(p.indices + j) * H + h) + erv; };
        float raw = 0.f;
        bool pos = true;
        auto wt_of = [&](int64_t e) { return attn_noise<KIND>(p, key, e, h, s, raw, pos); };
        if (!BWD) {
          float m = -INFINITY;
          for (int t = lane; t < total; t += 32) {
            const int j = edge_of(t);
            const float pre = pre_of(j);
            m = fmaxf(m, (pre > 0.f ? pre : p.slope * pre) * wt_of(__ldg(p.eid + j)));
          }
          m = head_reduce<true>(m, red);
          float sum = 0.f;
          for (int t = lane; t < total; t += 32) {
            const int j = edge_of(t);
            const float pre = pre_of(j);
            sum += expf((pre > 0.f ? pre : p.slope * pre) * wt_of(__ldg(p.eid + j)) - m);
          }
          sum = head_reduce<false>(sum, red);
          for (int t = lane; t < total; t += 32) {
            const int j = edge_of(t);
            const int64_t e = __ldg(p.eid + j);
            const float pre = pre_of(j);
            p.a[so + e * H + h] = expf((pre > 0.f ? pre : p.slope * pre) * wt_of(e) - m) / sum;
          }
        } else {
          float d = 0.f;  // sum_e a_e da_e of this head
          for (int t = lane; t < total; t += 32) {
            const int64_t o = so + (int64_t)__ldg(p.eid + edge_of(t)) * H + h;
            d = fmaf(__ldg(p.a + o), __ldg(p.da + o), d);
          }
          d = head_reduce<false>(d, red);
          float acc = 0.f, r0 = 0.f, r1 = 0.f;
          // warp-uniform trip count: the per-edge parameter gradient of POW2 sums the heads of an edge by shuffles
          for (int tb = 0; tb < total; tb += 32) {
            const int t = tb + lane;
            float c0 = 0.f, c1 = 0.f;
            int64_t e = 0;
            if (t < total) {
              const int j = edge_of(t);
              e = __ldg(p.eid + j);
              const int64_t o = so + e * H + h;
              const float dl = __ldg(p.a + o) * (__ldg(p.da + o) - d);
              const float pre = pre_of(j);
              const float w = wt_of(e);
              if (KIND == STAG_NOISE_EXTERNAL && p.dw) p.dw[o] = dl * (pre > 0.f ? pre : p.slope * pre);
              const float dp = dl * w * (pre > 0.f ? 1.0f : p.slope);
              p.t[o] = dp;
              acc += dp;
              if (PG) {
                // d logit / d w = leaky(pre), masked by w > 0 under relu;  w = p0 + p1 eps  |  p0 + (p1 - p0) u
                const float gw = (p.relu && !pos) ? 0.f : dl * (pre > 0.f ? pre : p.slope * pre);
                c1 = gw * raw;
                c0 = KIND == STAG_NOISE_NORMAL ? gw : gw - c1;
              }
            }
            if (edge_dp) {
              if (p.pshape == STAG_PARAM_EDGE_CHANNEL) {
                if (t < total) {
                  p.dp0[e * H + h] += c0;
                  p.dp1[e * H + h] += c1;
                }
              } else if (POW2) {  // [E,1]: the H lanes of an edge are adjacent
                for (int o = 1; o < H; o <<= 1) {
                  c0 += __shfl_xor_sync(0xffffffffu, c0, o);
                  c1 += __shfl_xor_sync(0xffffffffu, c1, o);
                }
                if (t < total && h == 0) {
                  p.dp0[e] += c0;
                  p.dp1[e] += c1;
                }
              } else if (t < total) {  // one head at a time: the lane owns the edge for every head
                p.dp0[e] += c0;
                p.dp1[e] += c1;
              }
            } else if (cta_dp) {
              if (POW2) {
                g0 += c0;
                g1 += c1;
              } else {
                r0 += c0;
                r1 += c1;
              }
            }
          }
          acc = head_reduce<false>(acc, red);
          if (POW2 ? lane < H : lane == 0) p.d_er[((int64_t)s * p.N + v) * H + h] = acc;
          if (!POW2 && cta_dp) {
            r0 = head_reduce<false>(r0, 1);
            r1 = head_reduce<false>(r1, 1);
            if (lane == 0) {
              wdp[h] += r0;
              wdp[H + h] += r1;
            }
          }
        }
      }
    }
  }
  if (cta_dp) {
    if (POW2) {
      g0 = head_reduce<false>(g0, H);
      g1 = head_reduce<false>(g1, H);
      if (lane < H) {
        wdp[lane] += g0;
        wdp[H + lane] += g1;
      }
    }
    __syncthreads();
    for (int c = threadIdx.x; c < 2 * H; c += SM_THREADS) {
      float acc = 0.f;
      for (int w = 0; w < SM_WARPS; ++w) acc += sdp[w * 2 * H + c];
      p.dp_partial[(int64_t)blockIdx.x * 2 * H + c] = acc;
    }
  }
}

static int attn_grid(int64_t rows) {
  const int64_t want = (rows + SM_WARPS - 1) / SM_WARPS;
  const int64_t cap = (int64_t)num_sms() * 16;
  return (int)(want < 1 ? 1 : (want < cap ? want : cap));
}

template <bool POW2, bool BWD>
static void attention_dispatch(int kind, const AttnParams& p, int grid, size_t smem, cudaStream_t stream) {
  switch (kind) {
    case STAG_NOISE_NONE: attention_softmax_kernel<POW2, BWD, STAG_NOISE_NONE><<<grid, SM_THREADS, smem, stream>>>(p); break;
    case STAG_NOISE_EXTERNAL: attention_softmax_kernel<POW2, BWD, STAG_NOISE_EXTERNAL><<<grid, SM_THREADS, smem, stream>>>(p); break;
    case STAG_NOISE_NORMAL: attention_softmax_kernel<POW2, BWD, STAG_NOISE_NORMAL><<<grid, SM_THREADS, smem, stream>>>(p); break;
    case STAG_NOISE_UNIFORM: attention_softmax_kernel<POW2, BWD, STAG_NOISE_UNIFORM><<<grid, SM_THREADS, smem, stream>>>(p); break;
    default: attention_softmax_kernel<POW2, BWD, STAG_NOISE_BERNOULLI><<<grid, SM_THREADS, smem, stream>>>(p); break;
  }
}

template <bool POW2, bool BWD, int KIND>
static int attention_smem_attr(size_t smem) {
  STAG_CUDA(cudaFuncSetAttribute(attention_softmax_kernel<POW2, BWD, KIND>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                 (int)smem));
  return STAG_OK;
}

// One launch of the attention kernel over S samples (and, for SCALAR / CHANNEL parameter gradients, the finalize).
static int attention_launch(const StagGraph* g, AttnParams p, const StagNoise* n, bool bwd, void* ws, size_t ws_bytes,
                            cudaStream_t stream, const char* who) {
  STAG_CHECK_ARG(g != nullptr && g->indptr != nullptr, "%s: null graph", who);
  STAG_CHECK_ARG(p.H > 0 && p.S > 0, "%s: H=%d and S=%d must be positive", who, p.H, p.S);
  STAG_CHECK_ARG(p.el_ss >= 0 && p.er_ss >= 0, "%s: negative sample stride", who);
  STAG_CHECK_ARG(n != nullptr, "%s: null noise spec", who);
  const int kind = n->kind;
  STAG_CHECK_ARG(kind >= STAG_NOISE_NONE && kind <= STAG_NOISE_NORMAL_HADAMARD, "%s: bad noise kind %d", who, kind);
  if (kind == STAG_NOISE_NORMAL_HADAMARD) {
    set_error("%s: the tensor-core generator works on 128-channel groups; the attention noise has one channel per head", who);
    return STAG_EUNSUPPORTED;
  }
  STAG_CHECK_ARG(!n->in_norm, "%s: in_norm is not fused into the attention (materialise the noise)", who);
  const bool gen = kind >= STAG_NOISE_NORMAL;
  if (kind != STAG_NOISE_NONE) STAG_CHECK_ARG(n->K == p.H, "%s: noise width K=%d must equal H=%d", who, n->K, p.H);
  if (gen) {
    STAG_CHECK_ARG(n->param_shape >= STAG_PARAM_SCALAR && n->param_shape <= STAG_PARAM_EDGE_CHANNEL,
                   "%s: bad param_shape %d", who, n->param_shape);
    STAG_CHECK_ARG(n->p0 != nullptr || g->num_edges == 0, "%s: null parameter p0", who);
    STAG_CHECK_ARG(kind == STAG_NOISE_BERNOULLI || n->p1 != nullptr || g->num_edges == 0, "%s: null parameter p1", who);
  }
  STAG_CHECK_ARG(kind != STAG_NOISE_EXTERNAL || n->external != nullptr || g->num_edges == 0,
                 "%s: EXTERNAL noise needs a tensor", who);
  if (g->num_rows == 0) return STAG_OK;
  STAG_CHECK_ARG(p.er && p.a && (g->num_edges == 0 || (g->eid && g->indices && p.el)) && (!bwd || (p.da && p.t && p.d_er)),
                 "%s: null argument", who);
  p.indptr = g->indptr; p.indices = g->indices; p.eid = g->eid; p.N = g->num_rows; p.E = g->num_edges;
  p.pshape = n->param_shape; p.relu = n->relu; p.sample_base = n->sample_base;
  p.p0 = n->p0; p.p1 = n->p1; p.ext = n->external;
  p.key = make_key(n->seed, n->offset);
  p.ctr = n->counter;
  const int grid = attn_grid(g->num_rows);
  const bool pg = bwd && (kind == STAG_NOISE_NORMAL || kind == STAG_NOISE_UNIFORM) && p.dp0 != nullptr;
  const bool cta_dp = pg && p.pshape <= STAG_PARAM_CHANNEL;
  size_t smem = 0;
  if (cta_dp) {
    const size_t need = align_up((size_t)grid * 2 * p.H * sizeof(float) + 16, 256);
    if (!ws || ws_bytes < need) {
      set_error("%s: workspace %zu < required %zu (stag_attention_workspace_bytes)", who, ws_bytes, need);
      return STAG_EWORKSPACE;
    }
    p.dp_partial = (float*)ws;
    smem = (size_t)SM_WARPS * 2 * p.H * sizeof(float);
    if (smem > 200 * 1024) {
      set_error("%s: H=%d too wide for the shared-memory parameter-gradient staging", who, p.H);
      return STAG_EUNSUPPORTED;
    }
  } else {
    p.dp_partial = nullptr;
  }
  if (!pg) p.dp0 = p.dp1 = nullptr;
  const bool pow2 = p.H <= 32 && (p.H & (p.H - 1)) == 0;
  if (smem > 48 * 1024) {
    int rc = pow2 ? (kind == STAG_NOISE_NORMAL ? attention_smem_attr<true, true, STAG_NOISE_NORMAL>(smem)
                                               : attention_smem_attr<true, true, STAG_NOISE_UNIFORM>(smem))
                  : (kind == STAG_NOISE_NORMAL ? attention_smem_attr<false, true, STAG_NOISE_NORMAL>(smem)
                                               : attention_smem_attr<false, true, STAG_NOISE_UNIFORM>(smem));
    if (rc) return rc;
  }
  if (pow2) {
    if (bwd) attention_dispatch<true, true>(kind, p, grid, smem, stream);
    else attention_dispatch<true, false>(kind, p, grid, 0, stream);
  } else {
    if (bwd) attention_dispatch<false, true>(kind, p, grid, smem, stream);
    else attention_dispatch<false, false>(kind, p, grid, 0, stream);
  }
  STAG_LAUNCH_CHECK();
  if (cta_dp) {
    const int scalar = p.pshape == STAG_PARAM_SCALAR;
    param_finalize_kernel<<<scalar ? 1 : (p.H + 255) / 256, 256, 0, stream>>>(p.dp_partial, grid, p.H, p.H, scalar,
                                                                              p.dp0, p.dp1);
    STAG_LAUNCH_CHECK();
  }
  return STAG_OK;
}

}  // namespace stag

using namespace stag;

extern "C" int stag_edge_softmax(const StagGraph* csc, const float* logits, int32_t H, float* out, void* stream) {
  return softmax_launch(csc, logits, nullptr, H, out, false, (cudaStream_t)stream, "stag_edge_softmax");
}

extern "C" int stag_edge_softmax_bwd(const StagGraph* csc, const float* a, const float* da, int32_t H, float* dlogits,
                                     void* stream) {
  return softmax_launch(csc, a, da, H, dlogits, true, (cudaStream_t)stream, "stag_edge_softmax_bwd");
}

// the S = 1 entry points: no noise (w == NULL) or an external [E,H] tensor
static StagNoise legacy_noise(const float* w, int32_t H) {
  StagNoise n = {};
  n.kind = w ? STAG_NOISE_EXTERNAL : STAG_NOISE_NONE;
  n.K = H;
  n.external = w;
  return n;
}

extern "C" int stag_attention_softmax(const StagGraph* csc, const float* el, const float* er, const float* w, float slope,
                                      int32_t H, float* a, void* stream) {
  AttnParams p = {};
  p.H = H; p.S = 1; p.el = el; p.er = er; p.slope = slope; p.a = a;
  if (csc && csc->num_edges == 0) return STAG_OK;
  const StagNoise n = legacy_noise(w, H);
  return attention_launch(csc, p, &n, false, nullptr, 0, (cudaStream_t)stream, "stag_attention_softmax");
}

extern "C" int stag_attention_softmax_bwd(const StagGraph* csc, const float* el, const float* er, const float* w, float slope,
                                          int32_t H, const float* a, const float* da, float* dw, float* dpre, float* d_er,
                                          void* stream) {
  AttnParams p = {};
  p.H = H; p.S = 1; p.el = el; p.er = er; p.slope = slope; p.a = const_cast<float*>(a); p.da = da; p.dw = dw; p.t = dpre;
  p.d_er = d_er;
  const StagNoise n = legacy_noise(w, H);
  return attention_launch(csc, p, &n, true, nullptr, 0, (cudaStream_t)stream, "stag_attention_softmax_bwd");
}

extern "C" size_t stag_attention_workspace_bytes(const StagGraph* csc, int32_t H, int32_t S) {
  (void)S;
  if (H <= 0) return 0;
  const int grid = attn_grid(csc ? csc->num_rows : ((int64_t)1 << 40));
  return align_up((size_t)grid * 2 * H * sizeof(float) + 16, 256);
}

extern "C" int stag_attention_softmax_s(const StagGraph* csc, const float* el, int64_t el_sample_stride, const float* er,
                                        int64_t er_sample_stride, int32_t H, int32_t S, const StagNoise* noise, float slope,
                                        float* a, void* ws, size_t ws_bytes, void* stream) {
  AttnParams p = {};
  p.H = H; p.S = S; p.el = el; p.el_ss = el_sample_stride; p.er = er; p.er_ss = er_sample_stride; p.slope = slope; p.a = a;
  return attention_launch(csc, p, noise, false, ws, ws_bytes, (cudaStream_t)stream, "stag_attention_softmax_s");
}

extern "C" int stag_attention_softmax_s_bwd(const StagGraph* csc, const float* el, int64_t el_sample_stride, const float* er,
                                            int64_t er_sample_stride, int32_t H, int32_t S, const StagNoise* noise,
                                            float slope, const float* a, const float* da, float* dpre, float* d_er,
                                            float* dparam0, float* dparam1, float* dw_external, void* ws, size_t ws_bytes,
                                            void* stream) {
  STAG_CHECK_ARG((dparam0 == nullptr) == (dparam1 == nullptr), "stag_attention_softmax_s_bwd: pass both parameter "
                 "gradient outputs or neither");
  AttnParams p = {};
  p.H = H; p.S = S; p.el = el; p.el_ss = el_sample_stride; p.er = er; p.er_ss = er_sample_stride; p.slope = slope;
  p.a = const_cast<float*>(a); p.da = da; p.t = dpre; p.d_er = d_er; p.dp0 = dparam0; p.dp1 = dparam1;
  p.dw = (noise && noise->kind == STAG_NOISE_EXTERNAL) ? dw_external : nullptr;
  return attention_launch(csc, p, noise, true, ws, ws_bytes, (cudaStream_t)stream, "stag_attention_softmax_s_bwd");
}
