// Fused stochastic neighbour aggregation for sm_100a.
//
// One kernel family does, in a single pass over a compressed adjacency and without ever
// writing the [E,K] noise tensor to HBM:
//   counter-based Philox noise -> reparameterisation (loc/scale, low/high, probs) -> relu
//   -> message scaling -> segmented reduction (+ in-norm, + degree scalings)
// and, in the gradient instantiation, the transposed aggregation (dX) together with the
// SDDMM term reduced straight into the noise-parameter gradients.
//
// Reference path replaced (file:line in /root/reference):
//   StagLayer.rsample_noise        stag/layers.py:115-129
//   relu / _in_norm                stag/layers.py:98-105, 8-36
//   update_all(u_mul_e, sum|mean)  stag/zoo/gcn.py:63,95  stag/zoo/graph_sage.py:57,72,86
//   degree scalings                stag/zoo/gcn.py:67-75,100-108
//   autograd of the above          DGL GSpMM.backward (gspmm on the reverse graph + gsddmm)
//
// Three kernel families share one edge schedule (StagGraph: stream items = consecutive rows holding about 64
// stored edges, rows longer than kHubThreshold cut into segments combined in a fixed order by a finalize
// kernel: deterministic):
//   agg_stream_kernel        the hot one: generated per-channel noise (or none) with scalar / per-edge
//                            parameters, forward and transposed pass; 16 channels per lane
//   agg_stream_grads_kernel  the two-sum form: parameter gradients (vi=True), per-channel parameters, relu,
//                            per-edge weights
//   agg_kernel               row per lane group, the general fallback:
//     MODE 0  per-edge scalar weight (none / external [E,1] / generated K == 1)
//     MODE 1  external per-channel weights [E,K] read from memory (the shared-noise parity seam)
//     MODE 2  per-channel noise generated in registers; PSH 0: scalar or per-edge parameters
//             (travel with the edge record, folded with the gather scale), 1: per-channel
//             parameters in registers, 2: per-edge-per-channel parameters read from memory
// A row (destination node for CSC, source node for CSR) is owned by a group of LPR lanes; a lane owns one or
// two OCTs of channels (8 floats = two 128-bit loads = one Philox block per edge).
#include <stdlib.h>
#include "common.cuh"
#include "noise.cuh"
#include "param_finalize.cuh"

#ifndef STAG_PACK2
#define STAG_PACK2 1  // packed fp32 (FFMA2 / FMUL2) Box-Muller + accumulate in agg_stream_kernel
#endif

namespace stag {

constexpr int AGG_THREADS = 256;
constexpr int AGG_WARPS = AGG_THREADS / 32;

struct AggParams {
  // structure
  const int32_t* indptr;
  const int32_t* indices;
  const int32_t* eid;
  const int32_t* hub_rows;
  const int32_t* hub_seg_ptr;
  const int32_t* row_order;  // rows in processing order (by degree), or null
  const int32_t* items;      // stream items {row0, row1, e0, e1}
  const int32_t* erow;       // row of every stored edge
  const int32_t* eidf;       // edge id of every stored edge, bit 31 set on the last edge of its row
  const int4* rec;           // per-call edge records (edge_record_kernel), workspace
  int num_items;
  uint32_t rk[2 * kPhiloxRounds];  // Philox round keys
  uint32_t kf;                     // 0x4B000000 (2^23 as float bits), read from the constant bank by PRMT
  int num_hubs, num_hub_segs;
  int N;
  int64_t ncols;  // rows of the gathered operand
  int64_t E;
  // gathered operand (x[indices[j]]), its per-node scale, row-side scale
  const float* x;
  int64_t ldx, x_ss;
  const float* gscale;
  const float* rscale;
  float* out;
  int64_t ldo, out_ss;
  int D, S, nblk, dpad;  // nblk Philox blocks per row; dpad = D rounded up to whole 64-channel groups
  int lpr_log2;
  // column blocks: the channels are processed in ncb blocks of cw floats so that the gathered
  // operand of one block ([N, cw]) stays L2-resident; cb_major orders the blocks outermost
  // (operand shared by all samples), otherwise the samples are outermost
  int ncb, cw, cb_major;
  // noise
  int kind, K, pshape, relu, in_norm, sample_base;
  const float* p0;
  const float* p1;
  const float* ext;
  PhiloxKey key;
  const uint32_t* ctr_dev;  // optional device-side addend to key.c3 (StagNoise::counter)
  float* norm_scale_out;
  // hub partial sums [S][num_hub_segs][dpad]
  float* part_acc;
  float* part_w;
  // gradient mode
  const float* xrow;
  int64_t ldxr, xr_ss;
  float* dp0;
  float* dp1;
  float* dw_ext;
  float* dp_partial;  // [grid][2][dpad]
};

// The Philox key of this launch: the host-side (seed, offset) plus the optional device-side call counter.
__device__ __forceinline__ PhiloxKey live_key(const AggParams& p) {
  PhiloxKey k = p.key;
  if (p.ctr_dev) k.c3 += __ldg(p.ctr_dev);
  return k;
}

// Channel layout of a lane: Philox block b (= lane's index among the blocks of a row) owns the two
// quads of channels starting at c = 64*(b/8) + 4*(b%8) and at c + 32, so that the 8 lanes of a
// 64-channel group read two contiguous 128-byte lines with their two 128-bit loads (noise.cuh).
__device__ __forceinline__ int chan(int c, int i) { return i < 4 ? c + i : c + 28 + i; }
__device__ __forceinline__ int first_chan(int c0, int sl) { return c0 + ((sl >> 3) << 6) + ((sl & 7) << 2); }

template <bool VEC>
__device__ __forceinline__ void load8(const float* __restrict__ row, int c, int D, float (&v)[8]) {
  if (VEC) {
    float4 a = make_float4(0.f, 0.f, 0.f, 0.f), b = a;
    if (c < D) a = __ldg(reinterpret_cast<const float4*>(row + c));
    if (c + 32 < D) b = __ldg(reinterpret_cast<const float4*>(row + c + 32));
    v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w;
    v[4] = b.x; v[5] = b.y; v[6] = b.z; v[7] = b.w;
  } else {
#pragma unroll
    for (int i = 0; i < 8; ++i) v[i] = (chan(c, i) < D) ? __ldg(row + chan(c, i)) : 0.f;
  }
}

// STREAM: evict-first store for the big output stream, so that it does not push the gathered
// operand out of L2
template <bool VEC, bool STREAM>
__device__ __forceinline__ void store8(float* __restrict__ row, int c, int D, const float (&v)[8]) {
  if (VEC) {
    const float4 a = make_float4(v[0], v[1], v[2], v[3]), b = make_float4(v[4], v[5], v[6], v[7]);
    if (STREAM) {
      if (c < D) __stcs(reinterpret_cast<float4*>(row + c), a);
      if (c + 32 < D) __stcs(reinterpret_cast<float4*>(row + c + 32), b);
    } else {
      if (c < D) *reinterpret_cast<float4*>(row + c) = a;
      if (c + 32 < D) *reinterpret_cast<float4*>(row + c + 32) = b;
    }
  } else {
#pragma unroll
    for (int i = 0; i < 8; ++i)
      if (chan(c, i) < D) row[chan(c, i)] = v[i];
  }
}

__device__ __forceinline__ float group_sum(float v, int lpr) {
  for (int o = lpr >> 1; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

__device__ __forceinline__ float sum8(const float (&v)[8]) {
  return ((v[0] + v[1]) + (v[2] + v[3])) + ((v[4] + v[5]) + (v[6] + v[7]));
}

// Hot path of MODE 2 / PSH 0 without relu / in-norm / gradients: the weights of one oct with the
// gather scale already folded into the two per-edge values (A, B) by the lane that loaded the
// edge record:   NORMAL  A = sc*loc, B = sc*scale      w*sc = A + B*eps
//                UNIFORM A = sc*low, B = sc*(high-low)  w*sc = A + B*u
//                BERNOULLI A = p,    B = sc             w*sc = u < A ? B : 0
template <int KIND>
__device__ __forceinline__ void folded_oct(uint32_t eid, uint32_t oct, uint32_t smp, const PhiloxKey& key, float A,
                                           float B, float (&w)[8]) {
  const uint4 r = philox4x32<kPhiloxRounds>(oct, eid, smp, key.c3, key.k0, key.k1);
  const uint32_t q[4] = {r.x, r.y, r.z, r.w};
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    if (KIND == STAG_NOISE_NORMAL) {
      float rad, c, s;
      bm_parts(q[i], rad, c, s);
      const float rb = rad * B;
      w[2 * i] = fmaf(c, rb, A);
      w[2 * i + 1] = fmaf(s, rb, A);
    } else if (KIND == STAG_NOISE_UNIFORM) {
      w[2 * i] = fmaf(half_uniform<false>(q[i]), B, A);
      w[2 * i + 1] = fmaf(half_uniform<true>(q[i]), B, A);
    } else {
      w[2 * i] = half_uniform<false>(q[i]) < A ? B : 0.f;
      w[2 * i + 1] = half_uniform<true>(q[i]) < A ? B : 0.f;
    }
  }
}

// ---- shared pieces of the streaming kernels -------------------------------------------------------------
// 16-byte async copy global -> shared; `ignore` set: the source is not read and zeros are written
__device__ __forceinline__ void cp_async16(uint32_t dst_smem, const void* src, bool ignore) {
  asm volatile(
      "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %2, 0;\n\tcp.async.cg.shared.global [%0], [%1], 16, p;\n\t}" ::"r"(dst_smem),
      "l"(src), "r"((int)ignore)
      : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() {
  asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory");
}

// Philox with the round keys read straight from the kernel-parameter constant bank (AggParams::rk):
// one LOP3 per key injection, no per-thread key schedule.
__device__ __forceinline__ uint4 philox_rk(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, const AggParams& p) {
  constexpr uint32_t M0 = 0xD2511F53u, M1 = 0xCD9E8D57u;
#pragma unroll
  for (int r = 0; r < kPhiloxRounds; ++r) {
    const uint64_t p0 = (uint64_t)M0 * c0;
    const uint64_t p1 = (uint64_t)M1 * c2;
    const uint32_t n0 = (uint32_t)(p1 >> 32) ^ c1 ^ p.rk[2 * r];
    const uint32_t n2 = (uint32_t)(p0 >> 32) ^ c3 ^ p.rk[2 * r + 1];
    c1 = (uint32_t)p1;
    c3 = (uint32_t)p0;
    c0 = n0;
    c2 = n2;
  }
  return make_uint4(c0, c1, c2, c3);
}

// Per-call edge records of the streaming kernel: {neighbour, eid | last-of-row << 31, A, B} with BOTH
// degree scalings (gather side and row side) and the distribution parameters folded into the pair
// (A, B) (see folded_oct), so that the stream has no dependent loads and a row is finished by a plain
// store.  Hub rows keep their row scale out of (A, B): hub_finalize_kernel applies it once.
template <int KIND>
__global__ void edge_record_kernel(const AggParams p, int4* __restrict__ rec, int scales_only) {
  // scales_only: 0 = (A, B) as documented above, 1 = the two scalings only (gradient / two-sum kernels),
  // 2 = like 0 with sqrt(2 ln 2) folded into B of Normal noise (agg_stream3_kernel takes sqrt(-lg2 u1) as radius)
  // 3 = like 0 with the variance constant of the Hadamard mix folded into B (agg_wh_stream_kernel)
  const int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (scales_only >= 2 && j == 0) reinterpret_cast<int*>(rec + p.E)[0] = 0;  // the work queue of agg_stream_kernel / agg_wh_quad_kernel (spare slot behind the records)
  if (j >= p.E) return;
  const int idx = __ldg(p.indices + j);
  const int ef = __ldg(p.eidf + j);
  const int row = __ldg(p.erow + j);
  float sc = p.gscale ? __ldg(p.gscale + idx) : 1.0f;
  if (p.rscale && __ldg(p.indptr + row + 1) - __ldg(p.indptr + row) <= kHubThreshold) sc *= __ldg(p.rscale + row);
  if (scales_only == 1 || KIND == STAG_NOISE_NONE) {  // gradient kernel: the parameters stay in registers, only the two scalings are folded
    rec[j] = make_int4(idx, ef, __float_as_int(sc), 0);
    return;
  }
  const int64_t pi = p.pshape >= STAG_PARAM_EDGE ? (ef & 0x7fffffff) : 0;
  const float pa = __ldg(p.p0 + pi);
  const float pb = KIND != STAG_NOISE_BERNOULLI ? __ldg(p.p1 + pi) : 0.f;
  float a, b;
  if (KIND == STAG_NOISE_NORMAL) { a = sc * pa; b = sc * pb * (scales_only == 2 ? 1.1774100225154747f : (scales_only == 3 ? kWhInvSd : 1.0f)); }
  else if (KIND == STAG_NOISE_UNIFORM) { a = sc * pa; b = sc * (pb - pa); }
  else { a = pa; b = sc; }
  if (scales_only == 2 && KIND == STAG_NOISE_UNIFORM) {
    // the hot kernel multiplies X = 2^23 + h (u = X / 65536 - 128) directly: w = A' + B' X, one FFMA
    a = fmaf(-128.0f, b, a);
    b *= 1.52587890625e-05f;
  }
  if (scales_only == 2 && KIND == STAG_NOISE_BERNOULLI) {
    // ... and compares X with 2^23 + ceil(65536 p): h < 65536 p  <=>  h < ceil(65536 p) for integer h (exact)
    a = 8388608.0f + ceilf(fminf(fmaxf(pa, 0.0f), 1.0f) * 65536.0f);
  }
  rec[j] = make_int4(idx, ef, __float_as_int(a), __float_as_int(b));
}

// Rows without stored edges are not visited by the edge stream: every warp of the grid checks 32 rows per load and
// writes the zeros of the empty ones (rows of the vectorised paths: D % 4 == 0, 16-byte aligned).
__device__ __forceinline__ void zero_empty_rows_tail(const AggParams& p, int64_t gwarp, int64_t nwarps, int lane) {
  if (!p.out) return;
  for (int64_t base = gwarp * 32; base < p.N; base += nwarps * 32) {
    const int64_t v = base + lane;
    const bool empty = v < p.N && __ldg(p.indptr + v + 1) == __ldg(p.indptr + v);
    unsigned m = __ballot_sync(0xffffffffu, empty);
    while (m) {
      const int64_t r = base + (__ffs(m) - 1);
      m &= m - 1;
      for (int s = 0; s < p.S; ++s) {
        float* o = p.out + (int64_t)s * p.out_ss + r * p.ldo;
        for (int c = lane * 4; c < p.D; c += 128) __stcs(reinterpret_cast<float4*>(o + c), make_float4(0.f, 0.f, 0.f, 0.f));
        if (p.in_norm && p.norm_scale_out) {  // in-norm factor of a row without edges is 1
          float* ns = p.norm_scale_out + ((int64_t)s * p.N + r) * p.K;
          for (int c = lane; c < p.K; c += 32) ns[c] = 1.0f;
        }
      }
    }
  }
}

// ---- hot kernel -------------------------------------------------------------------------------------
// Generated per-channel noise with scalar or per-edge parameters, no relu, no parameter gradients: the
// arxiv_mle configuration, forward AND transposed (dX) pass.  Template switches:
//   NB      Philox blocks (8 channels each) per lane: 2 for rows made of 128-channel groups (16 channels per
//           lane, 8 lanes per 128 channels), 1 otherwise (8 lanes per 64 channels)
//   FULL    every row is made of whole groups and there is one column block: no quad predicates
//   INNORM  Bernoulli + in-norm (the pairing the reference uses, scripts/arxiv_mle/gcn/run.py:70-74): the kept
//           in-edges per channel are counted next to the sum, the finished row is rescaled by indeg / count
//           (stag/layers.py:8-36) and the factor is written to norm_scale_out for the backward
//
// Unit of work of a lane group (LPR lanes): one STREAM ITEM = consecutive rows holding about kRangeEdges stored
// edges (StagGraph::items) or one hub segment, walked as ONE stream of edges:
//   * the edge records {neighbour, eid | last << 31, A, B'} (edge_record_kernel: both degree scalings and the
//     distribution parameters folded into (A, B'), w * scale = A + B' * raw) and the row of every edge reach
//     the group through a small shared-memory ring filled by cp.async two chunks (of LPR edges) ahead and are
//     read back with one broadcast LDS.128 (+ one LDS.32 for the neighbour of the edge being prefetched): no
//     record registers, no shuffles, no dependent global loads;
//   * the gathered row of edge t + RS is requested (cp.async, LDGSTS) into the ring slot edge t has just been
//     consumed from: RS = 4 edges in flight per lane, a lane only reads data slots it wrote itself;
//   * the loop is unrolled by RS, so every ring slot is an immediate offset;
//   * Box-Muller with sqrt(2 ln 2) folded into B' and the 2^23 magic of the half -> float conversion read
//     from the constant bank (AggParams::kf): a pair of normals costs PRMT, FFMA, LG2, SQRT | PRMT, FFMA,
//     FMUL.RZ, COS, SIN | FMUL, 2 FFMA (w) + 2 FFMA (accumulate);
//   * a row is written (st.global.cs) when the stream passes its last edge; rows without edges are cleared in
//     the kernel's tail (zero_empty_rows_tail); hub segments leave partial sums for hub_finalize_kernel.
// Where the time goes (B200, arxiv shape, 16 samples): DESIGN.md section 5.
constexpr int S3_RS = 4;    // data ring slots = edges in flight per lane
constexpr int S3_NBUF = 4;  // record chunks (of LPR edges) in the record ring
// per warp: [RS][2 NB quads][32 lanes] float4 data, then [groups][NBUF * LPR] int4 records and
// [groups][NBUF * LPR] int rows; group g starts 16 (4) bytes past a multiple of 128 so that the broadcast
// reads of the groups of a warp fall into different banks
constexpr uint32_t S3_REC_BYTES = S3_NBUF * 32 * 16 + 128;
constexpr uint32_t S3_ROW_BYTES = S3_NBUF * 32 * 4 + 128;
__host__ __device__ constexpr uint32_t s3_data_bytes(int nb) { return (uint32_t)(S3_RS * 2 * nb * 32 * 16); }
__host__ __device__ constexpr uint32_t s3_warp_bytes(int nb) { return s3_data_bytes(nb) + S3_REC_BYTES + S3_ROW_BYTES; }
__host__ __device__ constexpr int s3_min_blocks(int nb, bool innorm) { return (nb == 1 && !innorm) ? 3 : 2; }

__device__ __forceinline__ void cp_async4(uint32_t dst_smem, const void* src, bool ignore) {
  asm volatile(
      "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %2, 0;\n\tcp.async.ca.shared.global [%0], [%1], 4, p;\n\t}" ::"r"(dst_smem),
      "l"(src), "r"((int)ignore)
      : "memory");
}
__device__ __forceinline__ int4 lds128(uint32_t a) {
  int4 v;
  asm volatile("ld.shared.v4.b32 {%0,%1,%2,%3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(a));
  return v;
}
__device__ __forceinline__ float4 lds128f(uint32_t a) {
  float4 v;
  asm volatile("ld.shared.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(a));
  return v;
}
__device__ __forceinline__ int lds32(uint32_t a) {
  int v;
  asm volatile("ld.shared.b32 %0, [%1];" : "=r"(v) : "r"(a));
  return v;
}

// 8 warps x 2 CTAs per SM at 128 registers: 10 or 12 warps per CTA (96 / 80 registers) measured slower
constexpr int S3_THREADS = 256, S3_WARPS = S3_THREADS / 32;

template <int KIND, int NB, bool FULL, bool INNORM>
__global__ void __launch_bounds__(S3_THREADS, s3_min_blocks(NB, INNORM)) agg_stream_kernel(const AggParams p) {
  const PhiloxKey key = live_key(p);
  extern __shared__ float4 ring[];
  constexpr int RS = S3_RS, NQ = 2 * NB, GW = 64 * NB, NA = 4 * NQ;
  constexpr uint32_t DATA_BYTES = s3_data_bytes(NB), WARP_BYTES = s3_warp_bytes(NB), SLOT = NQ * 512u;
  static_assert(!INNORM || KIND == STAG_NOISE_BERNOULLI, "in-norm is fused for Bernoulli noise only");
  const int lane = threadIdx.x & 31;
  const int warp = threadIdx.x >> 5;
  const int LPR = 1 << p.lpr_log2;  // lanes per row (>= 8); a record chunk is LPR edges
  const int RPW = 32 >> p.lpr_log2;
  const int sub = lane >> p.lpr_log2;
  const int sl = lane & (LPR - 1);
  const int D8 = p.dpad;
  const uint32_t warp_s = (uint32_t)__cvta_generic_to_shared(ring) + (uint32_t)warp * WARP_BYTES;
  const uint32_t data_s = warp_s + (uint32_t)lane * 16u;  // + slot * SLOT + quad * 512
  const uint32_t rmask = (uint32_t)(S3_NBUF * LPR) - 1u;  // record ring positions of a group
  const uint32_t rec_g = warp_s + DATA_BYTES + (uint32_t)(sub * S3_NBUF * LPR) * 16u + (uint32_t)sub * 16u;
  const uint32_t row_g = warp_s + DATA_BYTES + S3_REC_BYTES + (uint32_t)(sub * S3_NBUF * LPR) * 4u + (uint32_t)sub * 4u;
  const uint32_t kf = p.kf;

  const int n_items = p.num_hub_segs + p.num_items;
  const int IG = (n_items + RPW - 1) / RPW;  // warp items per (sample, column block)
  const int64_t total = (int64_t)IG * p.S * p.ncb;
  const int64_t total_warps = (int64_t)gridDim.x * S3_WARPS;

  // warp items come from a queue (a counter behind the edge records, zeroed by edge_record_kernel): they differ in
  // length, and with a static stride the slowest warp had ~10 % more edges than the average (tools/item_balance.py).
  // The next index is requested before the current item is walked.
  int* const queue = reinterpret_cast<int*>(const_cast<int4*>(p.rec) + p.E);
  int64_t item;
  {
    int v = 0;
    if (lane == 0) v = atomicAdd(queue, 1);
    item = __shfl_sync(0xffffffffu, v, 0);
  }
  for (int nxt = 0; item < total; item = __shfl_sync(0xffffffffu, nxt, 0)) {
    if (lane == 0) nxt = atomicAdd(queue, 1);
    const int64_t outer = item / IG;
    const int gi = (int)(item - outer * IG) * RPW + sub;
    int s, cb;
    if (p.cb_major) {
      cb = (int)(outer / p.S);
      s = (int)(outer - (int64_t)cb * p.S);
    } else {
      s = (int)(outer / p.ncb);
      cb = (int)(outer - (int64_t)s * p.ncb);
    }
    const int c_begin = cb * p.cw;
    const int c_end = min(c_begin + p.cw, D8);
    // resolve the group's item: stored edges [e0, e1)
    int e0 = 0, e1 = 0, part_slot = -1;
    if (gi < p.num_hub_segs) {
      int lo = 0, hi = p.num_hubs;  // last hub with hub_seg_ptr[h] <= gi
      while (hi - lo > 1) {
        const int mid = (lo + hi) >> 1;
        if (__ldg(p.hub_seg_ptr + mid) <= gi) lo = mid; else hi = mid;
      }
      const int row = __ldg(p.hub_rows + lo);
      const int k = gi - __ldg(p.hub_seg_ptr + lo);
      e0 = __ldg(p.indptr + row) + k * kHubSegment;
      e1 = min(e0 + kHubSegment, __ldg(p.indptr + row + 1));
      part_slot = gi;
    } else if (gi < n_items) {
      const int4 it = __ldg(reinterpret_cast<const int4*>(p.items) + (gi - p.num_hub_segs));
      e0 = it.z;
      e1 = it.w >= 0 ? it.w : it.z;  // it.w < 0: placeholder of a hub row, nothing to do here
    }
    const int nedges = e1 - e0;
    const int rowlim = part_slot < 0 ? nedges : 0;  // edges that may close a row (none in a hub segment)
    int maxn = nedges;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) maxn = max(maxn, __shfl_xor_sync(0xffffffffu, maxn, o));

    const float* xs = p.x + (int64_t)s * p.x_ss;
    float* outs = p.out + (int64_t)s * p.out_ss;
    const uint32_t smp = (uint32_t)(p.sample_base + s);
    const uint32_t ldxb = (uint32_t)p.ldx * 4u;
    const int4* recp = p.rec + e0;
    const int32_t* rowp = p.erow + e0;

    for (int c0 = c_begin; c0 < c_end; c0 += (LPR >> 3) * GW) {
      const int c = c0 + (sl >> 3) * GW + ((sl & 7) << 2);  // quads at c + 32 j
      bool qv[NQ];
#pragma unroll
      for (int j = 0; j < NQ; ++j) qv[j] = FULL || (c + 32 * j < p.D && c + 32 * j < c_end);
      const uint32_t blk0 = (uint32_t)((c0 >> 3) + (sl >> 3) * 8 * NB + (sl & 7));  // Philox blocks blk0 + 8 g
      const char* xcb = reinterpret_cast<const char*>(xs + (qv[0] ? c : 0));
      float acc[NA], cntw[INNORM ? NA : 1];
#pragma unroll
      for (int i = 0; i < NA; ++i) acc[i] = 0.f;
      if (INNORM) {
#pragma unroll
        for (int i = 0; i < NA; ++i) cntw[INNORM ? i : 0] = 0.f;
      }
      int row_edges = 0;  // INNORM: in-edges of the current row seen so far

      // record chunk: edges first + sl of the item -> ring position (first + sl) & rmask (zeros past the end)
      auto fetch_chunk = [&](int first) {
        const int e = first + sl;
        const uint32_t pos = (uint32_t)e & rmask;
        const bool off = e >= nedges;
        cp_async16(rec_g + pos * 16u, recp + (off ? 0 : e), off);
        cp_async4(row_g + pos * 4u, rowp + (off ? 0 : e), off);
      };
      // gathered row of edge e (its neighbour read from the record ring) -> data ring slot
      auto issue = [&](int e, uint32_t rec_addr, int slot) {
        const uint32_t u = (uint32_t)lds32(rec_addr);
        const char* src = xcb + (uint64_t)u * ldxb;
        const uint32_t dst = data_s + (uint32_t)slot * SLOT;
        const bool off = e >= nedges;
#pragma unroll
        for (int j = 0; j < NQ; ++j) cp_async16(dst + (uint32_t)j * 512u, src + 128 * j, off || !qv[j]);
      };
      auto put_row = [&](float* rowq, int width, const float* v) {
#pragma unroll
        for (int j = 0; j < NQ; ++j)
          if (FULL || (c + 32 * j < width && qv[j]))
            __stcs(reinterpret_cast<float4*>(rowq + c + 32 * j),
                   make_float4(v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]));
      };

      // prologue: two record chunks, then the first RS gathered rows (one commit group each)
      fetch_chunk(0);
      fetch_chunk(LPR);
      cp_async_commit();
      cp_async_wait<0>();
      __syncwarp();
#pragma unroll
      for (int i = 0; i < RS; ++i) {
        issue(i, rec_g + (uint32_t)i * 16u, i);
        cp_async_commit();
      }

      for (int t = 0; t < maxn; t += RS) {
        if ((t & (LPR - 1)) == 0) fetch_chunk(t + 2 * LPR);  // joins the first group committed below
        const uint32_t rbase = rec_g + (((uint32_t)t & rmask) << 4);
        const uint32_t ibase = rec_g + (((uint32_t)(t + RS) & rmask) << 4);
        const uint32_t wbase = row_g + (((uint32_t)t & rmask) << 2);
#pragma unroll
        for (int j = 0; j < RS; ++j) {
          // groups committed so far: RS + t + j; all but the last RS - 1 are complete, i.e. the row of edge
          // t + j and every record chunk up to the one edge t + j + RS lives in
          cp_async_wait<RS - 1>();
          // records are written by other lanes of the group: a chunk requested at edge t0 has landed in every
          // lane by edge t0 + RS and is first read at t0 + 2 LPR - RS, so one warp barrier per RS edges orders it
          if (j == 0) __syncwarp();
          const int4 rc = lds128(rbase + (uint32_t)j * 16u);
          const int ef = rc.y;
          const float A = __int_as_float(rc.z), B = __int_as_float(rc.w);
          const uint32_t slot_s = data_s + (uint32_t)j * SLOT;
          uint32_t q[4 * NB];
          if (KIND != STAG_NOISE_NONE) {
#pragma unroll
            for (int g = 0; g < NB; ++g) {
              const uint4 r4 = philox_rk(blk0 + (uint32_t)(8 * g), (uint32_t)(ef & 0x7fffffff), smp, key.c3, p);
              q[4 * g] = r4.x; q[4 * g + 1] = r4.y; q[4 * g + 2] = r4.z; q[4 * g + 3] = r4.w;
            }
          }
#pragma unroll
          for (int g = 0; g < NB; ++g) {
#if STAG_PACK2
            if (KIND == STAG_NOISE_NORMAL) {
              // Same arithmetic as the scalar branch below (every operation is one IEEE fp32 fma / mul), issued
              // as packed FFMA2 / FMUL2 on register pairs: half the FMA-pipe instructions per variate.
              const float2 AA = make_float2(A, A), BB = make_float2(B, B);
              float2 wp[4];
#pragma unroll
              for (int ip = 0; ip < 2; ++ip) {
                const uint32_t qa = q[4 * g + 2 * ip], qb = q[4 * g + 2 * ip + 1];
                const float2 xl = make_float2(__uint_as_float(__byte_perm(qa, kf, 0x7610)),
                                              __uint_as_float(__byte_perm(qb, kf, 0x7610)));
                const float2 xh = make_float2(__uint_as_float(__byte_perm(qa, kf, 0x7632)),
                                              __uint_as_float(__byte_perm(qb, kf, 0x7632)));
                const float2 u1 = __ffma2_rn(xl, make_float2(1.52587890625e-05f, 1.52587890625e-05f),
                                             make_float2(-127.99999237060547f, -127.99999237060547f));
                const float2 ang = __ffma2_rn(xh, make_float2(9.58738019107841e-05f, 9.58738019107841e-05f),
                                              make_float2(-804.2476806640625f, -804.2476806640625f));
                const float2 rb = __fmul2_rn(make_float2(mufu_sqrt(-mufu_lg2(u1.x)), mufu_sqrt(-mufu_lg2(u1.y))), BB);
                wp[2 * ip] = __ffma2_rn(make_float2(mufu_cos(ang.x), mufu_sin(ang.x)), make_float2(rb.x, rb.x), AA);
                wp[2 * ip + 1] = __ffma2_rn(make_float2(mufu_cos(ang.y), mufu_sin(ang.y)), make_float2(rb.y, rb.y), AA);
              }
#pragma unroll
              for (int h = 0; h < 2; ++h) {
                const int jq = 2 * g + h;
                const float4 x4 = lds128f(slot_s + (uint32_t)jq * 512u);
                float* a4 = acc + 4 * jq;
                const float2 r0 = __ffma2_rn(wp[2 * h], make_float2(x4.x, x4.y), make_float2(a4[0], a4[1]));
                const float2 r1 = __ffma2_rn(wp[2 * h + 1], make_float2(x4.z, x4.w), make_float2(a4[2], a4[3]));
                a4[0] = r0.x; a4[1] = r0.y; a4[2] = r1.x; a4[3] = r1.y;
              }
            } else {
#else
            {
#endif
            float w[8], kept[INNORM ? 8 : 1];
#pragma unroll
            for (int i = 0; i < 4; ++i) {
              if (KIND == STAG_NOISE_NONE) {  // plain copy_u / sum: the folded scale is the weight
                w[2 * i] = w[2 * i + 1] = A;
                continue;
              }
              const float xl = __uint_as_float(__byte_perm(q[4 * g + i], kf, 0x7610));  // 2^23 + h_lo
              const float xh = __uint_as_float(__byte_perm(q[4 * g + i], kf, 0x7632));  // 2^23 + h_hi
              if (KIND == STAG_NOISE_NORMAL) {
                const float u1 = fmaf(xl, 1.52587890625e-05f, -127.99999237060547f);      // (h_lo + 1/2) / 65536
                const float rb = mufu_sqrt(-mufu_lg2(u1)) * B;                             // B' carries sqrt(2 ln 2)
                const float ang = fmaf(xh, 9.58738019107841e-05f, -804.2476806640625f);   // 2 pi (h_hi + 1/2) / 65536
                w[2 * i] = fmaf(mufu_cos(ang), rb, A);
                w[2 * i + 1] = fmaf(mufu_sin(ang), rb, A);
              } else if (KIND == STAG_NOISE_UNIFORM) {  // (A, B) carry the half -> uniform conversion
#if STAG_PACK2
                const float2 w2 = __ffma2_rn(make_float2(xl, xh), make_float2(B, B), make_float2(A, A));
                w[2 * i] = w2.x;
                w[2 * i + 1] = w2.y;
#else
                w[2 * i] = fmaf(xl, B, A);
                w[2 * i + 1] = fmaf(xh, B, A);
#endif
              } else {  // A = 2^23 + ceil(65536 p)
                const bool k0 = xl < A, k1 = xh < A;
                w[2 * i] = k0 ? B : 0.f;
                w[2 * i + 1] = k1 ? B : 0.f;
                if (INNORM) {
                  kept[INNORM ? 2 * i : 0] = k0 ? 1.0f : 0.0f;
                  kept[INNORM ? 2 * i + 1 : 0] = k1 ? 1.0f : 0.0f;
                }
              }
            }
#pragma unroll
            for (int h = 0; h < 2; ++h) {
              const int jq = 2 * g + h;
              const float4 x4 = lds128f(slot_s + (uint32_t)jq * 512u);
              float* a4 = acc + 4 * jq;
#if STAG_PACK2
              const float2 r0 = __ffma2_rn(make_float2(w[4 * h], w[4 * h + 1]), make_float2(x4.x, x4.y), make_float2(a4[0], a4[1]));
              const float2 r1 = __ffma2_rn(make_float2(w[4 * h + 2], w[4 * h + 3]), make_float2(x4.z, x4.w), make_float2(a4[2], a4[3]));
              a4[0] = r0.x; a4[1] = r0.y; a4[2] = r1.x; a4[3] = r1.y;
#else
              a4[0] = fmaf(w[4 * h + 0], x4.x, a4[0]);
              a4[1] = fmaf(w[4 * h + 1], x4.y, a4[1]);
              a4[2] = fmaf(w[4 * h + 2], x4.z, a4[2]);
              a4[3] = fmaf(w[4 * h + 3], x4.w, a4[3]);
#endif
              if (INNORM && t + j < nedges) {
#pragma unroll
                for (int i = 0; i < 4; ++i) cntw[INNORM ? 4 * jq + i : 0] += kept[INNORM ? 4 * h + i : 0];
              }
            }
            }  // scalar / non-Normal branch
          }
          if (INNORM && t + j < nedges) ++row_edges;
          if (ef < 0 && t + j < rowlim) {  // last edge of a row: write it, start the next one
            const int rw = lds32(wbase + (uint32_t)j * 4u);
            if (INNORM) {
              float sc[NA];
#pragma unroll
              for (int i = 0; i < NA; ++i) {
                // both are small integers: the fast division is exact to 2 ulp
                sc[i] = cntw[INNORM ? i : 0] != 0.f ? __fdividef((float)row_edges, cntw[INNORM ? i : 0]) : 1.0f;
                acc[i] *= sc[i];
                cntw[INNORM ? i : 0] = 0.f;
              }
              row_edges = 0;
              if (p.norm_scale_out) put_row(p.norm_scale_out + ((int64_t)s * p.N + rw) * p.K, p.K, sc);
            }
            put_row(outs + (int64_t)rw * p.ldo, p.D, acc);
#pragma unroll
            for (int i = 0; i < NA; ++i) acc[i] = 0.f;
          }
          // the slot just consumed takes the row of edge t + j + RS
          issue(t + j + RS, ibase + (uint32_t)j * 16u, j);
          cp_async_commit();
        }
      }
      cp_async_wait<0>();
      __syncwarp();
      if (part_slot >= 0) {  // hub segment: its partial sum, combined by hub_finalize_kernel
        const int64_t o = ((int64_t)s * p.num_hub_segs + part_slot) * D8;
        put_row(p.part_acc + o, D8, acc);
        if (INNORM) put_row(p.part_w + o, D8, cntw);
      }
    }
  }
  // rows without stored edges are not visited by the edge stream: their zeros are written here, by whichever
  // warps run out of items first
  zero_empty_rows_tail(p, (int64_t)blockIdx.x * S3_WARPS + warp, total_warps, lane);
}

// ---- streaming gradient kernel ---------------------------------------------------------------------
// Transposed pass with noise-parameter gradients (vi = True) for generated per-channel Normal / Uniform
// noise with scalar or per-channel parameters (the r1 / rc posteriors), D <= 256, no in-norm.  Rows are
// SOURCE nodes (CSR), the gathered operand is dOut.  Same edge stream as agg_stream_kernel; per row it
// keeps TWO sums over the out-edges,
//     a0[c] = sum_e m_e,c * A_e * dout[v_e,c]          a1[c] = sum_e m_e,c * A_e * dout[v_e,c] * r_e,c
// (A_e = dst_scale[v_e] * src_scale[u], r = eps or u regenerated from the edge id, m = relu mask), from
// which everything follows at the end of the row without ever touching x inside the edge loop:
//     dx[u,c]      = P0[c] * a0 + P1'[c] * a1            (P1' = scale, or high - low)
//     d P0[c]     += x[u,c] * a0   (Uniform: x * (a0 - a1))      d P1[c] += x[u,c] * a1
// The row of x needed at the end of a row is fetched by cp.async together with the row's last edge.
// The same kernel serves two more cases (template switches):
//   PG = false           the two-sum FORWARD for per-channel parameters (or relu): out = P0*a0 + P1'*a1
//   BODY = 1 (PG false)  per-edge weights (no noise / external [E,1] / generated K == 1 with scalar
//                        parameters): the lane that loads an edge record computes its weight, out = a0
// Shared-memory layout per warp: [RS][NQS quads][32 lanes] float4 (NQS = 2 NB quads of the gathered row, with PG
// as many again for the row's own features), then the record and row rings of the hot kernel; the
// parameter-gradient staging follows the warps.
// NB = 2 (16 channels per lane) serves scalar parameters and BODY 1 on rows made of 128-channel groups: the
// parameters and their gradients are then one register each; per-channel parameters keep NB = 1.
// (with PG and NB = 2 the ring keeps 2 edges in flight instead of 4, so that two CTAs still share an SM)
__host__ __device__ constexpr int s2_ring_slots(bool pg, int nb) { return (pg && nb == 2) ? 2 : S3_RS; }
__host__ __device__ constexpr uint32_t s2_warp_bytes(bool pg, int nb) {
  return (uint32_t)(s2_ring_slots(pg, nb) * (pg ? 4 : 2) * nb * 512) + S3_REC_BYTES + S3_ROW_BYTES;
}

template <int KIND, int BODY, bool PG, int NB>
__global__ void __launch_bounds__(AGG_THREADS, 2) agg_stream_grads_kernel(const AggParams p) {
  const PhiloxKey key = live_key(p);
  extern __shared__ float4 ring[];
  constexpr int RS = s2_ring_slots(PG, NB), NQ = 2 * NB, NA = 4 * NQ, GW = 64 * NB, NQS = PG ? 2 * NQ : NQ;
  constexpr int NP = NB == 1 ? 8 : 1;  // parameter (gradient) registers: per channel, or one scalar
  constexpr uint32_t SLOT = NQS * 512u, DATA_BYTES = RS * SLOT, WARP_BYTES = s2_warp_bytes(PG, NB);
  constexpr float kRad = 1.1774100225154747f;  // sqrt(2 ln 2): the radius is taken as sqrt(-lg2 u1)
  const int lane = threadIdx.x & 31;
  const int warp = threadIdx.x >> 5;
  const int LPR = 1 << p.lpr_log2;  // >= 8 (launcher)
  const int RPW = 32 >> p.lpr_log2;
  const int sub = lane >> p.lpr_log2;
  const int sl = lane & (LPR - 1);
  const int D8 = p.dpad;
  const uint32_t warp_s = (uint32_t)__cvta_generic_to_shared(ring) + (uint32_t)warp * WARP_BYTES;
  const uint32_t data_s = warp_s + (uint32_t)lane * 16u;
  const uint32_t rmask = (uint32_t)(S3_NBUF * LPR) - 1u;
  const uint32_t rec_g = warp_s + DATA_BYTES + (uint32_t)(sub * S3_NBUF * LPR) * 16u + (uint32_t)sub * 16u;
  const uint32_t row_g = warp_s + DATA_BYTES + S3_REC_BYTES + (uint32_t)(sub * S3_NBUF * LPR) * 4u + (uint32_t)sub * 4u;
  float* stage = reinterpret_cast<float*>(reinterpret_cast<char*>(ring) + (size_t)AGG_WARPS * WARP_BYTES);  // [AGG_WARPS][2][dpad]
  const uint32_t kf = p.kf;

  const int n_items = p.num_hub_segs + p.num_items;
  const int IG = (n_items + RPW - 1) / RPW;
  const int64_t total = (int64_t)IG * p.S;
  const int64_t total_warps = (int64_t)gridDim.x * AGG_WARPS;

  // this lane's channels (single pass: dpad <= LPR * 8 NB): quads at c + 32 j; element i is channel
  // c + 32 (i / 4) + i % 4.  Normal: P1 carries sqrt(2 ln 2)
  const int c = (sl >> 3) * GW + ((sl & 7) << 2);
  bool qv[NQ];
#pragma unroll
  for (int j = 0; j < NQ; ++j) qv[j] = c + 32 * j < p.D;
  const uint32_t blk0 = (uint32_t)((sl >> 3) * 8 * NB + (sl & 7));  // Philox blocks blk0 + 8 g
  float P0[NP], P1[NP], d0[NP], d1[NP];
#pragma unroll
  for (int i = 0; i < NP; ++i) {
    const int ch = c + 32 * (i >> 2) + (i & 3);
    const int64_t pi = (NB == 2 || p.pshape == STAG_PARAM_SCALAR) ? 0 : (ch < p.D ? ch : 0);
    P0[i] = BODY == 0 ? __ldg(p.p0 + pi) : 1.0f;
    P1[i] = BODY == 0 ? __ldg(p.p1 + pi) : 0.0f;
    if (BODY == 0 && KIND == STAG_NOISE_UNIFORM) P1[i] -= P0[i];  // w = low + u * (high - low)
    if (BODY == 0 && KIND == STAG_NOISE_NORMAL) P1[i] *= kRad;
    d0[i] = d1[i] = 0.f;
  }
  const uint32_t ldxb = (uint32_t)p.ldx * 4u, ldxrb = (uint32_t)p.ldxr * 4u;

  for (int64_t item = (int64_t)blockIdx.x * AGG_WARPS + warp; item < total; item += total_warps) {
    const int s = (int)(item / IG);
    const int gi = (int)(item - (int64_t)s * IG) * RPW + sub;
    int e0 = 0, e1 = 0, part_slot = -1, hub_row = 0;
    if (gi < p.num_hub_segs) {
      int lo = 0, hi = p.num_hubs;
      while (hi - lo > 1) {
        const int mid = (lo + hi) >> 1;
        if (__ldg(p.hub_seg_ptr + mid) <= gi) lo = mid; else hi = mid;
      }
      hub_row = __ldg(p.hub_rows + lo);
      const int k = gi - __ldg(p.hub_seg_ptr + lo);
      e0 = __ldg(p.indptr + hub_row) + k * kHubSegment;
      e1 = min(e0 + kHubSegment, __ldg(p.indptr + hub_row + 1));
      part_slot = gi;
    } else if (gi < n_items) {
      const int4 it = __ldg(reinterpret_cast<const int4*>(p.items) + (gi - p.num_hub_segs));
      e0 = it.z;
      e1 = it.w >= 0 ? it.w : it.z;
    }
    const int nedges = e1 - e0;
    const int rowlim = part_slot < 0 ? nedges : 0;
    int maxn = nedges;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) maxn = max(maxn, __shfl_xor_sync(0xffffffffu, maxn, o));

    const char* gsb = reinterpret_cast<const char*>(p.x + (int64_t)s * p.x_ss + (qv[0] ? c : 0));  // gathered operand
    const char* xrb = PG ? reinterpret_cast<const char*>(p.xrow + (int64_t)s * p.xr_ss + (qv[0] ? c : 0)) : nullptr;
    float* outs = p.out ? p.out + (int64_t)s * p.out_ss : nullptr;
    const uint32_t smp = (uint32_t)(p.sample_base + s);
    const int4* recp = p.rec + e0;
    const int32_t* rowp = p.erow + e0;
    float a0[NA], a1[NA];
#pragma unroll
    for (int i = 0; i < NA; ++i) a0[i] = a1[i] = 0.f;

    // records {neighbour, eid | last << 31, A, -} and rows -> rings (zeros past the end of the item)
    auto fetch_chunk = [&](int first) {
      const int e = first + sl;
      const uint32_t pos = (uint32_t)e & rmask;
      const bool off = e >= nedges;
      cp_async16(rec_g + pos * 16u, recp + (off ? 0 : e), off);
      cp_async4(row_g + pos * 4u, rowp + (off ? 0 : e), off);
    };
    // BODY 1 with a per-edge weight (external [E,1] or generated K == 1): the lane that owns ring position
    // first + sl folds the weight of its (edge, sample) into A once the chunk has landed
    auto weight_chunk = [&](int first) {
      if (BODY == 1 && p.kind != STAG_NOISE_NONE && first + sl < nedges) {
        const uint32_t a = rec_g + (((uint32_t)(first + sl) & rmask) << 4);
        const int eid = lds32(a + 4u) & 0x7fffffff;
        float w;
        if (p.kind == STAG_NOISE_EXTERNAL) {
          w = __ldg(p.ext + (int64_t)s * p.E + eid);
        } else {
          w = transform_rt(p.kind, raw_first(p.kind, (uint32_t)eid, smp, key), __ldg(p.p0), p.p1 ? __ldg(p.p1) : 0.f);
        }
        if (p.relu) w = fmaxf(w, 0.f);
        const float A = __int_as_float(lds32(a + 8u)) * w;
        asm volatile("st.shared.b32 [%0], %1;" ::"r"(a + 8u), "r"(__float_as_int(A)) : "memory");
      }
    };
    auto issue = [&](int e, uint32_t rec_addr, uint32_t row_addr, int slot) {
      const bool off = e >= nedges;
      const uint32_t dst = data_s + (uint32_t)slot * SLOT;
      if (PG) {
        const int4 r = lds128(rec_addr);
        const char* src = gsb + (uint64_t)(uint32_t)r.x * ldxb;
#pragma unroll
        for (int j = 0; j < NQ; ++j) cp_async16(dst + (uint32_t)j * 512u, src + 128 * j, off || !qv[j]);
        if (r.y < 0 && e < rowlim) {  // the row ends with this edge: fetch its own feature row as well
          const char* xs = xrb + (uint64_t)(uint32_t)lds32(row_addr) * ldxrb;
#pragma unroll
          for (int j = 0; j < NQ; ++j) cp_async16(dst + (uint32_t)(NQ + j) * 512u, xs + 128 * j, !qv[j]);
        }
      } else {
        const char* src = gsb + (uint64_t)(uint32_t)lds32(rec_addr) * ldxb;
#pragma unroll
        for (int j = 0; j < NQ; ++j) cp_async16(dst + (uint32_t)j * 512u, src + 128 * j, off || !qv[j]);
      }
    };
    auto put_row = [&](float* rowq, int width, const float* v, bool streaming) {
#pragma unroll
      for (int j = 0; j < NQ; ++j)
        if (c + 32 * j < width && qv[j]) {
          const float4 q4 = make_float4(v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]);
          if (streaming) __stcs(reinterpret_cast<float4*>(rowq + c + 32 * j), q4);
          else *reinterpret_cast<float4*>(rowq + c + 32 * j) = q4;
        }
    };
    // parameter gradients of a finished row (or hub segment) against the row's own features xr
    auto add_param_grads = [&](const float* xr) {
#pragma unroll
      for (int i = 0; i < NA; ++i) {
        const int k = NB == 1 ? i : 0;
        const float t1 = xr[i] * a1[i];
        d1[k] += t1;
        d0[k] += KIND == STAG_NOISE_NORMAL ? xr[i] * a0[i] : xr[i] * a0[i] - t1;
      }
    };

    fetch_chunk(0);
    fetch_chunk(LPR);
    cp_async_commit();
    cp_async_wait<0>();
    __syncwarp();
    weight_chunk(0);
    weight_chunk(LPR);
    __syncwarp();
#pragma unroll
    for (int i = 0; i < RS; ++i) {
      issue(i, rec_g + (uint32_t)i * 16u, row_g + (uint32_t)i * 4u, i);
      cp_async_commit();
    }

    for (int t = 0; t < maxn; t += RS) {
      if ((t & (LPR - 1)) == 0) {
        // chunk t / LPR + 2 is requested now; it is complete (and its weights are folded) one chunk later,
        // LPR - RS edges before its first record is needed
        if (t > 0) weight_chunk(t + LPR);
        fetch_chunk(t + 2 * LPR);
      }
      const uint32_t rbase = rec_g + (((uint32_t)t & rmask) << 4);
      const uint32_t ibase = rec_g + (((uint32_t)(t + RS) & rmask) << 4);
      const uint32_t wbase = row_g + (((uint32_t)t & rmask) << 2);
      const uint32_t vbase = row_g + (((uint32_t)(t + RS) & rmask) << 2);
#pragma unroll
      for (int j = 0; j < RS; ++j) {
        cp_async_wait<RS - 1>();
        if (j == 0) __syncwarp();  // one warp barrier per RS edges orders the record chunks (see agg_stream_kernel)
        const int4 rc = lds128(rbase + (uint32_t)j * 16u);
        const int ef = rc.y;
        const float A = __int_as_float(rc.z);
        const uint32_t slot_s = data_s + (uint32_t)j * SLOT;
        float raw[NA];
        if (BODY == 0) {
#pragma unroll
          for (int g = 0; g < NB; ++g) {
            const uint4 r4 = philox_rk(blk0 + (uint32_t)(8 * g), (uint32_t)(ef & 0x7fffffff), smp, key.c3, p);
            const uint32_t q[4] = {r4.x, r4.y, r4.z, r4.w};
#if STAG_PACK2
            // same operations as the scalar loop below, two words at a time on FFMA2 / FMUL2
#pragma unroll
            for (int ip = 0; ip < 2; ++ip) {
              const uint32_t qa = q[2 * ip], qb = q[2 * ip + 1];
              const float2 xl = make_float2(__uint_as_float(__byte_perm(qa, kf, 0x7610)),
                                            __uint_as_float(__byte_perm(qb, kf, 0x7610)));
              const float2 xh = make_float2(__uint_as_float(__byte_perm(qa, kf, 0x7632)),
                                            __uint_as_float(__byte_perm(qb, kf, 0x7632)));
              float2 ra, rb2;
              if (KIND == STAG_NOISE_NORMAL) {
                const float2 u1 = __ffma2_rn(xl, make_float2(1.52587890625e-05f, 1.52587890625e-05f),
                                             make_float2(-127.99999237060547f, -127.99999237060547f));
                const float2 ang = __ffma2_rn(xh, make_float2(9.58738019107841e-05f, 9.58738019107841e-05f),
                                              make_float2(-804.2476806640625f, -804.2476806640625f));
                const float rad0 = mufu_sqrt(-mufu_lg2(u1.x)), rad1 = mufu_sqrt(-mufu_lg2(u1.y));
                ra = __fmul2_rn(make_float2(mufu_cos(ang.x), mufu_sin(ang.x)), make_float2(rad0, rad0));
                rb2 = __fmul2_rn(make_float2(mufu_cos(ang.y), mufu_sin(ang.y)), make_float2(rad1, rad1));
              } else {
                const float2 k = make_float2(1.52587890625e-05f, 1.52587890625e-05f), o = make_float2(-128.0f, -128.0f);
                ra = __ffma2_rn(make_float2(xl.x, xh.x), k, o);
                rb2 = __ffma2_rn(make_float2(xl.y, xh.y), k, o);
              }
              raw[8 * g + 4 * ip] = ra.x; raw[8 * g + 4 * ip + 1] = ra.y;
              raw[8 * g + 4 * ip + 2] = rb2.x; raw[8 * g + 4 * ip + 3] = rb2.y;
            }
#else
#pragma unroll
            for (int i = 0; i < 4; ++i) {
              const float xl = __uint_as_float(__byte_perm(q[i], kf, 0x7610));
              const float xh = __uint_as_float(__byte_perm(q[i], kf, 0x7632));
              if (KIND == STAG_NOISE_NORMAL) {  // eps / sqrt(2 ln 2)
                const float rad = mufu_sqrt(-mufu_lg2(fmaf(xl, 1.52587890625e-05f, -127.99999237060547f)));
                const float ang = fmaf(xh, 9.58738019107841e-05f, -804.2476806640625f);
                raw[8 * g + 2 * i] = rad * mufu_cos(ang);
                raw[8 * g + 2 * i + 1] = rad * mufu_sin(ang);
              } else {
                raw[8 * g + 2 * i] = fmaf(xl, 1.52587890625e-05f, -128.0f);
                raw[8 * g + 2 * i + 1] = fmaf(xh, 1.52587890625e-05f, -128.0f);
              }
            }
#endif
          }
        }
        float xv[NA];
#pragma unroll
        for (int jq = 0; jq < NQ; ++jq) {
          const float4 x4 = lds128f(slot_s + (uint32_t)jq * 512u);
          xv[4 * jq] = x4.x; xv[4 * jq + 1] = x4.y; xv[4 * jq + 2] = x4.z; xv[4 * jq + 3] = x4.w;
        }
#if STAG_PACK2
        if (BODY == 0) {
#pragma unroll
          for (int i = 0; i < NA; i += 2) {
            float2 y = __fmul2_rn(make_float2(xv[i], xv[i + 1]), make_float2(A, A));
            const float2 r2 = make_float2(raw[i], raw[i + 1]);
            if (p.relu) {
              const float2 t2 = __ffma2_rn(r2, make_float2(P1[NB == 1 ? i : 0], P1[NB == 1 ? i + 1 : 0]),
                                           make_float2(P0[NB == 1 ? i : 0], P0[NB == 1 ? i + 1 : 0]));
              if (!(t2.x > 0.f)) y.x = 0.f;
              if (!(t2.y > 0.f)) y.y = 0.f;
            }
            const float2 s0 = __fadd2_rn(make_float2(a0[i], a0[i + 1]), y);
            const float2 s1 = __ffma2_rn(r2, y, make_float2(a1[i], a1[i + 1]));
            a0[i] = s0.x; a0[i + 1] = s0.y; a1[i] = s1.x; a1[i + 1] = s1.y;
          }
        } else
#endif
#pragma unroll
        for (int i = 0; i < NA; ++i) {
          if (BODY == 1) {
            a0[i] = fmaf(A, xv[i], a0[i]);
          } else {
            float y = A * xv[i];
            if (p.relu && !(fmaf(raw[i], P1[NB == 1 ? i : 0], P0[NB == 1 ? i : 0]) > 0.f)) y = 0.f;
            a0[i] += y;
            a1[i] = fmaf(raw[i], y, a1[i]);
          }
        }
        if (ef < 0 && t + j < rowlim) {  // end of a row: group-uniform
          const int rw = lds32(wbase + (uint32_t)j * 4u);
          float dxv[NA];
#pragma unroll
          for (int i = 0; i < NA; ++i)
            dxv[i] = BODY == 1 ? a0[i] : fmaf(P1[NB == 1 ? i : 0], a1[i], P0[NB == 1 ? i : 0] * a0[i]);
          if (outs) put_row(outs + (int64_t)rw * p.ldo, p.D, dxv, true);
          if (PG) {
            float xr[NA];
#pragma unroll
            for (int jq = 0; jq < NQ; ++jq) {
              const float4 r4 = lds128f(slot_s + (uint32_t)(NQ + jq) * 512u);
              xr[4 * jq] = r4.x; xr[4 * jq + 1] = r4.y; xr[4 * jq + 2] = r4.z; xr[4 * jq + 3] = r4.w;
            }
            add_param_grads(xr);
          }
#pragma unroll
          for (int i = 0; i < NA; ++i) a0[i] = a1[i] = 0.f;
        }
        issue(t + j + RS, ibase + (uint32_t)j * 16u, vbase + (uint32_t)j * 4u, j);
        cp_async_commit();
      }
    }
    cp_async_wait<0>();
    __syncwarp();
    if (part_slot >= 0) {
      // hub segment: partial sums (row scale applied by hub_finalize_kernel); parameter gradients against the
      // hub row's own features, scaled here
      if (outs) {
        float dxv[NA];
#pragma unroll
        for (int i = 0; i < NA; ++i)
          dxv[i] = BODY == 1 ? a0[i] : fmaf(P1[NB == 1 ? i : 0], a1[i], P0[NB == 1 ? i : 0] * a0[i]);
        put_row(p.part_acc + ((int64_t)s * p.num_hub_segs + part_slot) * D8, D8, dxv, false);
      }
      if (PG && nedges > 0) {
        const float* xrow = p.xrow + (int64_t)s * p.xr_ss + (int64_t)hub_row * p.ldxr;
        const float rs = p.rscale ? __ldg(p.rscale + hub_row) : 1.0f;
        float xr[NA];
#pragma unroll
        for (int jq = 0; jq < NQ; ++jq) {
          float4 r4 = make_float4(0.f, 0.f, 0.f, 0.f);
          if (qv[jq]) r4 = __ldg(reinterpret_cast<const float4*>(xrow + c + 32 * jq));
          xr[4 * jq] = r4.x * rs; xr[4 * jq + 1] = r4.y * rs; xr[4 * jq + 2] = r4.z * rs; xr[4 * jq + 3] = r4.w * rs;
        }
        add_param_grads(xr);
      }
    }
  }
  zero_empty_rows_tail(p, (int64_t)blockIdx.x * AGG_WARPS + warp, total_warps, lane);
  if (!PG) return;

  // ---- parameter-gradient partials: groups of a warp -> warp slice -> CTA row of dp_partial -----------
  // (scalar parameters with NB = 2: the lane's single partial sits at its first channel, the finalize sums all)
  if (KIND == STAG_NOISE_NORMAL) {
#pragma unroll
    for (int i = 0; i < NP; ++i) d1[i] *= kRad;  // a1 was accumulated against eps / sqrt(2 ln 2)
  }
  for (int o = LPR; o < 32; o <<= 1) {
#pragma unroll
    for (int i = 0; i < NP; ++i) {
      d0[i] += __shfl_xor_sync(0xffffffffu, d0[i], o);
      d1[i] += __shfl_xor_sync(0xffffffffu, d1[i], o);
    }
  }
  float* my_stage = stage + (size_t)warp * 2 * D8;
  for (int i = lane; i < 2 * D8; i += 32) my_stage[i] = 0.f;
  __syncwarp();
  if (sub == 0) {
#pragma unroll
    for (int i = 0; i < NP; ++i) {
      const int ch = c + 32 * (i >> 2) + (i & 3);
      if (ch < D8) {
        my_stage[ch] = d0[i];
        my_stage[D8 + ch] = d1[i];
      }
    }
  }
  __syncthreads();
  float* dst = p.dp_partial + (size_t)blockIdx.x * 2 * D8;
  for (int i = threadIdx.x; i < 2 * D8; i += AGG_THREADS) {
    float v = 0.f;
#pragma unroll
    for (int w = 0; w < AGG_WARPS; ++w) v += stage[(size_t)w * 2 * D8 + i];
    dst[i] = v;
  }
}

template <int MODE, int KIND, int PSH, bool VEC, bool GRADS, bool FOLD>
__global__ void __launch_bounds__(AGG_THREADS, FOLD ? 3 : 1) agg_kernel(const AggParams p) {
  const PhiloxKey key = live_key(p);
  extern __shared__ float smem[];  // param grads: [AGG_WARPS][2][dpad]
  constexpr int U = GRADS ? 1 : 2;  // edges in flight per lane
  constexpr bool GEN = MODE == 2;
  // parameter gradients exist for generated Normal / Uniform noise only
  constexpr bool PGRADS_C = GRADS && GEN && (KIND == STAG_NOISE_NORMAL || KIND == STAG_NOISE_UNIFORM);
  const bool pgrads_e = GRADS && MODE == 0 && (p.kind == STAG_NOISE_NORMAL || p.kind == STAG_NOISE_UNIFORM);
  const bool dense_pg = (PGRADS_C || pgrads_e) && p.pshape <= STAG_PARAM_CHANNEL;  // reduced to [1] / [K]
  // FOLD (hot path: MODE 2 / PSH 0 without relu / in-norm / gradients): the gather scale is folded
  // into the per-edge parameters
  constexpr bool fold = FOLD;

  const int lane = threadIdx.x & 31;
  const int warp = threadIdx.x >> 5;
  const int LPR = 1 << p.lpr_log2;
  const int RPW = 32 >> p.lpr_log2;
  const int sub = lane >> p.lpr_log2;
  const int sl = lane & (LPR - 1);
  const int D8 = p.dpad;

  float* my_sm = nullptr;
  if (GRADS && dense_pg) {
    my_sm = smem + (size_t)warp * 2 * D8;
    for (int i = lane; i < 2 * D8; i += 32) my_sm[i] = 0.f;
    __syncwarp();
  }

  const int HG = (p.num_hub_segs + RPW - 1) / RPW;
  const int RG = (p.N + RPW - 1) / RPW;
  const int64_t per_sample = (int64_t)HG + RG;
  const int64_t total = per_sample * p.S * p.ncb;
  const int64_t total_warps = (int64_t)gridDim.x * AGG_WARPS;

  for (int64_t item = (int64_t)blockIdx.x * AGG_WARPS + warp; item < total; item += total_warps) {
    const int64_t outer = item / per_sample;
    const int r = (int)(item - outer * per_sample);
    int s, cb;
    if (p.cb_major) {
      cb = (int)(outer / p.S);
      s = (int)(outer - (int64_t)cb * p.S);
    } else {
      s = (int)(outer / p.ncb);
      cb = (int)(outer - (int64_t)s * p.ncb);
    }
    const int c_begin = cb * p.cw;
    const int c_end = min(c_begin + p.cw, D8);
    // resolve this lane-group's row and edge range
    int row = -1, beg = 0, len = 0, part_slot = -1;
    if (r < HG) {
      const int seg = r * RPW + sub;
      if (seg < p.num_hub_segs) {
        int lo = 0, hi = p.num_hubs;  // last hub with hub_seg_ptr[h] <= seg
        while (hi - lo > 1) {
          const int mid = (lo + hi) >> 1;
          if (__ldg(p.hub_seg_ptr + mid) <= seg) lo = mid; else hi = mid;
        }
        row = __ldg(p.hub_rows + lo);
        const int k = seg - __ldg(p.hub_seg_ptr + lo);
        const int rb = __ldg(p.indptr + row), re = __ldg(p.indptr + row + 1);
        beg = rb + k * kHubSegment;
        len = min(kHubSegment, re - beg);
        part_slot = seg;
      }
    } else {
      const int vi = (r - HG) * RPW + sub;
      if (vi < p.N) {
        const int v = p.row_order ? __ldg(p.row_order + vi) : vi;
        const int rb = __ldg(p.indptr + v), re = __ldg(p.indptr + v + 1);
        if (re - rb <= kHubThreshold) {
          row = v;
          beg = rb;
          len = re - rb;
        }
      }
    }
    int maxlen = len;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) maxlen = max(maxlen, __shfl_xor_sync(0xffffffffu, maxlen, o));
    if (!__any_sync(0xffffffffu, row >= 0)) continue;

    const float* xs = p.x + (int64_t)s * p.x_ss;
    const float rs = (row >= 0 && p.rscale) ? __ldg(p.rscale + row) : 1.0f;
    const uint32_t smp = (uint32_t)(p.sample_base + s);

    for (int c0 = c_begin; c0 < c_end; c0 += max(LPR * 8, 64)) {
      const int c = first_chan(c0, sl);
      const bool qvalid = c < p.D && c < c_end;
      const uint32_t oct = (uint32_t)((c0 >> 3) + sl);  // Philox block of this lane
      float P0[8], P1[8];
      if (GEN && PSH == 1) {
        load8<VEC>(p.p0, c, p.D, P0);
        if (KIND != STAG_NOISE_BERNOULLI) load8<VEC>(p.p1, c, p.D, P1);
      }
      float acc[8], wsum[8], xr[8], d0[8], d1[8];
#pragma unroll
      for (int i = 0; i < 8; ++i) acc[i] = wsum[i] = d0[i] = d1[i] = xr[i] = 0.f;
      float wsum_e = 0.f;  // MODE 0 in-norm: sum of the per-edge weights of this row
      float d0_e = 0.f, d1_e = 0.f;
      if (GRADS && row >= 0 && qvalid) {
        load8<VEC>(p.xrow + (int64_t)s * p.xr_ss + (int64_t)row * p.ldxr, c, p.D, xr);
#pragma unroll
        for (int i = 0; i < 8; ++i) xr[i] *= rs;
      }

      for (int off = 0; off < maxlen; off += LPR) {
        // ---- edge records of this batch: lane sl owns edge off + sl ---------------------------
        //   MODE 0        my_a = gather scale * weight, my_b = weight
        //   MODE 2 PSH 0  my_a / my_b = the two parameters (folded with the gather scale if `fold`)
        int my_idx = 0, my_eid = 0;
        float my_sc = 0.f, my_a = 0.f, my_b = 0.f, my_raw = 0.f, my_pre = 0.f;
        if (off + sl < len) {
          my_idx = __ldg(p.indices + beg + off + sl);
          my_eid = __ldg(p.eid + beg + off + sl);
          my_sc = p.gscale ? __ldg(p.gscale + my_idx) : 1.0f;
          if (MODE == 0) {
            float w = 1.0f;
            if (p.kind == STAG_NOISE_EXTERNAL) {
              w = __ldg(p.ext + (int64_t)s * p.E + my_eid);
              my_raw = w;
            } else if (p.kind >= STAG_NOISE_NORMAL) {
              const int64_t pi = p.pshape >= STAG_PARAM_EDGE ? my_eid : 0;
              const float a = __ldg(p.p0 + pi);
              const float b = p.p1 ? __ldg(p.p1 + pi) : 0.f;
              my_raw = raw_first(p.kind, (uint32_t)my_eid, smp, key);
              w = transform_rt(p.kind, my_raw, a, b);
            }
            my_pre = w;
            if (p.relu) w = fmaxf(w, 0.f);
            my_b = w;
            my_a = my_sc * w;
          } else if (GEN && PSH == 0) {
            const int64_t pi = p.pshape >= STAG_PARAM_EDGE ? my_eid : 0;
            const float a = __ldg(p.p0 + pi);
            const float b = KIND != STAG_NOISE_BERNOULLI ? __ldg(p.p1 + pi) : 0.f;
            if (fold) {
              if (KIND == STAG_NOISE_NORMAL) { my_a = my_sc * a; my_b = my_sc * b; }
              else if (KIND == STAG_NOISE_UNIFORM) { my_a = my_sc * a; my_b = my_sc * (b - a); }
              else { my_a = a; my_b = my_sc; }
            } else {
              my_a = a;
              my_b = b;
            }
          }
        }
        const int cnt = min(LPR, maxlen - off);
        for (int t0 = 0; t0 < cnt; t0 += U) {
          float xv[U][8];
          int ee[U];
          float sa[U], sb[U], ssc[U];
          bool act[U];
#pragma unroll
          for (int k = 0; k < U; ++k) {
            const int t = t0 + k;
            const int u = __shfl_sync(0xffffffffu, my_idx, t, LPR);
            ee[k] = __shfl_sync(0xffffffffu, my_eid, t, LPR);
            ssc[k] = __shfl_sync(0xffffffffu, my_sc, t, LPR);
            sa[k] = 0.f;
            sb[k] = 0.f;
            if (MODE == 0 || (GEN && PSH == 0)) {
              sa[k] = __shfl_sync(0xffffffffu, my_a, t, LPR);
              sb[k] = __shfl_sync(0xffffffffu, my_b, t, LPR);
            }
            act[k] = (t < LPR) && (off + t < len) && qvalid;
            if (act[k]) {
              load8<VEC>(xs + (int64_t)u * p.ldx, c, p.D, xv[k]);
            } else {
#pragma unroll
              for (int i = 0; i < 8; ++i) xv[k][i] = 0.f;
            }
          }
#pragma unroll
          for (int k = 0; k < U; ++k) {
            if (t0 + k >= cnt) break;  // warp-uniform
            const bool edge_ok = (t0 + k < LPR) && (off + t0 + k < len);
            if (MODE == 0) {
              // -------- per-edge weight ------------------------------------------------------
              if (!GRADS) {
#pragma unroll
                for (int i = 0; i < 8; ++i) acc[i] = fmaf(xv[k][i], sa[k], acc[i]);
                if (edge_ok) wsum_e += sb[k];
              } else {
                float dwc[8];
#pragma unroll
                for (int i = 0; i < 8; ++i) {
                  const float g = xv[k][i] * ssc[k];
                  acc[i] = fmaf(sb[k], g, acc[i]);
                  dwc[i] = xr[i] * g;
                }
                if (p.kind != STAG_NOISE_NONE && (p.dw_ext || pgrads_e)) {
                  const float tot = group_sum(sum8(dwc), LPR);
                  const float raw = __shfl_sync(0xffffffffu, my_raw, t0 + k, LPR);
                  const float pre = __shfl_sync(0xffffffffu, my_pre, t0 + k, LPR);
                  if (sl == 0 && edge_ok) {
                    if (p.kind == STAG_NOISE_EXTERNAL) {
                      if (p.dw_ext) {
                        float* base = p.dw_ext + (int64_t)s * p.E;
                        // several channel chunks accumulate into the same slot, from the same thread
                        if (c0 == c_begin) base[ee[k]] = tot; else base[ee[k]] += tot;
                      }
                    } else if (pgrads_e) {
                      const float e = (p.relu && !(pre > 0.f)) ? 0.f : tot;
                      const float e1 = e * raw;
                      const float e0 = p.kind == STAG_NOISE_NORMAL ? e : e - e1;
                      if (p.pshape <= STAG_PARAM_CHANNEL) {
                        d0_e += e0;
                        d1_e += e1;
                      } else {
                        p.dp0[ee[k]] += e0;
                        p.dp1[ee[k]] += e1;
                      }
                    }
                  }
                }
              }
            } else if (fold) {
              // -------- generated per-channel noise, hot path ------------------------------------
              float w[8];
              folded_oct<KIND>((uint32_t)ee[k], oct, smp, key, sa[k], sb[k], w);
#pragma unroll
              for (int i = 0; i < 8; ++i) acc[i] = fmaf(w[i], xv[k][i], acc[i]);
            } else {
              // -------- per-channel weights, general path -----------------------------------------
              float w[8], raw[8], pre[8];
              if (MODE == 1) {
                if (act[k]) {
                  load8<VEC>(p.ext + ((int64_t)s * p.E + ee[k]) * p.K, c, p.K, w);
                } else {
#pragma unroll
                  for (int i = 0; i < 8; ++i) w[i] = 0.f;
                }
#pragma unroll
                for (int i = 0; i < 8; ++i) pre[i] = raw[i] = w[i];
              } else {
                raw_oct<KIND>((uint32_t)ee[k], oct, smp, key, raw);
                if (PSH == 0) {
#pragma unroll
                  for (int i = 0; i < 8; ++i) w[i] = transform<KIND>(raw[i], sa[k], sb[k]);
                } else if (PSH == 1) {
#pragma unroll
                  for (int i = 0; i < 8; ++i) w[i] = transform<KIND>(raw[i], P0[i], P1[i]);
                } else {
                  float a[8], b[8];
                  if (act[k]) {
                    load8<VEC>(p.p0 + (int64_t)ee[k] * p.K, c, p.K, a);
                    if (KIND != STAG_NOISE_BERNOULLI) load8<VEC>(p.p1 + (int64_t)ee[k] * p.K, c, p.K, b);
                  } else {
#pragma unroll
                    for (int i = 0; i < 8; ++i) a[i] = b[i] = 0.f;
                  }
#pragma unroll
                  for (int i = 0; i < 8; ++i) w[i] = transform<KIND>(raw[i], a[i], b[i]);
                }
#pragma unroll
                for (int i = 0; i < 8; ++i) pre[i] = w[i];
              }
              if (p.relu) {
#pragma unroll
                for (int i = 0; i < 8; ++i) w[i] = fmaxf(w[i], 0.f);
              }
              float g[8];
#pragma unroll
              for (int i = 0; i < 8; ++i) {
                g[i] = xv[k][i] * ssc[k];
                acc[i] = fmaf(w[i], g[i], acc[i]);
              }
              if (!GRADS) {
                if (p.in_norm && act[k]) {
#pragma unroll
                  for (int i = 0; i < 8; ++i) wsum[i] += w[i];
                }
              } else {
                float dw[8];
#pragma unroll
                for (int i = 0; i < 8; ++i) dw[i] = xr[i] * g[i];
                if (MODE == 1) {
                  if (p.dw_ext && act[k])
                    store8<VEC, false>(p.dw_ext + ((int64_t)s * p.E + ee[k]) * p.K, c, p.K, dw);
                } else if (PGRADS_C) {
                  float e0[8], e1[8];
#pragma unroll
                  for (int i = 0; i < 8; ++i) {
                    const float e = (p.relu && !(pre[i] > 0.f)) ? 0.f : dw[i];
                    e1[i] = e * raw[i];
                    e0[i] = KIND == STAG_NOISE_NORMAL ? e : e - e1[i];
                  }
                  if (p.pshape <= STAG_PARAM_CHANNEL) {
#pragma unroll
                    for (int i = 0; i < 8; ++i) {
                      d0[i] += e0[i];
                      d1[i] += e1[i];
                    }
                  } else if (p.pshape == STAG_PARAM_EDGE) {
                    const float t0s = group_sum(sum8(e0), LPR);
                    const float t1s = group_sum(sum8(e1), LPR);
                    if (sl == 0 && edge_ok) {
                      p.dp0[ee[k]] += t0s;
                      p.dp1[ee[k]] += t1s;
                    }
                  } else if (act[k]) {
                    float* q0 = p.dp0 + (int64_t)ee[k] * p.K;
                    float* q1 = p.dp1 + (int64_t)ee[k] * p.K;
                    float o0[8], o1[8];
                    load8<VEC>(q0, c, p.K, o0);
                    load8<VEC>(q1, c, p.K, o1);
#pragma unroll
                    for (int i = 0; i < 8; ++i) {
                      o0[i] += e0[i];
                      o1[i] += e1[i];
                    }
                    store8<VEC, false>(q0, c, p.K, o0);
                    store8<VEC, false>(q1, c, p.K, o1);
                  }
                }
              }
            }
          }
        }
      }

      // ---- epilogue of this channel chunk --------------------------------------------------------
      if (MODE == 0) {
#pragma unroll
        for (int i = 0; i < 8; ++i) wsum[i] = wsum_e;
      }
      if (row >= 0 && qvalid) {
        if (part_slot >= 0) {
          if (p.out) {
            const int64_t o = ((int64_t)s * p.num_hub_segs + part_slot) * D8;
            store8<true, false>(p.part_acc + o, c, D8, acc);
            if (!GRADS && p.in_norm) store8<true, false>(p.part_w + o, c, D8, wsum);
          }
        } else if (p.out) {
          if (!GRADS && p.in_norm) {
            const float indeg = (float)len;
            float sc8[8];
#pragma unroll
            for (int i = 0; i < 8; ++i) {
              sc8[i] = wsum[i] != 0.f ? indeg / wsum[i] : 1.f;
              acc[i] *= sc8[i];
            }
            if (p.norm_scale_out) {
              float* ns = p.norm_scale_out + ((int64_t)s * p.N + row) * p.K;
              if (p.K == 1) {
                if (c == 0) ns[0] = sc8[0];
              } else {
                store8<VEC, false>(ns, c, p.K, sc8);
              }
            }
          }
#pragma unroll
          for (int i = 0; i < 8; ++i) acc[i] *= rs;
          store8<VEC, true>(p.out + (int64_t)s * p.out_ss + (int64_t)row * p.ldo, c, p.D, acc);
        }
      }
      if (GRADS && dense_pg) {
        if (MODE == 0) {
          // scalar parameter, per-edge noise: lane sl == 0 of each group holds this chunk's totals
          float a = sl == 0 ? d0_e : 0.f, b = sl == 0 ? d1_e : 0.f;
#pragma unroll
          for (int o = 16; o > 0; o >>= 1) {
            a += __shfl_xor_sync(0xffffffffu, a, o);
            b += __shfl_xor_sync(0xffffffffu, b, o);
          }
          if (lane == 0) {
            my_sm[0] += a;
            my_sm[D8] += b;
          }
        } else {
          // fold the row groups of this warp, then add into the warp's shared slice
          for (int o = LPR; o < 32; o <<= 1) {
#pragma unroll
            for (int i = 0; i < 8; ++i) {
              d0[i] += __shfl_xor_sync(0xffffffffu, d0[i], o);
              d1[i] += __shfl_xor_sync(0xffffffffu, d1[i], o);
            }
          }
          if (sub == 0 && c < D8) {
#pragma unroll
            for (int i = 0; i < 8; ++i) {
              my_sm[chan(c, i)] += d0[i];
              my_sm[D8 + chan(c, i)] += d1[i];
            }
          }
        }
        __syncwarp();
      }
    }
  }

  if (GRADS && dense_pg) {
    __syncthreads();
    float* dst = p.dp_partial + (size_t)blockIdx.x * 2 * D8;
    for (int i = threadIdx.x; i < 2 * D8; i += AGG_THREADS) {
      float v = 0.f;
#pragma unroll
      for (int w = 0; w < AGG_WARPS; ++w) v += smem[(size_t)w * 2 * D8 + i];
      dst[i] = v;
    }
  }
}

// Combine the partial sums of hub rows in segment order and finish the row.
__global__ void hub_finalize_kernel(const AggParams p, int grads) {
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int D8 = p.dpad;
  const int64_t total = (int64_t)p.S * p.num_hubs * p.D;
  if (idx >= total) return;
  const int c = (int)(idx % p.D);
  const int h = (int)((idx / p.D) % p.num_hubs);
  const int s = (int)(idx / ((int64_t)p.D * p.num_hubs));
  const int row = p.hub_rows[h];
  const int s0 = p.hub_seg_ptr[h], s1 = p.hub_seg_ptr[h + 1];
  float acc = 0.f, wsum = 0.f;
  for (int seg = s0; seg < s1; seg += 8) {  // 8 loads in flight, summed in segment order
    float v[8], w[8];
#pragma unroll
    for (int k = 0; k < 8; ++k) {
      const int64_t o = ((int64_t)s * p.num_hub_segs + seg + k) * D8 + c;
      v[k] = seg + k < s1 ? p.part_acc[o] : 0.f;
      w[k] = (!grads && p.in_norm && seg + k < s1) ? p.part_w[o] : 0.f;
    }
#pragma unroll
    for (int k = 0; k < 8; ++k) {
      acc += v[k];
      wsum += w[k];
    }
  }
  if (!grads && p.in_norm) {
    const float indeg = (float)(p.indptr[row + 1] - p.indptr[row]);
    const float sc = wsum != 0.f ? indeg / wsum : 1.f;
    acc *= sc;
    if (p.norm_scale_out && (p.K != 1 || c == 0))
      p.norm_scale_out[((int64_t)s * p.N + row) * p.K + (p.K == 1 ? 0 : c)] = sc;
  }
  if (p.rscale) acc *= p.rscale[row];
  if (p.out) p.out[(int64_t)s * p.out_ss + (int64_t)row * p.ldo + c] = acc;
}

// Per-edge parameter gradients (EDGE / EDGE_CHANNEL shapes: the [E,1] / [E,K] outputs of AmortizedDistribution,
// stag/distributions.py:221-242) for any number of samples in one launch.  Edge-parallel: half a warp owns one stored
// edge, a lane one Philox block (8 channels) of it at a time; it reads the source row x[u] and the upstream row
// dout[v], regenerates the raw variates of (edge, sample) and reduces
//     dw[s,e,c] = (src_scale[u] x[s,u,c]) (dst_scale[v] dout[s,v,c])          (the SDDMM term, never stored)
//     NORMAL : d p0 += dw, d p1 += dw eps        UNIFORM: d p0 += dw (1 - u), d p1 += dw u        (relu: dw masked)
// over the samples (and, for the EDGE shape, over the channels: 4 shuffle steps).  One writer per edge, fixed
// summation order: deterministic.  Results ACCUMULATE into dp0 / dp1 (the caller zeroes them once).
// p holds the transposed roles of stag_spmm_bwd: p.x = dout (gscale = dst_scale), p.xrow = x (rscale = src_scale).
template <int KIND, bool VEC>
__global__ void __launch_bounds__(256) edge_param_grads_kernel(const AggParams p) {
  const PhiloxKey key = live_key(p);
  const int lane = threadIdx.x & 31, hl = lane & 15;
  const int64_t nhw = (int64_t)gridDim.x * (blockDim.x >> 4);
  const int64_t hw0 = (int64_t)blockIdx.x * (blockDim.x >> 4) + (threadIdx.x >> 4);
  const int64_t trips = (p.E + nhw - 1) / nhw;  // both halves of a warp make the same number of trips (shuffles below)
  const int nblk = p.nblk;
  for (int64_t it = 0; it < trips; ++it) {
    const int64_t j = hw0 + it * nhw;
    const bool on = j < p.E;
    const int u = on ? __ldg(p.erow + j) : 0;
    const int v = on ? __ldg(p.indices + j) : 0;
    const int e = on ? __ldg(p.eid + j) : 0;
    float sc = p.gscale ? __ldg(p.gscale + v) : 1.0f;
    if (p.rscale) sc *= __ldg(p.rscale + u);
    const bool per_channel = p.pshape == STAG_PARAM_EDGE_CHANNEL;
    const float P0 = (on && !per_channel) ? __ldg(p.p0 + e) : 0.f;
    const float P1 = (on && !per_channel) ? __ldg(p.p1 + e) : 0.f;
    float t0 = 0.f, t1 = 0.f;
    if (on) {
      for (int b = hl; b < nblk; b += 16) {
        const int c = first_chan(0, b);
        float d0[8], d1[8], pa[8], pb[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          d0[i] = d1[i] = 0.f;
          const int ch = chan(c, i);
          pa[i] = per_channel ? (ch < p.D ? __ldg(p.p0 + (int64_t)e * p.K + ch) : 0.f) : P0;
          pb[i] = per_channel ? (ch < p.D ? __ldg(p.p1 + (int64_t)e * p.K + ch) : 0.f) : P1;
        }
        // the rows of sample s + 1 are requested before sample s is worked on
        const float* xrp = p.xrow + (int64_t)u * p.ldxr;
        const float* gvp = p.x + (int64_t)v * p.ldx;
        float xn[8], gn[8];
        load8<VEC>(xrp, c, p.D, xn);
        load8<VEC>(gvp, c, p.D, gn);
        for (int s = 0; s < p.S; ++s) {
          float xr[8], gv[8], raw[8];
#pragma unroll
          for (int i = 0; i < 8; ++i) { xr[i] = xn[i]; gv[i] = gn[i]; }
          if (s + 1 < p.S) {
            load8<VEC>(xrp + (int64_t)(s + 1) * p.xr_ss, c, p.D, xn);
            load8<VEC>(gvp + (int64_t)(s + 1) * p.x_ss, c, p.D, gn);
          }
          const uint32_t smp = (uint32_t)(p.sample_base + s);
          if (p.K == 1) {
            const float r1 = raw_first(KIND, (uint32_t)e, smp, key);
#pragma unroll
            for (int i = 0; i < 8; ++i) raw[i] = r1;
          } else {
            raw_oct<KIND>((uint32_t)e, (uint32_t)b, smp, key, raw);
          }
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            float dw = xr[i] * gv[i] * sc;  // zero beyond D (load8 pads)
            if (p.relu && !(transform<KIND>(raw[i], pa[i], pb[i]) > 0.f)) dw = 0.f;
            const float e1 = dw * raw[i];
            d1[i] += e1;
            d0[i] += KIND == STAG_NOISE_NORMAL ? dw : dw - e1;
          }
        }
        if (per_channel) {
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            const int ch = chan(c, i);
            if (ch < p.D) {
              p.dp0[(int64_t)e * p.K + ch] += d0[i];
              p.dp1[(int64_t)e * p.K + ch] += d1[i];
            }
          }
        } else {
          t0 += sum8(d0);
          t1 += sum8(d1);
        }
      }
    }
    if (!per_channel) {
#pragma unroll
      for (int o = 8; o > 0; o >>= 1) {
        t0 += __shfl_xor_sync(0xffffffffu, t0, o);
        t1 += __shfl_xor_sync(0xffffffffu, t1, o);
      }
      if (on && hl == 0) {
        p.dp0[e] += t0;
        p.dp1[e] += t1;
      }
    }
  }
}

// The common amortised case on the generator code of the hot kernel: Normal noise, [E,1] parameters (the `re`
// posteriors of scripts/arxiv_rec: AmortizedDistribution(in_features, 1)), no relu, K == D made of whole 128-channel
// groups, 128-bit rows.  8 lanes own one stored edge; a lane owns 16 channels of it (Philox blocks sl and sl + 8 of
// every group: the quads at c, c + 32, c + 64, c + 96 of agg_stream_kernel<NB = 2>), round keys from the constant bank,
// Box-Muller on packed FFMA2 / FMUL2:
//     d loc[e] += sc sum_{s,c} x g        d scale[e] += sc sum_{s,c} x g eps
// (eps = sqrt(2 ln 2) sqrt(-lg2 u1) cos / sin, the same variates as the forward).  4.8 ms -> see profiles/r02_modes.txt.
__global__ void __launch_bounds__(256) edge_param_grads_fast_kernel(const AggParams p) {
  const PhiloxKey key = live_key(p);
  const int lane = threadIdx.x & 31, sl = lane & 7;
  const int64_t ngr = (int64_t)gridDim.x * (blockDim.x >> 3);
  const int64_t g0 = (int64_t)blockIdx.x * (blockDim.x >> 3) + (threadIdx.x >> 3);
  const int64_t trips = (p.E + ngr - 1) / ngr;  // every group of a warp makes the same number of trips (shuffles below)
  const int G = p.D >> 7;
  const uint32_t kf = p.kf;
  for (int64_t it = 0; it < trips; ++it) {
    const int64_t j = g0 + it * ngr;
    const bool on = j < p.E;
    const int u = on ? __ldg(p.erow + j) : 0;
    const int v = on ? __ldg(p.indices + j) : 0;
    const uint32_t e = on ? (uint32_t)__ldg(p.eid + j) : 0u;
    float2 t0 = make_float2(0.f, 0.f), t1 = make_float2(0.f, 0.f);
    if (on) {
      for (int g = 0; g < G; ++g) {
        const float* xrp = p.xrow + (int64_t)u * p.ldxr + 128 * g + 4 * sl;
        const float* gvp = p.x + (int64_t)v * p.ldx + 128 * g + 4 * sl;
        float4 xn[4], gn[4];
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          xn[q] = __ldg(reinterpret_cast<const float4*>(xrp + 32 * q));
          gn[q] = __ldg(reinterpret_cast<const float4*>(gvp + 32 * q));
        }
        // samples innermost, the two rows of sample s + 1 requested before sample s is worked on (samples outermost,
        // one [N,D] operand pair resident in L2 at a time, measured slower: 2.6 - 3.0 against 1.9 ms)
        for (int s = 0; s < p.S; ++s) {
          float2 d[8];  // x g of this lane's 16 channels, as pairs
#pragma unroll
          for (int q = 0; q < 4; ++q) {
            d[2 * q] = __fmul2_rn(make_float2(xn[q].x, xn[q].y), make_float2(gn[q].x, gn[q].y));
            d[2 * q + 1] = __fmul2_rn(make_float2(xn[q].z, xn[q].w), make_float2(gn[q].z, gn[q].w));
          }
          if (s + 1 < p.S) {
#pragma unroll
            for (int q = 0; q < 4; ++q) {
              xn[q] = __ldg(reinterpret_cast<const float4*>(xrp + (int64_t)(s + 1) * p.xr_ss + 32 * q));
              gn[q] = __ldg(reinterpret_cast<const float4*>(gvp + (int64_t)(s + 1) * p.x_ss + 32 * q));
            }
          }
          const uint32_t smp = (uint32_t)(p.sample_base + s);
#pragma unroll
          for (int b = 0; b < 2; ++b) {
            // block 16 g + sl + 8 b: channels 64 b + 4 sl + {0..3} (slots 0..3) and 64 b + 32 + 4 sl + {0..3} (slots 4..7)
            const uint4 r4 = philox_rk((uint32_t)(16 * g + sl + 8 * b), e, smp, key.c3, p);
            const uint32_t w4[4] = {r4.x, r4.y, r4.z, r4.w};
#pragma unroll
            for (int ip = 0; ip < 2; ++ip) {
              const uint32_t qa = w4[2 * ip], qb = w4[2 * ip + 1];
              const float2 xl = make_float2(__uint_as_float(__byte_perm(qa, kf, 0x7610)), __uint_as_float(__byte_perm(qb, kf, 0x7610)));
              const float2 xh = make_float2(__uint_as_float(__byte_perm(qa, kf, 0x7632)), __uint_as_float(__byte_perm(qb, kf, 0x7632)));
              const float2 u1 = __ffma2_rn(xl, make_float2(1.52587890625e-05f, 1.52587890625e-05f),
                                           make_float2(-127.99999237060547f, -127.99999237060547f));
              const float2 ang = __ffma2_rn(xh, make_float2(9.58738019107841e-05f, 9.58738019107841e-05f),
                                            make_float2(-804.2476806640625f, -804.2476806640625f));
              const float ra = mufu_sqrt(-mufu_lg2(u1.x)), rb = mufu_sqrt(-mufu_lg2(u1.y));
              // slots 4 ip + {0, 1} (word qa) and 4 ip + {2, 3} (word qb) of the block -> pairs d[4 b + 2 ip], d[4 b + 2 ip + 1]
              const float2 za = __fmul2_rn(make_float2(mufu_cos(ang.x), mufu_sin(ang.x)), make_float2(ra, ra));
              const float2 zb = __fmul2_rn(make_float2(mufu_cos(ang.y), mufu_sin(ang.y)), make_float2(rb, rb));
              const float2 da = d[4 * b + 2 * ip], db = d[4 * b + 2 * ip + 1];
              t0 = __fadd2_rn(t0, __fadd2_rn(da, db));
              t1 = __ffma2_rn(da, za, t1);
              t1 = __ffma2_rn(db, zb, t1);
            }
          }
        }
      }
    }
    float a0 = t0.x + t0.y, a1 = t1.x + t1.y;
#pragma unroll
    for (int o = 4; o > 0; o >>= 1) {
      a0 += __shfl_xor_sync(0xffffffffu, a0, o);
      a1 += __shfl_xor_sync(0xffffffffu, a1, o);
    }
    if (on && sl == 0) {
      float sc = p.gscale ? __ldg(p.gscale + v) : 1.0f;
      if (p.rscale) sc *= __ldg(p.rscale + u);
      p.dp0[e] += sc * a0;
      p.dp1[e] += sc * a1 * 1.1774100225154747f;  // sqrt(2 ln 2): the radius above is sqrt(-lg2 u1)
    }
  }
}

// noise materialisation (compat path + RNG tests): w[s,e,c]
template <int KIND>
__global__ void emit_kernel(const AggParams p, float* __restrict__ w_out, float* __restrict__ eps_out) {
  const PhiloxKey key = live_key(p);
  const int nblk = p.nblk;
  const int64_t total = (int64_t)p.S * p.E * nblk;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total;
       i += (int64_t)gridDim.x * blockDim.x) {
    const int q = (int)(i % nblk);
    const int64_t e = (i / nblk) % p.E;
    const int s = (int)(i / ((int64_t)nblk * p.E));
    const int c = first_chan(0, q);
    float raw[8];
    raw_oct<KIND>((uint32_t)e, (uint32_t)q, (uint32_t)(p.sample_base + s), key, raw);
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const int ch = chan(c, j);
      if (ch < p.K) {
        int64_t pi;
        switch (p.pshape) {
          case STAG_PARAM_SCALAR: pi = 0; break;
          case STAG_PARAM_CHANNEL: pi = ch; break;
          case STAG_PARAM_EDGE: pi = e; break;
          default: pi = e * p.K + ch; break;
        }
        float w = transform<KIND>(raw[j], p.p0[pi], p.p1 ? p.p1[pi] : 0.f);
        if (p.relu) w = fmaxf(w, 0.f);
        const int64_t o = ((int64_t)s * p.E + e) * p.K + ch;
        w_out[o] = w;
        if (eps_out) eps_out[o] = raw[j];
      }
    }
  }
}

__global__ void segment_reduce_kernel(const float* __restrict__ feat, int64_t ldf, const int32_t* __restrict__ ptr,
                                      int B, int D, int mean, float* __restrict__ out, int64_t ldo) {
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= (int64_t)B * D) return;
  const int c = (int)(idx % D);
  const int b = (int)(idx / D);
  const int n0 = ptr[b], n1 = ptr[b + 1];
  float acc = 0.f;
  for (int n = n0; n < n1; ++n) acc += feat[(int64_t)n * ldf + c];
  if (mean) acc /= (float)max(n1 - n0, 1);
  out[(int64_t)b * ldo + c] = acc;
}

// noise materialisation of STAG_NOISE_NORMAL_HADAMARD: one warp per (sample, edge, 128-channel group)
__global__ void emit_wh_kernel(const AggParams p, float* __restrict__ w_out, float* __restrict__ eps_out) {
  const PhiloxKey key = live_key(p);
  const int lane = threadIdx.x & 31;
  const int G = p.K >> 7;
  const int64_t total = (int64_t)p.S * p.E * G;
  const int64_t nwarps = (int64_t)gridDim.x * (blockDim.x >> 5);
  for (int64_t i = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); i < total; i += nwarps) {
    const int g = (int)(i % G);
    const int64_t e = (i / G) % p.E;
    const int s = (int)(i / ((int64_t)G * p.E));
    float v[4];
    wh_group_sums((uint32_t)e, (uint32_t)g, (uint32_t)(p.sample_base + s), key, lane, v);
    const int ch = 128 * g + 4 * lane;
    float w[4], z[4];
#pragma unroll
    for (int b = 0; b < 4; ++b) {
      int64_t pi;
      switch (p.pshape) {
        case STAG_PARAM_SCALAR: pi = 0; break;
        case STAG_PARAM_CHANNEL: pi = ch + b; break;
        case STAG_PARAM_EDGE: pi = e; break;
        default: pi = e * p.K + ch + b; break;
      }
      z[b] = v[b] * kWhInvSd;
      // the fused kernel evaluates w = loc + (scale * kWhInvSd) * sum with the constant folded into the edge record
      w[b] = fmaf(v[b], p.p1[pi] * kWhInvSd, p.p0[pi]);
      if (p.relu) w[b] = fmaxf(w[b], 0.f);
    }
    const int64_t o = ((int64_t)s * p.E + e) * p.K + ch;
#pragma unroll
    for (int b = 0; b < 4; ++b) {
      w_out[o + b] = w[b];
      if (eps_out) eps_out[o + b] = z[b];
    }
  }
}

}  // namespace stag
#include "spmm_tc.cuh"
#include "spmm_wq.cuh"
#include "noise_kl.cuh"
namespace stag {

// Philox blocks needed by `width` channels: 8 per whole 64-channel group, one per started quad of
// the first half of the last group
static int blocks_for(int width) {
  const int rem = width % 64;
  const int last = (rem + 3) / 4;
  return 8 * (width / 64) + (last < 8 ? last : 8);
}

static int lpr_log2_for(int nblk) {
  int l = 0;
  while ((1 << l) < nblk && l < 5) ++l;
  return l;
}

struct WsLayout {
  size_t part_acc, part_w, dp_partial, rec, total;
};

static WsLayout ws_layout(const StagGraph* g, int D, int S, int grid_max) {
  WsLayout L;
  const size_t D8 = (size_t)((D + 63) / 64) * 64;
  size_t off = 0;
  L.part_acc = off;
  off += align_up((size_t)S * g->num_hub_segs * D8 * 4 + 16, 256);
  L.part_w = off;
  off += align_up((size_t)S * g->num_hub_segs * D8 * 4 + 16, 256);
  L.dp_partial = off;
  off += align_up((size_t)grid_max * 2 * D8 * 4 + 16, 256);
  L.rec = off;
  off += align_up((size_t)g->num_edges * 16 + 16, 256);
  L.total = off;
  return L;
}

static int grid_cap() { return num_sms() * 8; }

static bool aligned16(const void* p) { return ((uintptr_t)p & 15) == 0; }

static int check_noise(const StagNoise* n, int D, int64_t E, const char* who) {
  STAG_CHECK_ARG(n != nullptr, "%s: null noise spec", who);
  STAG_CHECK_ARG(n->kind >= STAG_NOISE_NONE && n->kind <= STAG_NOISE_NORMAL_HADAMARD, "%s: bad noise kind %d", who, n->kind);
  if (n->kind == STAG_NOISE_NONE) return STAG_OK;
  STAG_CHECK_ARG(n->K == 1 || n->K == D, "%s: noise width K=%d must be 1 or D=%d", who, n->K, D);
  if (n->kind == STAG_NOISE_EXTERNAL) {
    STAG_CHECK_ARG(n->external != nullptr || E == 0, "%s: EXTERNAL noise needs a tensor", who);
    return STAG_OK;
  }
  STAG_CHECK_ARG(n->param_shape >= STAG_PARAM_SCALAR && n->param_shape <= STAG_PARAM_EDGE_CHANNEL,
                 "%s: bad param_shape %d", who, n->param_shape);
  const bool per_edge = n->param_shape >= STAG_PARAM_EDGE;
  STAG_CHECK_ARG(n->p0 != nullptr || (per_edge && E == 0), "%s: null parameter p0", who);
  STAG_CHECK_ARG(n->kind == STAG_NOISE_BERNOULLI || n->p1 != nullptr || (per_edge && E == 0),
                 "%s: null parameter p1", who);
  if (n->kind == STAG_NOISE_NORMAL_HADAMARD)
    STAG_CHECK_ARG(n->K % 128 == 0, "%s: the Hadamard generator needs K %% 128 == 0 (K=%d)", who, n->K);
  return STAG_OK;
}

template <int MODE, int KIND, int PSH, bool GRADS, bool FOLD = false>
static int launch_vec(const AggParams& p, bool vec, int grid, size_t smem, cudaStream_t stream) {
  if (vec) {
    if (smem > 48 * 1024)
      STAG_CUDA(cudaFuncSetAttribute(agg_kernel<MODE, KIND, PSH, true, GRADS, FOLD>,
                                     cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    agg_kernel<MODE, KIND, PSH, true, GRADS, FOLD><<<grid, AGG_THREADS, smem, stream>>>(p);
  } else {
    if (smem > 48 * 1024)
      STAG_CUDA(cudaFuncSetAttribute(agg_kernel<MODE, KIND, PSH, false, GRADS, FOLD>,
                                     cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    agg_kernel<MODE, KIND, PSH, false, GRADS, FOLD><<<grid, AGG_THREADS, smem, stream>>>(p);
  }
  STAG_LAUNCH_CHECK();
  return STAG_OK;
}

// Launch of the streaming hot kernel (records, empty rows, kernel) for one instantiation.
template <int KIND, int NB, bool FULL, bool INNORM>
static int launch_stream_inst(const AggParams& q, cudaStream_t stream) {
  const int RPW = 32 >> q.lpr_log2;
  const int64_t witems = (int64_t)((q.num_hub_segs + q.num_items + RPW - 1) / RPW) * q.S * q.ncb;
  const int64_t nctas = (witems + S3_WARPS - 1) / S3_WARPS;
  const int64_t cap = (int64_t)num_sms() * s3_min_blocks(NB, INNORM);
  const int grid = (int)(nctas < 1 ? 1 : (nctas < cap ? nctas : cap));
  const size_t smem = (size_t)S3_WARPS * s3_warp_bytes(NB);
  STAG_CHECK_ARG(witems < (1ll << 30), "stag_spmm: too many work items for one launch");
  if (q.E > 0) {   // also zeroes the work queue behind the records
    edge_record_kernel<KIND><<<(unsigned)((q.E + 255) / 256), 256, 0, stream>>>(q, const_cast<int4*>(q.rec), 2);
    STAG_LAUNCH_CHECK();
  } else {
    STAG_CUDA(cudaMemsetAsync(const_cast<int4*>(q.rec), 0, 16, stream));
  }
  STAG_CUDA(cudaFuncSetAttribute(agg_stream_kernel<KIND, NB, FULL, INNORM>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                 (int)smem));
  agg_stream_kernel<KIND, NB, FULL, INNORM><<<grid, S3_THREADS, smem, stream>>>(q);
  STAG_LAUNCH_CHECK();
  return STAG_OK;
}

// NB = 2 (16 channels per lane) when the rows are made of 128-channel groups, else NB = 1.
template <int KIND, bool INNORM>
static int launch_stream(const AggParams& p, cudaStream_t stream) {
  AggParams q = p;
  const int width = p.D < p.cw ? p.D : p.cw;
  const bool nb2 = p.dpad % 128 == 0 && p.cw % 128 == 0;
  const int nb = nb2 ? 2 : 1;
  q.lpr_log2 = lpr_log2_for((blocks_for(width) + nb - 1) / nb);
  if (q.lpr_log2 < 3) q.lpr_log2 = 3;  // a group of 8 lanes owns one 64 NB-channel group
  // FULL (no quad predicates): one column block and every lane of every pass over the channels owns real ones
  const int pass = (1 << q.lpr_log2) / 8 * 64 * nb;
  const bool full = p.D % pass == 0 && p.ncb == 1 && p.cw == p.dpad;
  if (nb2) return full ? launch_stream_inst<KIND, 2, true, INNORM>(q, stream) : launch_stream_inst<KIND, 2, false, INNORM>(q, stream);
  return full ? launch_stream_inst<KIND, 1, true, INNORM>(q, stream) : launch_stream_inst<KIND, 1, false, INNORM>(q, stream);
}

template <int KIND, bool GRADS>
static int launch_psh(int psh, const AggParams& p, bool vec, int grid, size_t smem, cudaStream_t stream) {
  // streaming hot kernel: 128-bit rows, row offsets of the gathered operand fit 32 bits
  const bool stream_ok = !GRADS && psh == 0 && !p.relu && vec && p.items && p.erow && p.eidf && p.rec &&
                         p.ncols * p.ldx < (1ll << 31);
  if (stream_ok && p.in_norm && KIND == STAG_NOISE_BERNOULLI && (p.norm_scale_out == nullptr || p.K == p.D))
    return launch_stream<STAG_NOISE_BERNOULLI, true>(p, stream);
  if (stream_ok && !p.in_norm) return launch_stream<KIND, false>(p, stream);
  if (!GRADS && psh == 0 && !p.relu && !p.in_norm) return launch_vec<2, KIND, 0, false, true>(p, vec, grid, smem, stream);
  switch (psh) {
    case 0: return launch_vec<2, KIND, 0, GRADS>(p, vec, grid, smem, stream);
    case 1: return launch_vec<2, KIND, 1, GRADS>(p, vec, grid, smem, stream);
    default: return launch_vec<2, KIND, 2, GRADS>(p, vec, grid, smem, stream);
  }
}

// forward (or dX-only) launches of the two-sum / per-edge-weight streaming kernel
template <int KIND, int BODY, int NB>
static int launch_stream2_inst(const AggParams& p, cudaStream_t stream) {
  const int RPW = 32 >> p.lpr_log2;
  const int64_t warp_items = (int64_t)((p.num_hub_segs + p.num_items + RPW - 1) / RPW) * p.S;
  const int64_t ctas = (warp_items + AGG_WARPS - 1) / AGG_WARPS;
  const int sgrid = (int)(ctas < 1 ? 1 : (ctas < num_sms() * 2 ? ctas : num_sms() * 2));
  const size_t ring_bytes = (size_t)AGG_WARPS * s2_warp_bytes(false, NB);
  if (p.E > 0) {
    edge_record_kernel<STAG_NOISE_NORMAL><<<(unsigned)((p.E + 255) / 256), 256, 0, stream>>>(
        p, const_cast<int4*>(p.rec), 1);
    STAG_LAUNCH_CHECK();
  }
  STAG_CUDA(cudaFuncSetAttribute(agg_stream_grads_kernel<KIND, BODY, false, NB>,
                                 cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ring_bytes));
  agg_stream_grads_kernel<KIND, BODY, false, NB><<<sgrid, AGG_THREADS, ring_bytes, stream>>>(p);
  STAG_LAUNCH_CHECK();
  return STAG_OK;
}

// lanes per row of the two-sum kernel: NB = 2 (16 channels per lane) for scalar parameters / per-edge weights on
// rows made of 128-channel groups, else NB = 1; record chunks of at least 8 edges (narrow rows leave lanes idle)
static int two_sum_blocks_per_lane(AggParams& p, bool scalar_params) {
  const int nb = (scalar_params && p.dpad % 128 == 0) ? 2 : 1;
  p.lpr_log2 = lpr_log2_for((blocks_for(p.D) + nb - 1) / nb);
  if (p.lpr_log2 < 3) p.lpr_log2 = 3;
  return nb;
}

// forward (or dX-only) launches of the two-sum / per-edge-weight streaming kernel
template <int KIND, int BODY>
static int launch_stream2(const AggParams& p_, cudaStream_t stream) {
  AggParams p = p_;
  const int nb = two_sum_blocks_per_lane(p, BODY == 1 || p.pshape == STAG_PARAM_SCALAR);
  return nb == 2 ? launch_stream2_inst<KIND, BODY, 2>(p, stream) : launch_stream2_inst<KIND, BODY, 1>(p, stream);
}

template <bool GRADS>
static int launch_agg(const AggParams& p, bool vec, int grid, size_t smem, cudaStream_t stream) {
  // streaming variants (single channel chunk, 128-bit rows, 32-bit row offsets, no in-norm)
  const bool stream2 = !GRADS && vec && p.items && p.erow && p.eidf && p.rec && !p.in_norm && p.ncb == 1 &&
                       p.dpad <= 256 && p.ncols * p.ldx < (1ll << 31);
  if (stream2) {
    if (p.kind == STAG_NOISE_NONE) return launch_stream<STAG_NOISE_NONE, false>(p, stream);
    if (p.K == 1 && (p.kind == STAG_NOISE_EXTERNAL || p.pshape == STAG_PARAM_SCALAR)) return launch_stream2<0, 1>(p, stream);
    if (p.K != 1 && p.pshape <= STAG_PARAM_CHANNEL && (p.pshape == STAG_PARAM_CHANNEL || p.relu)) {
      if (p.kind == STAG_NOISE_NORMAL) return launch_stream2<STAG_NOISE_NORMAL, 0>(p, stream);
      if (p.kind == STAG_NOISE_UNIFORM) return launch_stream2<STAG_NOISE_UNIFORM, 0>(p, stream);
    }
  }
  if (p.kind == STAG_NOISE_NONE || p.K == 1) return launch_vec<0, 0, 0, GRADS>(p, vec, grid, smem, stream);
  if (p.kind == STAG_NOISE_EXTERNAL) return launch_vec<1, 0, 0, GRADS>(p, vec, grid, smem, stream);
  // generated per-channel noise: scalar / per-edge parameters travel with the edge record (PSH 0),
  // per-channel parameters live in registers (1), per-edge-per-channel ones are read per edge (2)
  const int psh = (p.pshape == STAG_PARAM_SCALAR || p.pshape == STAG_PARAM_EDGE) ? 0
                  : (p.pshape == STAG_PARAM_CHANNEL ? 1 : 2);
  switch (p.kind) {
    case STAG_NOISE_NORMAL: return launch_psh<STAG_NOISE_NORMAL, GRADS>(psh, p, vec, grid, smem, stream);
    case STAG_NOISE_UNIFORM: return launch_psh<STAG_NOISE_UNIFORM, GRADS>(psh, p, vec, grid, smem, stream);
    case STAG_NOISE_BERNOULLI: return launch_psh<STAG_NOISE_BERNOULLI, GRADS>(psh, p, vec, grid, smem, stream);
  }
  set_error("launch_agg: bad kind %d", p.kind);
  return STAG_EINVAL;
}

static void fill_noise(AggParams& p, const StagNoise* n, int D) {
  p.kind = n->kind;
  p.K = n->kind == STAG_NOISE_NONE ? D : n->K;
  p.pshape = n->param_shape;
  if (p.K == 1 && p.pshape == STAG_PARAM_CHANNEL) p.pshape = STAG_PARAM_SCALAR;
  if (p.K == 1 && p.pshape == STAG_PARAM_EDGE_CHANNEL) p.pshape = STAG_PARAM_EDGE;
  if (n->kind <= STAG_NOISE_EXTERNAL) p.pshape = STAG_PARAM_SCALAR;
  p.relu = n->relu;
  p.in_norm = n->in_norm;
  p.sample_base = n->sample_base;
  p.p0 = n->p0;
  p.p1 = n->p1;
  p.ext = n->external;
  p.key = make_key(n->seed, n->offset);
  p.ctr_dev = n->counter;
  p.kf = 0x4B000000u;
  for (int r = 0; r < kPhiloxRounds; ++r) {
    p.rk[2 * r] = p.key.k0 + (uint32_t)r * 0x9E3779B9u;
    p.rk[2 * r + 1] = p.key.k1 + (uint32_t)r * 0xBB67AE85u;
  }
}

static void fill_graph(AggParams& p, const StagGraph* g) {
  p.indptr = g->indptr;
  p.indices = g->indices;
  p.eid = g->eid;
  p.hub_rows = g->hub_rows;
  p.hub_seg_ptr = g->hub_seg_ptr;
  p.row_order = g->row_order;
  p.items = g->items;
  p.erow = g->erow;
  p.eidf = g->eidf;
  p.num_items = (int)g->num_items;
  p.num_hubs = g->num_hubs;
  p.num_hub_segs = g->num_hub_segs;
  p.N = (int)g->num_rows;
  p.ncols = g->num_cols;
  p.E = g->num_edges;
}

static int check_graph(const StagGraph* g, const char* who) {
  STAG_CHECK_ARG(g != nullptr, "%s: null graph", who);
  STAG_CHECK_ARG(g->num_rows >= 0 && g->num_rows < (1ll << 31) && g->num_edges >= 0 && g->num_edges < (1ll << 31),
                 "%s: graph sizes out of range", who);
  STAG_CHECK_ARG(g->indptr != nullptr, "%s: null indptr", who);
  STAG_CHECK_ARG(g->num_edges == 0 || (g->indices && g->eid), "%s: null indices/eid", who);
  STAG_CHECK_ARG(g->num_hubs == 0 || (g->hub_rows && g->hub_seg_ptr), "%s: null hub schedule", who);
  return STAG_OK;
}

// Channel tiling: D, S -> octs, column blocks, lanes per row.  `gathered_rows` is the number of
// rows of the gathered operand; blocks are only used when one [rows, D] operand does not fit the
// part of L2 a gather can count on (kL2Operand), and never in gradient mode (per-edge outputs
// are accumulated across channel chunks by one warp).
constexpr size_t kL2Operand = 96u << 20;

static void set_shape(AggParams& p, int D, int S, int64_t gathered_rows, bool shared_operand, bool grads) {
  p.D = D;
  p.S = S;
  p.nblk = blocks_for(D);
  p.dpad = (D + 63) / 64 * 64;
  const int D8 = p.dpad;
  int ncb = 1;
  if (!grads) {
    const size_t bytes = (size_t)gathered_rows * D * 4;
    ncb = (int)((bytes + kL2Operand - 1) / kL2Operand);
    if (ncb < 1) ncb = 1;
    // a small graph with wide rows (Cora: 10 556 edges x 1 433 channels) has too few stream items to fill the chip and
    // every item walks its edges once per 256-channel chunk: column blocks of whole 64-channel groups turn the chunks
    // into parallel work (set_shape runs after fill_graph: p.num_items is known)
    if (ncb == 1 && D8 >= 512) {
      const int64_t warp_items = ((int64_t)p.num_items + p.num_hub_segs + 3) / 4 * S;
      const int64_t slots = (int64_t)num_sms() * 16;
      if (warp_items > 0 && warp_items < slots) {
        const int64_t want = slots / warp_items;
        const int64_t most = D8 / 256;
        ncb = (int)(want < most ? want : most);
        if (ncb < 1) ncb = 1;
      }
    }
    static const char* force = getenv("STAG_NCB");  // tuning knob: force the number of column blocks
    if (force && atoi(force) > 0) ncb = atoi(force);
  }
  int cw = ((D8 + ncb - 1) / ncb + 63) / 64 * 64;  // whole 64-channel groups
  if (cw > D8) cw = D8;
  p.cw = cw;
  p.ncb = (D8 + cw - 1) / cw;
  p.cb_major = shared_operand && S > 1;
  p.lpr_log2 = lpr_log2_for(blocks_for(D < cw ? D : cw));
}

static int agg_grid(const AggParams& p) {
  const int RPW = 32 >> p.lpr_log2;
  const int64_t per_sample = (int64_t)(p.num_hub_segs + RPW - 1) / RPW + (p.N + RPW - 1) / RPW;
  const int64_t ctas = (per_sample * p.S * p.ncb + AGG_WARPS - 1) / AGG_WARPS;
  const int64_t cap = grid_cap();
  return (int)(ctas < 1 ? 1 : (ctas < cap ? ctas : cap));
}

}  // namespace stag

using namespace stag;

extern "C" size_t stag_spmm_workspace_bytes(const StagGraph* g, int32_t D, int32_t S) {
  if (!g || D <= 0 || S <= 0) return 0;
  return ws_layout(g, D, S, grid_cap()).total;
}

extern "C" int stag_spmm_fwd(const StagGraph* g, const float* x, int64_t ldx, int64_t x_sample_stride, int32_t D,
                             int32_t S, const StagNoise* noise, const float* src_scale, const float* dst_scale,
                             float* out, int64_t ldo, int64_t out_sample_stride, float* norm_scale_out, void* ws,
                             size_t ws_bytes, void* stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  int rc = check_graph(g, "stag_spmm_fwd");
  if (rc) return rc;
  STAG_CHECK_ARG(D > 0 && S > 0, "stag_spmm_fwd: D=%d S=%d must be positive", D, S);
  STAG_CHECK_ARG(out != nullptr, "stag_spmm_fwd: null output");
  STAG_CHECK_ARG(x != nullptr || g->num_edges == 0, "stag_spmm_fwd: null features");
  STAG_CHECK_ARG(ldx >= D && ldo >= D, "stag_spmm_fwd: row strides smaller than D");
  rc = check_noise(noise, D, g->num_edges, "stag_spmm_fwd");
  if (rc) return rc;
  if (g->num_rows == 0) return STAG_OK;
  const WsLayout L = ws_layout(g, D, S, grid_cap());
  if (!ws || ws_bytes < L.total) {
    set_error("stag_spmm_fwd: workspace %zu < required %zu", ws_bytes, L.total);
    return STAG_EWORKSPACE;
  }
  AggParams p = {};
  fill_graph(p, g);
  fill_noise(p, noise, D);
  p.x = x; p.ldx = ldx; p.x_ss = x_sample_stride;
  p.gscale = src_scale; p.rscale = dst_scale;
  p.out = out; p.ldo = ldo; p.out_ss = out_sample_stride;
  set_shape(p, D, S, g->num_cols, x_sample_stride == 0, false);
  p.norm_scale_out = norm_scale_out;
  p.part_acc = (float*)((char*)ws + L.part_acc);
  p.part_w = (float*)((char*)ws + L.part_w);
  p.rec = (const int4*)((char*)ws + L.rec);
  bool vec = (D % 4 == 0) && (ldx % 4 == 0) && (ldo % 4 == 0) && (x_sample_stride % 4 == 0) &&
             (out_sample_stride % 4 == 0) && aligned16(x) && aligned16(out);
  if (noise->kind == STAG_NOISE_EXTERNAL && noise->K != 1) vec = vec && aligned16(noise->external);
  if (noise->kind >= STAG_NOISE_NORMAL && noise->param_shape != STAG_PARAM_SCALAR && noise->K != 1)
    vec = vec && aligned16(noise->p0) && (noise->p1 == nullptr || aligned16(noise->p1));
  if (norm_scale_out && noise->K != 1) vec = vec && aligned16(norm_scale_out);
  if (noise->kind == STAG_NOISE_NORMAL_HADAMARD) {
    // tensor-core noise path (spmm_wq.cuh)
    if (g->num_edges == 0) {
      p.kind = STAG_NOISE_NONE;  // nothing to draw: the streaming kernel's tail clears the rows
    } else {
      // 256-bit gathers and row stores: 32-byte aligned rows
      const bool a32 = (((uintptr_t)x | (uintptr_t)out) & 31) == 0 && ldx % 8 == 0 && ldo % 8 == 0 &&
                       x_sample_stride % 8 == 0 && out_sample_stride % 8 == 0;
      const bool ok = noise->K == D && D % 128 == 0 && vec && a32 && !noise->relu && !noise->in_norm &&
                      (noise->param_shape == STAG_PARAM_SCALAR || noise->param_shape == STAG_PARAM_EDGE) &&
                      g->erow && g->eidf && g->items && g->num_cols * ldx * 4 < (1ll << 32) && g->num_rows * ldo * 4 < (1ll << 32);
      if (!ok) {
        set_error("stag_spmm_fwd: STAG_NOISE_NORMAL_HADAMARD needs K == D, D %% 128 == 0, 32-byte aligned rows, scalar "
                  "or per-edge parameters, no relu / in_norm, a graph built with items / erow / eidf and a gathered operand "
                  "below 4 GB (K=%d D=%d)", noise->K, D);
        return STAG_EUNSUPPORTED;
      }
      rc = launch_wh_quad(p, stream);
      if (rc) return rc;
      if (g->num_hubs > 0) {
        const int64_t total = (int64_t)S * g->num_hubs * D;
        hub_finalize_kernel<<<(unsigned)((total + 255) / 256), 256, 0, stream>>>(p, 0);
        STAG_LAUNCH_CHECK();
      }
      return STAG_OK;
    }
  }
  rc = launch_agg<false>(p, vec, agg_grid(p), 0, stream);
  if (rc) return rc;
  if (g->num_hubs > 0) {
    const int64_t total = (int64_t)S * g->num_hubs * D;
    hub_finalize_kernel<<<(unsigned)((total + 255) / 256), 256, 0, stream>>>(p, 0);
    STAG_LAUNCH_CHECK();
  }
  return STAG_OK;
}

extern "C" int stag_spmm_bwd(const StagGraph* g, const float* x, int64_t ldx, int64_t x_sample_stride,
                             const float* dout, int64_t ldg, int64_t dout_sample_stride, int32_t D, int32_t S,
                             const StagNoise* noise, const float* src_scale, const float* dst_scale, float* dx,
                             int64_t lddx, int64_t dx_sample_stride, float* dparam0, float* dparam1,
                             float* dw_external, void* ws, size_t ws_bytes, void* stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  int rc = check_graph(g, "stag_spmm_bwd");
  if (rc) return rc;
  STAG_CHECK_ARG(D > 0 && S > 0, "stag_spmm_bwd: D=%d S=%d must be positive", D, S);
  STAG_CHECK_ARG(dout != nullptr || g->num_edges == 0, "stag_spmm_bwd: null upstream gradient");
  STAG_CHECK_ARG(x != nullptr || g->num_edges == 0, "stag_spmm_bwd: null features");
  STAG_CHECK_ARG(ldx >= D && ldg >= D && (dx == nullptr || lddx >= D), "stag_spmm_bwd: row strides smaller than D");
  rc = check_noise(noise, D, g->num_edges, "stag_spmm_bwd");
  if (rc) return rc;
  if (noise->kind == STAG_NOISE_NORMAL_HADAMARD) {
    set_error("stag_spmm_bwd: STAG_NOISE_NORMAL_HADAMARD has no parameter-gradient path (dX: stag_spmm_fwd on the CSR)");
    return STAG_EUNSUPPORTED;
  }
  if (noise->in_norm) {
    set_error("stag_spmm_bwd: in_norm has no fused parameter-gradient path (use the emitted-noise path)");
    return STAG_EUNSUPPORTED;
  }
  const bool param_grads = noise->kind == STAG_NOISE_NORMAL || noise->kind == STAG_NOISE_UNIFORM;
  if (param_grads) STAG_CHECK_ARG(dparam0 && dparam1, "stag_spmm_bwd: null parameter-gradient outputs");
  AggParams p = {};
  fill_graph(p, g);
  fill_noise(p, noise, D);
  const bool edge_params = param_grads && p.pshape >= STAG_PARAM_EDGE;
  // per-edge parameter gradients for any S need the row of every stored edge (edge-parallel kernel); without it the
  // row-per-group family takes one sample per launch
  const bool edge_parallel = edge_params && g->erow != nullptr;
  STAG_CHECK_ARG(!edge_params || edge_parallel || S == 1,
                 "stag_spmm_bwd: per-edge parameter gradients on a graph without erow require S == 1 (got %d)", S);
  if (g->num_rows == 0) {
    if (param_grads && !edge_params) {
      const size_t n = p.pshape == STAG_PARAM_SCALAR ? 1 : (size_t)D;
      STAG_CUDA(cudaMemsetAsync(dparam0, 0, n * 4, stream));
      STAG_CUDA(cudaMemsetAsync(dparam1, 0, n * 4, stream));
    }
    return STAG_OK;
  }
  const WsLayout L = ws_layout(g, D, S, grid_cap());
  if (!ws || ws_bytes < L.total) {
    set_error("stag_spmm_bwd: workspace %zu < required %zu", ws_bytes, L.total);
    return STAG_EWORKSPACE;
  }
  // transposed roles: gather dout rows scaled by dst_scale, rows are sources scaled by src_scale
  p.x = dout; p.ldx = ldg; p.x_ss = dout_sample_stride;
  p.gscale = dst_scale; p.rscale = src_scale;
  p.out = dx; p.ldo = lddx; p.out_ss = dx_sample_stride;
  p.xrow = x; p.ldxr = ldx; p.xr_ss = x_sample_stride;
  set_shape(p, D, S, g->num_cols, false, true);
  p.dp0 = dparam0; p.dp1 = dparam1; p.dw_ext = dw_external;
  p.part_acc = (float*)((char*)ws + L.part_acc);
  p.part_w = (float*)((char*)ws + L.part_w);
  p.dp_partial = (float*)((char*)ws + L.dp_partial);
  bool vec = (D % 4 == 0) && (ldx % 4 == 0) && (ldg % 4 == 0) && (x_sample_stride % 4 == 0) &&
             (dout_sample_stride % 4 == 0) && aligned16(x) && aligned16(dout);
  if (dx) vec = vec && (lddx % 4 == 0) && (dx_sample_stride % 4 == 0) && aligned16(dx);
  if (noise->kind == STAG_NOISE_EXTERNAL && noise->K != 1)
    vec = vec && aligned16(noise->external) && (dw_external == nullptr || aligned16(dw_external));
  const bool vec_rows = vec;  // feature / gradient rows take 128-bit accesses (the parameter tensors may still not)
  if (param_grads && noise->param_shape != STAG_PARAM_SCALAR && noise->K != 1)
    vec = vec && aligned16(noise->p0) && aligned16(noise->p1) && aligned16(dparam0) && aligned16(dparam1);
  if (edge_parallel) {
    // dX: the transposed aggregation on the forward kernels (streaming kernel for per-edge parameters without relu)
    if (dx) {
      AggParams q = p;
      set_shape(q, D, S, g->num_cols, false, false);
      q.rec = (const int4*)((char*)ws + L.rec);
      q.xrow = nullptr; q.dp0 = q.dp1 = nullptr; q.dw_ext = nullptr;
      // (the dX pass reads the parameters, never the gradient tensors: their alignment does not matter here)
      const bool vec_dx = vec_rows && (noise->param_shape != STAG_PARAM_EDGE_CHANNEL ||
                                       (aligned16(noise->p0) && aligned16(noise->p1)));
      rc = launch_agg<false>(q, vec_dx, agg_grid(q), 0, stream);
      if (rc) return rc;
      if (g->num_hubs > 0) {
        const int64_t total = (int64_t)S * g->num_hubs * D;
        hub_finalize_kernel<<<(unsigned)((total + 255) / 256), 256, 0, stream>>>(q, 0);
        STAG_LAUNCH_CHECK();
      }
    }
    if (p.E > 0) {
      const int64_t want = (p.E + 15) / 16;
      const int egrid = (int)(want < (int64_t)num_sms() * 16 ? want : (int64_t)num_sms() * 16);
      const bool fast = noise->kind == STAG_NOISE_NORMAL && noise->param_shape == STAG_PARAM_EDGE && !noise->relu &&
                        noise->K == D && D % 128 == 0 && vec_rows;   // [E,1] parameters: scalar reads / writes per edge
      if (fast) {
        const int64_t want8 = (p.E + 31) / 32;
        edge_param_grads_fast_kernel<<<(int)(want8 < (int64_t)num_sms() * 16 ? want8 : (int64_t)num_sms() * 16), 256, 0, stream>>>(p);
      } else if (noise->kind == STAG_NOISE_NORMAL) {
        if (vec) edge_param_grads_kernel<STAG_NOISE_NORMAL, true><<<egrid, 256, 0, stream>>>(p);
        else edge_param_grads_kernel<STAG_NOISE_NORMAL, false><<<egrid, 256, 0, stream>>>(p);
      } else {
        if (vec) edge_param_grads_kernel<STAG_NOISE_UNIFORM, true><<<egrid, 256, 0, stream>>>(p);
        else edge_param_grads_kernel<STAG_NOISE_UNIFORM, false><<<egrid, 256, 0, stream>>>(p);
      }
      STAG_LAUNCH_CHECK();
    }
    return STAG_OK;
  }
  const int grid = agg_grid(p);
  const size_t smem = (param_grads && !edge_params) ? (size_t)AGG_WARPS * 2 * p.dpad * sizeof(float) : 0;
  if (smem > 200 * 1024) {
    set_error("stag_spmm_bwd: D=%d too wide for the shared-memory parameter-gradient staging", D);
    return STAG_EUNSUPPORTED;
  }
  // streaming gradient kernel: generated per-channel Normal / Uniform noise, scalar or per-channel
  // parameters, one channel chunk (D <= 256), 128-bit rows, 32-bit row offsets
  const bool stream_ok = param_grads && !edge_params && noise->K == D && vec && p.items && p.erow && p.eidf &&
                         p.dpad <= 256 && p.ncols * p.ldx < (1ll << 31) && (int64_t)p.N * p.ldxr < (1ll << 31);
  int sgrid = grid;
  if (stream_ok) {
    p.rec = (const int4*)((char*)ws + L.rec);
    const int nb = two_sum_blocks_per_lane(p, p.pshape == STAG_PARAM_SCALAR);
    const int RPW = 32 >> p.lpr_log2;
    const int64_t warp_items = (int64_t)((p.num_hub_segs + p.num_items + RPW - 1) / RPW) * p.S;
    const int64_t ctas = (warp_items + AGG_WARPS - 1) / AGG_WARPS;
    sgrid = (int)(ctas < 1 ? 1 : (ctas < num_sms() * 2 ? ctas : num_sms() * 2));
    const size_t ring_bytes = (size_t)AGG_WARPS * s2_warp_bytes(true, nb) + smem;
    if (p.E > 0) {
      edge_record_kernel<STAG_NOISE_NORMAL><<<(unsigned)((p.E + 255) / 256), 256, 0, stream>>>(
          p, const_cast<int4*>(p.rec), 1);
      STAG_LAUNCH_CHECK();
    }
    auto launch = [&](auto kern) -> int {
      STAG_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ring_bytes));
      kern<<<sgrid, AGG_THREADS, ring_bytes, stream>>>(p);
      return STAG_OK;
    };
    int lrc;
    if (noise->kind == STAG_NOISE_NORMAL)
      lrc = nb == 2 ? launch(agg_stream_grads_kernel<STAG_NOISE_NORMAL, 0, true, 2>)
                    : launch(agg_stream_grads_kernel<STAG_NOISE_NORMAL, 0, true, 1>);
    else
      lrc = nb == 2 ? launch(agg_stream_grads_kernel<STAG_NOISE_UNIFORM, 0, true, 2>)
                    : launch(agg_stream_grads_kernel<STAG_NOISE_UNIFORM, 0, true, 1>);
    if (lrc) return lrc;
    STAG_LAUNCH_CHECK();
  } else {
    rc = launch_agg<true>(p, vec, grid, smem, stream);
    if (rc) return rc;
  }
  if (g->num_hubs > 0 && dx) {
    const int64_t total = (int64_t)S * g->num_hubs * D;
    hub_finalize_kernel<<<(unsigned)((total + 255) / 256), 256, 0, stream>>>(p, 1);
    STAG_LAUNCH_CHECK();
  }
  if (param_grads && !edge_params) {
    const int scalar = p.pshape == STAG_PARAM_SCALAR;
    const int blocks = scalar ? 1 : (D + 255) / 256;
    param_finalize_kernel<<<blocks, 256, 0, stream>>>(p.dp_partial, stream_ok ? sgrid : grid, p.dpad, D, scalar, dparam0,
                                                     dparam1);
    STAG_LAUNCH_CHECK();
  }
  return STAG_OK;
}

extern "C" int stag_noise_emit(const StagNoise* noise, int64_t num_edges, int32_t S, float* w_out, float* eps_out,
                               void* stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  STAG_CHECK_ARG(noise != nullptr && w_out != nullptr, "stag_noise_emit: null argument");
  STAG_CHECK_ARG(noise->kind >= STAG_NOISE_NORMAL && noise->kind <= STAG_NOISE_NORMAL_HADAMARD,
                 "stag_noise_emit: kind %d is not a generated distribution", noise->kind);
  STAG_CHECK_ARG(noise->K > 0 && S > 0 && num_edges >= 0 && num_edges < (1ll << 31), "stag_noise_emit: bad sizes");
  int rc = check_noise(noise, noise->K, num_edges, "stag_noise_emit");
  if (rc) return rc;
  if (num_edges == 0) return STAG_OK;
  AggParams p = {};
  fill_noise(p, noise, noise->K);
  p.ncb = 1;
  p.E = num_edges;
  p.S = S;
  p.D = noise->K;
  p.nblk = blocks_for(noise->K);
  p.dpad = (noise->K + 63) / 64 * 64;
  const int64_t total = (int64_t)S * num_edges * p.nblk;
  const int64_t want = (total + 255) / 256;
  const int grid = (int)(want < (int64_t)num_sms() * 16 ? want : (int64_t)num_sms() * 16);
  if (noise->kind == STAG_NOISE_NORMAL_HADAMARD) {
    const int64_t warps = (int64_t)S * num_edges * (noise->K >> 7);
    const int64_t ctas = (warps + 7) / 8;
    emit_wh_kernel<<<(unsigned)(ctas < (int64_t)num_sms() * 16 ? ctas : (int64_t)num_sms() * 16), 256, 0, stream>>>(
        p, w_out, eps_out);
    STAG_LAUNCH_CHECK();
    return STAG_OK;
  }
  switch (noise->kind) {
    case STAG_NOISE_NORMAL: emit_kernel<STAG_NOISE_NORMAL><<<grid, 256, 0, stream>>>(p, w_out, eps_out); break;
    case STAG_NOISE_UNIFORM: emit_kernel<STAG_NOISE_UNIFORM><<<grid, 256, 0, stream>>>(p, w_out, eps_out); break;
    default: emit_kernel<STAG_NOISE_BERNOULLI><<<grid, 256, 0, stream>>>(p, w_out, eps_out); break;
  }
  STAG_LAUNCH_CHECK();
  return STAG_OK;
}

extern "C" size_t stag_noise_kl_workspace_bytes(int32_t K) {
  if (K <= 0) return 0;
  const size_t kpad = (size_t)((K + 63) / 64) * 64;
  const size_t grid = (size_t)num_sms() * 4;
  return align_up(grid * 4 * sizeof(double), 256) + align_up(grid * 2 * kpad * sizeof(float), 256);
}

extern "C" int stag_noise_kl(const StagNoise* noise, int64_t num_edges, int32_t S, const StagPrior* prior, double* sums,
                             float* dparam0, float* dparam1, void* ws, size_t ws_bytes, void* stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  STAG_CHECK_ARG(noise != nullptr && prior != nullptr && sums != nullptr, "stag_noise_kl: null argument");
  STAG_CHECK_ARG(noise->K > 0 && S > 0 && num_edges >= 0 && num_edges < (1ll << 31), "stag_noise_kl: bad sizes");
  int rc = check_noise(noise, noise->K, num_edges, "stag_noise_kl");
  if (rc) return rc;
  if (noise->kind != STAG_NOISE_NORMAL && noise->kind != STAG_NOISE_UNIFORM) {
    set_error("stag_noise_kl: the posterior must be a reparameterised Normal or Uniform drawn by the Box-Muller / uniform "
              "generators (kind %d)", noise->kind);
    return STAG_EUNSUPPORTED;
  }
  if (noise->in_norm) {
    set_error("stag_noise_kl: in-norm rescales the sample by a per-row factor the edge pass does not have");
    return STAG_EUNSUPPORTED;
  }
  STAG_CHECK_ARG(prior->kind == STAG_PRIOR_NORMAL_MIXTURE && prior->M >= 1 && prior->M <= STAG_PRIOR_MAX_COMPONENTS,
                 "stag_noise_kl: prior must be a mixture of 1..%d Normals", STAG_PRIOR_MAX_COMPONENTS);
  STAG_CHECK_ARG((dparam0 == nullptr) == (dparam1 == nullptr), "stag_noise_kl: pass both gradient outputs or neither");
  const size_t need = stag_noise_kl_workspace_bytes(noise->K);
  if (!ws || ws_bytes < need) {
    set_error("stag_noise_kl: workspace %zu < required %zu", ws_bytes, need);
    return STAG_EWORKSPACE;
  }
  KlParams p = {};
  p.E = num_edges; p.S = S; p.K = noise->K;
  p.nblk = blocks_for(noise->K);
  p.kpad = (noise->K + 63) / 64 * 64;
  p.pshape = noise->param_shape; p.relu = noise->relu; p.sample_base = noise->sample_base;
  p.p0 = noise->p0; p.p1 = noise->p1;
  p.key = make_key(noise->seed, noise->offset);
  p.ctr_dev = noise->counter;
  p.M = prior->M;
  double wsum = 0.0;
  for (int m = 0; m < prior->M; ++m) {
    STAG_CHECK_ARG(prior->weight[m] > 0.f && prior->scale[m] > 0.f, "stag_noise_kl: prior weights and scales must be positive");
    wsum += prior->weight[m];
  }
  for (int m = 0; m < prior->M; ++m) {
    p.c_m[m] = (float)(log((double)prior->weight[m] / wsum) - log((double)prior->scale[m]) - 0.9189385332046727);
    p.mu_m[m] = prior->loc[m];
    p.is_m[m] = 1.0f / prior->scale[m];
  }
  p.dp0 = dparam0; p.dp1 = dparam1;
  const int grid = kl_grid(num_edges);
  p.cta_sums = (double*)ws;
  p.cta_ch = (float*)((char*)ws + align_up((size_t)num_sms() * 4 * 4 * sizeof(double), 256));
  const bool grads = dparam0 != nullptr;
  const size_t smem = (grads && p.pshape == STAG_PARAM_CHANNEL) ? (size_t)KL_WARPS * 2 * p.kpad * sizeof(float) : 0;
  if (num_edges > 0) {
#define STAG_KL_LAUNCH(KIND, G)                                                                                      \
  do {                                                                                                               \
    if (smem > 48 * 1024)                                                                                            \
      STAG_CUDA(cudaFuncSetAttribute(noise_kl_kernel<KIND, G>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)); \
    noise_kl_kernel<KIND, G><<<grid, KL_THREADS, smem, stream>>>(p);                                                  \
  } while (0)
    if (noise->kind == STAG_NOISE_NORMAL) { if (grads) STAG_KL_LAUNCH(STAG_NOISE_NORMAL, true); else STAG_KL_LAUNCH(STAG_NOISE_NORMAL, false); }
    else { if (grads) STAG_KL_LAUNCH(STAG_NOISE_UNIFORM, true); else STAG_KL_LAUNCH(STAG_NOISE_UNIFORM, false); }
#undef STAG_KL_LAUNCH
    STAG_LAUNCH_CHECK();
  }
  noise_kl_finalize<<<1, 256, 0, stream>>>(p, num_edges > 0 ? grid : 0, grads ? 1 : 0, sums);
  STAG_LAUNCH_CHECK();
  return STAG_OK;
}

extern "C" int stag_segment_reduce(const float* feat, int64_t ldf, const int32_t* node_ptr, int32_t num_graphs,
                                   int32_t D, int mean, float* out, int64_t ldo, void* stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  STAG_CHECK_ARG(num_graphs >= 0 && D > 0, "stag_segment_reduce: bad sizes");
  if (num_graphs == 0) return STAG_OK;
  STAG_CHECK_ARG(feat && node_ptr && out, "stag_segment_reduce: null argument");
  const int64_t total = (int64_t)num_graphs * D;
  segment_reduce_kernel<<<(unsigned)((total + 255) / 256), 256, 0, stream>>>(feat, ldf, node_ptr, num_graphs, D, mean,
                                                                             out, ldo);
  STAG_LAUNCH_CHECK();
  return STAG_OK;
}
#include "spmm_max.cuh"
