// Stochastic max aggregation (included at the end of spmm.cu): DGL's update_all(u_mul_e, fn.max) with the edge noise
// drawn in the kernel, as GraphSAGE 'pool' and GIN 'max' use it.
//
//   out[s,v,c] = max over the in-edges e = (u -> v) of  w_s[e,c] * x[s,u,c]      (fp32 product, then compare)
//   arg[s,v,c] = ORIGINAL id of the winning edge
//
// Ties go to the first edge in stored order (edge-id order: the CSC is a stable sort): an edge replaces the running
// maximum only when its product is strictly greater.  Rows without in-edges get out = 0, arg = -1.  The variates are
// the ones stag_noise_emit writes (same Philox / Hadamard stream, same transform), so the fused max equals the max
// over the materialised noise bit for bit.
//
// Kernels (one writer per output element and fixed orders everywhere: bitwise deterministic, no float atomics):
//   max_row_kernel<KIND, VEC, BWD>  row per group of LPR lanes, a lane owns one Philox oct (8 channels) of the row at a
//                                   time and walks the row's edges in stored order.
//     BWD = false  forward on the CSC: (max, arg) per channel in registers
//     BWD = true   transposed pass on the CSR: dx[s,u,c] = sum over out-edges e = (u -> v) with arg[s,v,c] == e of
//                  w_s[e,c] g[s,v,c]; the scalar / per-channel parameter gradients ride along (per-warp slices in
//                  shared memory -> per-CTA partial rows -> param_finalize_kernel).  The noise of an edge is only
//                  regenerated when it wins one of the lane's channels.
//   max_wh_kernel<BWD>              the same two passes for STAG_NOISE_NORMAL_HADAMARD: one warp per (row, sample,
//                                   128-channel group), lane = 4 consecutive channels (wh_group_sums).
//   max_edge_kernel<KIND, VEC>      edge-parallel: dw_external of EXTERNAL noise and the per-edge ([E,1]) parameter
//                                   gradients; half a warp per stored edge, samples in order.
//   max_hub_finalize_kernel         hub rows (more than kHubThreshold edges) run as segments; their (max, arg) pairs
//                                   are combined in segment order with the same strict comparison ("first wins").
// Not here: src / dst scales, in-norm and [E,K] parameters (the Python operator routes those through the materialised
// noise tensor), the streaming / tensor-core sum kernels.
//
// Why a sibling of agg_kernel rather than a template switch in it: the max forward keeps an int per channel, writes
// two outputs per row and needs no edge records or shuffles, and the backward reads one extra int row per edge and
// skips the noise of losing edges; in agg_kernel each of these would be a branch on the caller.
#pragma once

namespace stag {

// The noise of one (edge, sample) on the 8 channels of a lane (chan(c, i)), as stag_noise_emit writes it.  `raw` are
// the variates before the transform (parameter gradients), `pre` the weights before relu (relu mask).
template <int KIND, bool VEC>
__device__ __forceinline__ void max_weights(const AggParams& p, const PhiloxKey& key, int s, uint32_t smp, int e,
                                            uint32_t oct, int c, const float (&P0)[8], const float (&P1)[8],
                                            float (&w)[8], float (&raw)[8], float (&pre)[8]) {
  if (KIND == STAG_NOISE_NONE) {
#pragma unroll
    for (int i = 0; i < 8; ++i) w[i] = raw[i] = pre[i] = 1.0f;
    return;
  }
  if (KIND == STAG_NOISE_EXTERNAL) {
    if (p.K == 1) {
      const float v = __ldg(p.ext + (int64_t)s * p.E + e);
#pragma unroll
      for (int i = 0; i < 8; ++i) w[i] = v;
    } else {
      load8<VEC>(p.ext + ((int64_t)s * p.E + e) * p.K, c, p.D, w);
    }
#pragma unroll
    for (int i = 0; i < 8; ++i) raw[i] = pre[i] = w[i];
    return;
  }
  if (p.K == 1) {
    const float r = raw_first(KIND, (uint32_t)e, smp, key);
#pragma unroll
    for (int i = 0; i < 8; ++i) raw[i] = r;
  } else {
    raw_oct<KIND>((uint32_t)e, oct, smp, key, raw);
  }
  float a[8], b[8];
  if (p.pshape == STAG_PARAM_EDGE) {
    const float ea = __ldg(p.p0 + e), eb = KIND != STAG_NOISE_BERNOULLI ? __ldg(p.p1 + e) : 0.f;
#pragma unroll
    for (int i = 0; i < 8; ++i) { a[i] = ea; b[i] = eb; }
  } else {
#pragma unroll
    for (int i = 0; i < 8; ++i) { a[i] = P0[i]; b[i] = P1[i]; }
  }
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    pre[i] = transform<KIND>(raw[i], a[i], b[i]);
    w[i] = p.relu ? fmaxf(pre[i], 0.f) : pre[i];
  }
}

// Rows / hub segments of a launch: items r < HG are hub-segment groups, the rest row groups (as agg_kernel).
__device__ __forceinline__ void max_resolve(const AggParams& p, int r, int HG, int RPW, int sub, int& row, int& beg,
                                            int& len, int& part_slot) {
  row = -1; beg = 0; len = 0; part_slot = -1;
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
    const int v = (r - HG) * RPW + sub;
    if (v < p.N) {
      const int rb = __ldg(p.indptr + v), re = __ldg(p.indptr + v + 1);
      if (re - rb <= kHubThreshold) {
        row = v;
        beg = rb;
        len = re - rb;
      }
    }
  }
}

// Forward (BWD = false): p.x = features (gathered), p.out / arg_out [S,N,D] at (ldo, out_ss).
// Backward (BWD = true): p.x = dout (gathered, rows v), arg_in at the strides of dout, p.xrow = features (rows u),
// p.out = dx (may be null), p.dp0 / p.dp1 set: scalar / per-channel parameter gradients into p.dp_partial.
template <int KIND, bool VEC, bool BWD>
__global__ void __launch_bounds__(AGG_THREADS) max_row_kernel(const AggParams p, const int32_t* __restrict__ arg_in,
                                                              int32_t* __restrict__ arg_out) {
  const PhiloxKey key = live_key(p);
  extern __shared__ float smem[];  // parameter gradients: [AGG_WARPS][2][dpad]
  constexpr bool PG_KIND = BWD && (KIND == STAG_NOISE_NORMAL || KIND == STAG_NOISE_UNIFORM);
  const bool dense_pg = PG_KIND && p.dp0 != nullptr;
  const int lane = threadIdx.x & 31;
  const int warp = threadIdx.x >> 5;
  const int LPR = 1 << p.lpr_log2;
  const int RPW = 32 >> p.lpr_log2;
  const int sub = lane >> p.lpr_log2;
  const int sl = lane & (LPR - 1);
  const int D8 = p.dpad;

  float* my_sm = nullptr;
  if (dense_pg) {
    my_sm = smem + (size_t)warp * 2 * D8;
    for (int i = lane; i < 2 * D8; i += 32) my_sm[i] = 0.f;
    __syncwarp();
  }

  const int HG = (p.num_hub_segs + RPW - 1) / RPW;
  const int RG = (p.N + RPW - 1) / RPW;
  const int64_t per_sample = (int64_t)HG + RG;
  const int64_t total = per_sample * p.S;
  const int64_t total_warps = (int64_t)gridDim.x * AGG_WARPS;

  for (int64_t item = (int64_t)blockIdx.x * AGG_WARPS + warp; item < total; item += total_warps) {
    const int s = (int)(item / per_sample);
    const int r = (int)(item - (int64_t)s * per_sample);
    int row, beg, len, part_slot;
    max_resolve(p, r, HG, RPW, sub, row, beg, len, part_slot);
    if (!__any_sync(0xffffffffu, row >= 0)) continue;
    const float* xs = p.x + (int64_t)s * p.x_ss;
    const uint32_t smp = (uint32_t)(p.sample_base + s);

    for (int c0 = 0; c0 < D8; c0 += max(LPR * 8, 64)) {
      const int c = first_chan(c0, sl);
      const bool qvalid = row >= 0 && c < p.D;
      const uint32_t oct = (uint32_t)((c0 >> 3) + sl);
      float P0[8], P1[8];
#pragma unroll
      for (int i = 0; i < 8; ++i) P0[i] = P1[i] = 0.f;
      if (KIND >= STAG_NOISE_NORMAL && p.pshape == STAG_PARAM_SCALAR) {
        const float a = __ldg(p.p0), b = KIND != STAG_NOISE_BERNOULLI ? __ldg(p.p1) : 0.f;
#pragma unroll
        for (int i = 0; i < 8; ++i) { P0[i] = a; P1[i] = b; }
      } else if (KIND >= STAG_NOISE_NORMAL && p.pshape == STAG_PARAM_CHANNEL && qvalid) {
        load8<VEC>(p.p0, c, p.D, P0);
        if (KIND != STAG_NOISE_BERNOULLI) load8<VEC>(p.p1, c, p.D, P1);
      }
      float acc[8], d0[8], d1[8], xr[8];
      int am[8];
#pragma unroll
      for (int i = 0; i < 8; ++i) { acc[i] = d0[i] = d1[i] = xr[i] = 0.f; am[i] = -1; }
      if (dense_pg && qvalid) load8<VEC>(p.xrow + (int64_t)s * p.xr_ss + (int64_t)row * p.ldxr, c, p.D, xr);

      if (qvalid) {
        for (int j = beg; j < beg + len; ++j) {
          const int nb = __ldg(p.indices + j);
          const int e = __ldg(p.eid + j);
          float xv[8], w[8], raw[8], pre[8];
          load8<VEC>(xs + (int64_t)nb * p.ldx, c, p.D, xv);
          if (!BWD) {
            max_weights<KIND, VEC>(p, key, s, smp, e, oct, c, P0, P1, w, raw, pre);
#pragma unroll
            for (int i = 0; i < 8; ++i) {
              const float v = w[i] * xv[i];
              if (am[i] < 0 || v > acc[i]) { acc[i] = v; am[i] = e; }
            }
          } else {
            float av[8];
            load8<VEC>(reinterpret_cast<const float*>(arg_in) + (int64_t)s * p.x_ss + (int64_t)nb * p.ldx, c, p.D, av);
            bool win[8], any = false;
#pragma unroll
            for (int i = 0; i < 8; ++i) {
              win[i] = __float_as_int(av[i]) == e && chan(c, i) < p.D;
              any |= win[i];
            }
            if (!any) continue;
            max_weights<KIND, VEC>(p, key, s, smp, e, oct, c, P0, P1, w, raw, pre);
#pragma unroll
            for (int i = 0; i < 8; ++i) {
              if (!win[i]) continue;
              acc[i] = fmaf(w[i], xv[i], acc[i]);
              if (PG_KIND && dense_pg) {
                const float dw = (p.relu && !(pre[i] > 0.f)) ? 0.f : xr[i] * xv[i];
                const float e1 = dw * raw[i];
                d1[i] += e1;
                d0[i] += KIND == STAG_NOISE_NORMAL ? dw : dw - e1;
              }
            }
          }
        }
        if (!BWD) {
#pragma unroll
          for (int i = 0; i < 8; ++i) if (am[i] < 0) acc[i] = 0.f;  // no in-edges
        }
        float amf[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) amf[i] = __int_as_float(am[i]);
        if (part_slot >= 0) {
          if (!BWD || p.out) {
            const int64_t o = ((int64_t)s * p.num_hub_segs + part_slot) * D8;
            store8<true, false>(p.part_acc + o, c, D8, acc);
            if (!BWD) store8<true, false>(p.part_w + o, c, D8, amf);
          }
        } else if (!BWD || p.out) {
          store8<VEC, false>(p.out + (int64_t)s * p.out_ss + (int64_t)row * p.ldo, c, p.D, acc);
          if (!BWD) store8<VEC, false>(reinterpret_cast<float*>(arg_out) + (int64_t)s * p.out_ss + (int64_t)row * p.ldo, c, p.D, amf);
        }
      }
      if (dense_pg) {
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
        __syncwarp();
      }
    }
  }

  if (dense_pg) {
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

// STAG_NOISE_NORMAL_HADAMARD: one warp per (sample, row or hub segment, 128-channel group); the noise of a group comes
// from wh_group_sums and is evaluated as stag_noise_emit does, w = fmaf(sum, scale * kWhInvSd, loc).  K == D,
// D % 128 == 0, 16-byte aligned rows; scalar, per-channel or per-edge parameters, relu.
template <bool BWD>
__global__ void __launch_bounds__(256) max_wh_kernel(const AggParams p, const int32_t* __restrict__ arg_in,
                                                     int32_t* __restrict__ arg_out) {
  const PhiloxKey key = live_key(p);
  const int lane = threadIdx.x & 31;
  const int G = p.D >> 7;
  const int64_t per_sample = (int64_t)(p.num_hub_segs + p.N) * G;
  const int64_t total = per_sample * p.S;
  const int64_t nwarps = (int64_t)gridDim.x * (blockDim.x >> 5);
  for (int64_t item = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); item < total; item += nwarps) {
    const int s = (int)(item / per_sample);
    const int64_t rg = item - (int64_t)s * per_sample;
    const int r = (int)(rg / G);
    const int g = (int)(rg - (int64_t)r * G);
    int row, beg, len, part_slot;
    max_resolve(p, r, p.num_hub_segs, 1, 0, row, beg, len, part_slot);
    if (row < 0) continue;  // warp-uniform: a hub row outside its segments
    const int ch = 128 * g + 4 * lane;
    const uint32_t smp = (uint32_t)(p.sample_base + s);
    float a[4] = {0.f, 0.f, 0.f, 0.f}, b[4] = {0.f, 0.f, 0.f, 0.f};
    if (p.pshape == STAG_PARAM_SCALAR) {
      a[0] = a[1] = a[2] = a[3] = __ldg(p.p0);
      b[0] = b[1] = b[2] = b[3] = __ldg(p.p1) * kWhInvSd;
    } else if (p.pshape == STAG_PARAM_CHANNEL) {
#pragma unroll
      for (int k = 0; k < 4; ++k) { a[k] = __ldg(p.p0 + ch + k); b[k] = __ldg(p.p1 + ch + k) * kWhInvSd; }
    }
    const float* xs = p.x + (int64_t)s * p.x_ss;
    float acc[4] = {0.f, 0.f, 0.f, 0.f};
    int am[4] = {-1, -1, -1, -1};
    for (int j = beg; j < beg + len; ++j) {
      const int nb = __ldg(p.indices + j);
      const int e = __ldg(p.eid + j);
      const float4 xv4 = __ldg(reinterpret_cast<const float4*>(xs + (int64_t)nb * p.ldx + ch));
      const float xv[4] = {xv4.x, xv4.y, xv4.z, xv4.w};
      bool win[4] = {true, true, true, true};
      if (BWD) {
        const int4 a4 = __ldg(reinterpret_cast<const int4*>(arg_in + (int64_t)s * p.x_ss + (int64_t)nb * p.ldx + ch));
        win[0] = a4.x == e; win[1] = a4.y == e; win[2] = a4.z == e; win[3] = a4.w == e;
        if (!__any_sync(0xffffffffu, win[0] || win[1] || win[2] || win[3])) continue;
      }
      if (p.pshape == STAG_PARAM_EDGE) {
        const float ea = __ldg(p.p0 + e), eb = __ldg(p.p1 + e) * kWhInvSd;
        a[0] = a[1] = a[2] = a[3] = ea;
        b[0] = b[1] = b[2] = b[3] = eb;
      }
      float v[4];
      wh_group_sums((uint32_t)e, (uint32_t)g, smp, key, lane, v);
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        float w = fmaf(v[k], b[k], a[k]);
        if (p.relu) w = fmaxf(w, 0.f);
        if (!BWD) {
          const float m = w * xv[k];
          if (am[k] < 0 || m > acc[k]) { acc[k] = m; am[k] = e; }
        } else if (win[k]) {
          acc[k] = fmaf(w, xv[k], acc[k]);
        }
      }
    }
    if (!BWD) {
#pragma unroll
      for (int k = 0; k < 4; ++k) if (am[k] < 0) acc[k] = 0.f;
    }
    if (BWD && !p.out) continue;
    const float4 o4 = make_float4(acc[0], acc[1], acc[2], acc[3]);
    const int4 a4 = make_int4(am[0], am[1], am[2], am[3]);
    if (part_slot >= 0) {
      const int64_t o = ((int64_t)s * p.num_hub_segs + part_slot) * p.dpad + ch;
      *reinterpret_cast<float4*>(p.part_acc + o) = o4;
      if (!BWD) *reinterpret_cast<int4*>(reinterpret_cast<int*>(p.part_w) + o) = a4;
    } else {
      const int64_t o = (int64_t)s * p.out_ss + (int64_t)row * p.ldo + ch;
      *reinterpret_cast<float4*>(p.out + o) = o4;
      if (!BWD) *reinterpret_cast<int4*>(arg_out + o) = a4;
    }
  }
}

// Combine the (max, arg) pairs of the segments of a hub row in segment order: strict > keeps the first winner.
__global__ void max_hub_finalize_kernel(const AggParams p, int32_t* __restrict__ arg_out) {
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t total = (int64_t)p.S * p.num_hubs * p.D;
  if (idx >= total) return;
  const int c = (int)(idx % p.D);
  const int h = (int)((idx / p.D) % p.num_hubs);
  const int s = (int)(idx / ((int64_t)p.D * p.num_hubs));
  const int row = p.hub_rows[h];
  const int s0 = p.hub_seg_ptr[h], s1 = p.hub_seg_ptr[h + 1];
  const int* part_arg = reinterpret_cast<const int*>(p.part_w);
  float m = 0.f;
  int a = -1;
  for (int seg = s0; seg < s1; ++seg) {
    const int64_t o = ((int64_t)s * p.num_hub_segs + seg) * p.dpad + c;
    const float v = p.part_acc[o];
    if (a < 0 || v > m) { m = v; a = part_arg[o]; }
  }
  p.out[(int64_t)s * p.out_ss + (int64_t)row * p.ldo + c] = m;
  arg_out[(int64_t)s * p.out_ss + (int64_t)row * p.ldo + c] = a;
}

// Edge-parallel part of the backward on the CSR (p.x = dout with arg_in at its strides, p.xrow = features): half a
// warp owns one stored edge j = (u -> v), a lane one oct of channels at a time, the samples in order.
//   dw[s,e,c] = x[s,u,c] g[s,v,c] where arg[s,v,c] == e, else 0
//   EXTERNAL, p.dw_ext:  K == D: dw written per (s, e, c);  K == 1: its sum over the channels, per (s, e)
//   Normal / Uniform [E,1] parameters:  dp0[e] += sum_{s,c} dw (1 | 1 - u),  dp1[e] += sum_{s,c} dw (eps | u)
// One writer per edge, fixed order: deterministic.
template <int KIND, bool VEC>
__global__ void __launch_bounds__(256) max_edge_kernel(const AggParams p, const int32_t* __restrict__ arg_in) {
  const PhiloxKey key = live_key(p);
  const int lane = threadIdx.x & 31, hl = lane & 15;
  const int64_t nhw = (int64_t)gridDim.x * (blockDim.x >> 4);
  const int64_t hw0 = (int64_t)blockIdx.x * (blockDim.x >> 4) + (threadIdx.x >> 4);
  const int64_t trips = (p.E + nhw - 1) / nhw;  // both halves of a warp make the same number of trips (shuffles below)
  constexpr bool PG = KIND == STAG_NOISE_NORMAL || KIND == STAG_NOISE_UNIFORM;
  float P0[8], P1[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) P0[i] = P1[i] = 0.f;
  for (int64_t it = 0; it < trips; ++it) {
    const int64_t j = hw0 + it * nhw;
    const bool on = j < p.E;
    const int u = on ? __ldg(p.erow + j) : 0;
    const int v = on ? __ldg(p.indices + j) : 0;
    const int e = on ? __ldg(p.eid + j) : 0;
    float t0 = 0.f, t1 = 0.f;
    for (int s = 0; s < p.S; ++s) {
      const uint32_t smp = (uint32_t)(p.sample_base + s);
      const float* xrp = p.xrow + (int64_t)s * p.xr_ss + (int64_t)u * p.ldxr;
      const float* gvp = p.x + (int64_t)s * p.x_ss + (int64_t)v * p.ldx;
      const float* avp = reinterpret_cast<const float*>(arg_in) + (int64_t)s * p.x_ss + (int64_t)v * p.ldx;
      float tw = 0.f;
      if (on) {
        for (int b = hl; b < p.nblk; b += 16) {
          const int c = first_chan(0, b);
          float xr[8], gv[8], av[8], dw[8];
          load8<VEC>(avp, c, p.D, av);
          bool any = false;
#pragma unroll
          for (int i = 0; i < 8; ++i) any |= __float_as_int(av[i]) == e && chan(c, i) < p.D;
          if (any) {
            load8<VEC>(xrp, c, p.D, xr);
            load8<VEC>(gvp, c, p.D, gv);
          }
#pragma unroll
          for (int i = 0; i < 8; ++i)
            dw[i] = (any && __float_as_int(av[i]) == e && chan(c, i) < p.D) ? xr[i] * gv[i] : 0.f;
          if (KIND == STAG_NOISE_EXTERNAL) {
            if (p.K == 1) tw += sum8(dw);
            else store8<VEC, false>(p.dw_ext + ((int64_t)s * p.E + e) * p.K, c, p.D, dw);
          } else if (PG && any) {
            float w[8], raw[8], pre[8];
            max_weights<KIND, VEC>(p, key, s, smp, e, (uint32_t)b, c, P0, P1, w, raw, pre);
            float e0[8], e1[8];
#pragma unroll
            for (int i = 0; i < 8; ++i) {
              const float d = (p.relu && !(pre[i] > 0.f)) ? 0.f : dw[i];
              e1[i] = d * raw[i];
              e0[i] = KIND == STAG_NOISE_NORMAL ? d : d - e1[i];
            }
            t0 += sum8(e0);
            t1 += sum8(e1);
          }
        }
      }
      if (KIND == STAG_NOISE_EXTERNAL && p.K == 1) {
#pragma unroll
        for (int o = 8; o > 0; o >>= 1) tw += __shfl_xor_sync(0xffffffffu, tw, o);
        if (on && hl == 0) p.dw_ext[(int64_t)s * p.E + e] = tw;
      }
    }
    if (PG) {
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

// Checks shared by the two entry points: no in-norm, no [E,K] parameters (both go through the materialised noise).
static int check_max_noise(const StagNoise* n, int D, int64_t E, const char* who) {
  int rc = check_noise(n, D, E, who);
  if (rc) return rc;
  STAG_CHECK_ARG(!n->in_norm, "%s: in_norm is not fused with max (materialise the noise)", who);
  STAG_CHECK_ARG(n->kind <= STAG_NOISE_EXTERNAL || (n->param_shape != STAG_PARAM_EDGE_CHANNEL || n->K == 1),
                 "%s: [E,K] parameters are not fused with max (materialise the noise)", who);
  if (n->kind == STAG_NOISE_NORMAL_HADAMARD)
    STAG_CHECK_ARG(n->K == D, "%s: the Hadamard generator needs K == D (K=%d D=%d)", who, n->K, D);
  return STAG_OK;
}

template <bool BWD>
static int launch_max_row(const AggParams& p, bool vec, const int32_t* arg_in, int32_t* arg_out, int grid, size_t smem,
                          cudaStream_t stream) {
  auto go = [&](auto kern) -> int {
    if (smem > 48 * 1024) STAG_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    kern<<<grid, AGG_THREADS, smem, stream>>>(p, arg_in, arg_out);
    STAG_LAUNCH_CHECK();
    return STAG_OK;
  };
#define STAG_MAX_KIND(K) \
  case K: return vec ? go(max_row_kernel<K, true, BWD>) : go(max_row_kernel<K, false, BWD>);
  switch (p.kind) {
    STAG_MAX_KIND(STAG_NOISE_NONE)
    STAG_MAX_KIND(STAG_NOISE_EXTERNAL)
    STAG_MAX_KIND(STAG_NOISE_NORMAL)
    STAG_MAX_KIND(STAG_NOISE_UNIFORM)
    STAG_MAX_KIND(STAG_NOISE_BERNOULLI)
  }
#undef STAG_MAX_KIND
  set_error("stag_spmm_max: bad kind %d", p.kind);
  return STAG_EINVAL;
}

static int launch_max_wh(const AggParams& p, bool bwd, const int32_t* arg_in, int32_t* arg_out, cudaStream_t stream) {
  const int64_t warps = (int64_t)(p.num_hub_segs + p.N) * (p.D >> 7) * p.S;
  const int64_t ctas = (warps + 7) / 8;
  const int64_t cap = (int64_t)num_sms() * 8;
  const int grid = (int)(ctas < 1 ? 1 : (ctas < cap ? ctas : cap));
  if (bwd) max_wh_kernel<true><<<grid, 256, 0, stream>>>(p, arg_in, arg_out);
  else max_wh_kernel<false><<<grid, 256, 0, stream>>>(p, arg_in, arg_out);
  STAG_LAUNCH_CHECK();
  return STAG_OK;
}

}  // namespace stag

extern "C" int stag_spmm_max_fwd(const StagGraph* g, const float* x, int64_t ldx, int64_t x_sample_stride, int32_t D,
                                 int32_t S, const StagNoise* noise, float* out, int32_t* arg, int64_t ldo,
                                 int64_t out_sample_stride, void* ws, size_t ws_bytes, void* stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  int rc = check_graph(g, "stag_spmm_max_fwd");
  if (rc) return rc;
  STAG_CHECK_ARG(D > 0 && S > 0, "stag_spmm_max_fwd: D=%d S=%d must be positive", D, S);
  STAG_CHECK_ARG(out != nullptr && arg != nullptr, "stag_spmm_max_fwd: null output");
  STAG_CHECK_ARG(x != nullptr || g->num_edges == 0, "stag_spmm_max_fwd: null features");
  STAG_CHECK_ARG(ldx >= D && ldo >= D, "stag_spmm_max_fwd: row strides smaller than D");
  rc = check_max_noise(noise, D, g->num_edges, "stag_spmm_max_fwd");
  if (rc) return rc;
  if (g->num_rows == 0) return STAG_OK;
  const WsLayout L = ws_layout(g, D, S, grid_cap());
  if (!ws || ws_bytes < L.total) {
    set_error("stag_spmm_max_fwd: workspace %zu < required %zu", ws_bytes, L.total);
    return STAG_EWORKSPACE;
  }
  AggParams p = {};
  fill_graph(p, g);
  fill_noise(p, noise, D);
  p.x = x; p.ldx = ldx; p.x_ss = x_sample_stride;
  p.out = out; p.ldo = ldo; p.out_ss = out_sample_stride;
  set_shape(p, D, S, g->num_cols, false, true);
  p.part_acc = (float*)((char*)ws + L.part_acc);
  p.part_w = (float*)((char*)ws + L.part_w);
  bool vec = (D % 4 == 0) && (ldx % 4 == 0) && (ldo % 4 == 0) && (x_sample_stride % 4 == 0) &&
             (out_sample_stride % 4 == 0) && aligned16(x) && aligned16(out) && aligned16(arg);
  if (noise->kind == STAG_NOISE_EXTERNAL && noise->K != 1) vec = vec && aligned16(noise->external);
  if (noise->kind >= STAG_NOISE_NORMAL && p.pshape == STAG_PARAM_CHANNEL)
    vec = vec && aligned16(noise->p0) && (noise->p1 == nullptr || aligned16(noise->p1));
  if (noise->kind == STAG_NOISE_NORMAL_HADAMARD) {
    STAG_CHECK_ARG(vec, "stag_spmm_max_fwd: STAG_NOISE_NORMAL_HADAMARD needs 16-byte aligned rows");
    rc = launch_max_wh(p, false, nullptr, arg, stream);
  } else {
    rc = launch_max_row<false>(p, vec, nullptr, arg, agg_grid(p), 0, stream);
  }
  if (rc) return rc;
  if (g->num_hubs > 0) {
    const int64_t total = (int64_t)S * g->num_hubs * D;
    max_hub_finalize_kernel<<<(unsigned)((total + 255) / 256), 256, 0, stream>>>(p, arg);
    STAG_LAUNCH_CHECK();
  }
  return STAG_OK;
}

extern "C" int stag_spmm_max_bwd(const StagGraph* g, const float* x, int64_t ldx, int64_t x_sample_stride,
                                 const float* dout, const int32_t* arg, int64_t ldg, int64_t dout_sample_stride,
                                 int32_t D, int32_t S, const StagNoise* noise, float* dx, int64_t lddx,
                                 int64_t dx_sample_stride, float* dparam0, float* dparam1, float* dw_external,
                                 void* ws, size_t ws_bytes, void* stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  int rc = check_graph(g, "stag_spmm_max_bwd");
  if (rc) return rc;
  STAG_CHECK_ARG(D > 0 && S > 0, "stag_spmm_max_bwd: D=%d S=%d must be positive", D, S);
  STAG_CHECK_ARG((dout != nullptr && arg != nullptr) || g->num_edges == 0,
                 "stag_spmm_max_bwd: null upstream gradient or argument tensor");
  STAG_CHECK_ARG(ldx >= D && ldg >= D && (dx == nullptr || lddx >= D), "stag_spmm_max_bwd: row strides smaller than D");
  rc = check_max_noise(noise, D, g->num_edges, "stag_spmm_max_bwd");
  if (rc) return rc;
  const bool param_grads = (noise->kind == STAG_NOISE_NORMAL || noise->kind == STAG_NOISE_UNIFORM) && dparam0 != nullptr;
  if (param_grads) STAG_CHECK_ARG(dparam1 != nullptr, "stag_spmm_max_bwd: pass both parameter-gradient outputs");
  const bool ext_grads = noise->kind == STAG_NOISE_EXTERNAL && dw_external != nullptr;
  STAG_CHECK_ARG(x != nullptr || g->num_edges == 0 || !(param_grads || ext_grads), "stag_spmm_max_bwd: null features");
  AggParams p = {};
  fill_graph(p, g);
  fill_noise(p, noise, D);
  const bool edge_params = param_grads && p.pshape == STAG_PARAM_EDGE;
  const bool dense_params = param_grads && !edge_params;
  STAG_CHECK_ARG(!(edge_params || ext_grads) || g->erow != nullptr || g->num_edges == 0,
                 "stag_spmm_max_bwd: per-edge gradients need a graph built with erow");
  if (g->num_rows == 0) {
    if (dense_params) {
      const size_t n = p.pshape == STAG_PARAM_SCALAR ? 1 : (size_t)D;
      STAG_CUDA(cudaMemsetAsync(dparam0, 0, n * 4, stream));
      STAG_CUDA(cudaMemsetAsync(dparam1, 0, n * 4, stream));
    }
    return STAG_OK;
  }
  const WsLayout L = ws_layout(g, D, S, grid_cap());
  if (!ws || ws_bytes < L.total) {
    set_error("stag_spmm_max_bwd: workspace %zu < required %zu", ws_bytes, L.total);
    return STAG_EWORKSPACE;
  }
  // transposed roles: gather dout / arg rows of the destinations, rows are sources
  p.x = dout; p.ldx = ldg; p.x_ss = dout_sample_stride;
  p.out = dx; p.ldo = lddx; p.out_ss = dx_sample_stride;
  p.xrow = x; p.ldxr = ldx; p.xr_ss = x_sample_stride;
  set_shape(p, D, S, g->num_cols, false, true);
  p.dw_ext = ext_grads ? dw_external : nullptr;
  p.part_acc = (float*)((char*)ws + L.part_acc);
  p.dp_partial = (float*)((char*)ws + L.dp_partial);
  bool vec = (D % 4 == 0) && (ldg % 4 == 0) && (dout_sample_stride % 4 == 0) && aligned16(dout) && aligned16(arg);
  if (dx) vec = vec && (lddx % 4 == 0) && (dx_sample_stride % 4 == 0) && aligned16(dx);
  if (param_grads || ext_grads) vec = vec && (ldx % 4 == 0) && (x_sample_stride % 4 == 0) && aligned16(x);
  if (noise->kind == STAG_NOISE_EXTERNAL && noise->K != 1)
    vec = vec && aligned16(noise->external) && (dw_external == nullptr || aligned16(dw_external));
  if (noise->kind >= STAG_NOISE_NORMAL && p.pshape == STAG_PARAM_CHANNEL)
    vec = vec && aligned16(noise->p0) && (noise->p1 == nullptr || aligned16(noise->p1));
  // dX and the scalar / per-channel parameter gradients: the CSR walk
  const int grid = agg_grid(p);
  if (dx || dense_params) {
    AggParams q = p;
    q.dp0 = dense_params ? dparam0 : nullptr;
    q.dp1 = dense_params ? dparam1 : nullptr;
    const size_t smem = dense_params ? (size_t)AGG_WARPS * 2 * p.dpad * sizeof(float) : 0;
    if (smem > 200 * 1024) {
      set_error("stag_spmm_max_bwd: D=%d too wide for the shared-memory parameter-gradient staging", D);
      return STAG_EUNSUPPORTED;
    }
    if (noise->kind == STAG_NOISE_NORMAL_HADAMARD) {
      STAG_CHECK_ARG(vec, "stag_spmm_max_bwd: STAG_NOISE_NORMAL_HADAMARD needs 16-byte aligned rows");
      rc = launch_max_wh(q, true, arg, nullptr, stream);
    } else {
      rc = launch_max_row<true>(q, vec, arg, nullptr, grid, smem, stream);
    }
    if (rc) return rc;
    if (g->num_hubs > 0 && dx) {
      const int64_t total = (int64_t)S * g->num_hubs * D;
      hub_finalize_kernel<<<(unsigned)((total + 255) / 256), 256, 0, stream>>>(q, 1);
      STAG_LAUNCH_CHECK();
    }
    if (dense_params) {
      const int scalar = p.pshape == STAG_PARAM_SCALAR;
      param_finalize_kernel<<<scalar ? 1 : (D + 255) / 256, 256, 0, stream>>>(p.dp_partial, grid, p.dpad, D, scalar,
                                                                            dparam0, dparam1);
      STAG_LAUNCH_CHECK();
    }
  }
  // dw_external and the per-edge parameter gradients: edge-parallel
  if ((edge_params || ext_grads) && p.E > 0) {
    AggParams q = p;
    q.dp0 = edge_params ? dparam0 : nullptr;
    q.dp1 = edge_params ? dparam1 : nullptr;
    const int64_t want = (p.E + 15) / 16;
    const int egrid = (int)(want < (int64_t)num_sms() * 16 ? want : (int64_t)num_sms() * 16);
    auto go = [&](auto kern) { kern<<<egrid, 256, 0, stream>>>(q, arg); };
    if (ext_grads) { if (vec) go(max_edge_kernel<STAG_NOISE_EXTERNAL, true>); else go(max_edge_kernel<STAG_NOISE_EXTERNAL, false>); }
    else if (noise->kind == STAG_NOISE_NORMAL) { if (vec) go(max_edge_kernel<STAG_NOISE_NORMAL, true>); else go(max_edge_kernel<STAG_NOISE_NORMAL, false>); }
    else { if (vec) go(max_edge_kernel<STAG_NOISE_UNIFORM, true>); else go(max_edge_kernel<STAG_NOISE_UNIFORM, false>); }
    STAG_LAUNCH_CHECK();
  }
  return STAG_OK;
}
