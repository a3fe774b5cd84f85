// Dense feature transform  out = act(row_scale * (A @ W) + bias)  on the 5th-generation tensor
// cores (tcgen05.mma, accumulator in TMEM), fp32 in / fp32 out at fp32-level accuracy by the
// 3xTF32 split  A*W ~= A_hi*W_hi + A_lo*W_hi + A_hi*W_lo  (hi = tf32(x), lo = tf32(x - hi)).
//
// Replaces  rst = th.matmul(rst, weight)  [+ dst-norm, bias, activation]  of the reference's
// GCN.forward (stag/zoo/gcn.py:97-114) and the fc_neigh / fc_self Linear layers of GraphSAGE
// (stag/zoo/graph_sage.py:74-75,91,107).
//
// Two kernels:
//   gemm_tma_kernel      persistent, one CTA of 10 warps per SM, W_hi / W_lo of every K block resident in shared memory,
//                        A tiles by TMA into a ring, split / MMA / epilogue in separate warps, two TMEM accumulators
//                        (taken when rows of A are 16-byte aligned and W fits: the layer shapes; see further down);
//   gemm_tcgen05_kernel  the first form, below: one CTA (4 warps) owns a 128-row tile of A and ALL output columns
//                        (N <= 256); with few row tiles and a long K (Cora: 2 708 x 1 433 x 16) the K blocks of one row
//                        tile are split over a thread-block cluster and added in rank 0's shared memory (DSMEM).
// First form, per K block of 32 floats:  threads load the A tile and the W^T tile with 128-bit loads, split
//   them into hi / lo parts and store them into shared memory in the canonical K-major
//   SWIZZLE_128B layout (rows of 128 bytes, 16-byte chunks XOR-ed with row % 8);  one elected
//   thread issues 4 k-steps x 3 tcgen05.mma (kind::tf32, M = 128, N = Npad, K = 8) accumulating
//   into TMEM;  tcgen05.commit -> mbarrier releases the shared tiles.
//   epilogue: each warp reads its 32 TMEM lanes (tcgen05.ld 32x32b.x32), applies row scale, bias,
//   activation and writes 128-byte row segments.
// Two CTAs of the first form are resident per SM (96 KB of shared memory each), which overlaps one CTA's loads with
// the other's MMAs.  Timings and the ncu reading: profiles/r02_gemm.txt.
#include <cuda.h>  // CUtensorMap: types only, the encoder comes from cudaGetDriverEntryPoint
#include <stdlib.h>

#include "common.cuh"

namespace stag {

constexpr int GM = 128;       // rows per CTA tile (UMMA M)
constexpr int GK = 32;        // floats per K block = one 128-byte swizzle row
constexpr int GTHREADS = 128;

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

// relu that leaves NaN as NaN, as torch.relu does (fmaxf(NaN, 0) is 0: a diverged row would come out as zeros)
__device__ __forceinline__ float relu_keep_nan(float y) { return y < 0.f ? 0.f : y; }

__device__ __forceinline__ float to_tf32(float x) {
  uint32_t y;
  asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(y) : "f"(x));
  return __uint_as_float(y);
}

// K-major SWIZZLE_128B shared-memory matrix descriptor (cute::UMMA::SmemDescriptor):
//   bits [0,14) start address >> 4, [16,30) leading byte offset >> 4 (1 for swizzled K-major),
//   [32,46) stride byte offset >> 4 (8 rows x 128 B = 1024 B -> 64), [46,48) version = 1,
//   [61,64) layout type = 2 (SWIZZLE_128B)
__device__ __forceinline__ uint64_t make_desc(uint32_t saddr) {
  return (uint64_t)((saddr & 0x3FFFFu) >> 4) | (1ull << 16) | (64ull << 32) | (1ull << 46) | (2ull << 61);
}

// instruction descriptor (cute::UMMA::InstrDescriptor), kind::tf32, fp32 accumulate, A and B K-major
__device__ __forceinline__ uint32_t make_idesc(int n) {
  return (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(GM >> 4) << 24);
}

__device__ __forceinline__ void mma_tf32(uint32_t tmem_d, uint64_t da, uint64_t db, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_d), "l"(da), "l"(db), "r"(idesc), "r"(accumulate)
      : "memory");
}

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
// bounded spin: a lost arrival must become an error, never a hung GPU
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  uint32_t done = 0;
  for (uint32_t spin = 0; !done; ++spin) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(done)
        : "r"(smem_u32(bar)), "r"(parity)
        : "memory");
    if (spin > (1u << 24)) __trap();
  }
}

struct GemmParams {
  const float* a;
  int64_t lda;
  const float* wt;  // [Nout, K] row-major (W transposed)
  int64_t ldw;
  int64_t M;
  int Nout, K, npad;  // npad: Nout rounded up to a multiple of 16 (UMMA N)
  const float* row_scale;
  const float* bias;
  int act;
  float* out;
  int64_t ldo;
  uint32_t tmem_cols;
  int ksplit;  // > 1: a cluster of ksplit CTAs (blockIdx.x) shares one row tile (blockIdx.y), each taking a range of K blocks
};

// store one 16-byte chunk (4 floats) of row r, chunk index ch (0..7) of a [rows][32] tile, split hi/lo
__device__ __forceinline__ void put_split(float* hi, float* lo, int r, int ch, float4 v) {
  const int o = r * GK + ((ch ^ (r & 7)) << 2);
  float4 h, l;
  h.x = to_tf32(v.x); h.y = to_tf32(v.y); h.z = to_tf32(v.z); h.w = to_tf32(v.w);
  l.x = to_tf32(v.x - h.x); l.y = to_tf32(v.y - h.y); l.z = to_tf32(v.z - h.z); l.w = to_tf32(v.w - h.w);
  *reinterpret_cast<float4*>(hi + o) = h;
  *reinterpret_cast<float4*>(lo + o) = l;
}

__device__ __forceinline__ float4 load_row4(const float* base, int64_t ld, int64_t r, int64_t nrows, int k, int K,
                                            bool vec) {
  float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
  if (r < nrows) {
    const float* p = base + r * ld + k;
    if (vec && k + 3 < K) {
      v = __ldg(reinterpret_cast<const float4*>(p));
    } else {
      if (k + 0 < K) v.x = __ldg(p + 0);
      if (k + 1 < K) v.y = __ldg(p + 1);
      if (k + 2 < K) v.z = __ldg(p + 2);
      if (k + 3 < K) v.w = __ldg(p + 3);
    }
  }
  return v;
}

__global__ void __launch_bounds__(GTHREADS) gemm_tcgen05_kernel(const GemmParams p) {
  extern __shared__ __align__(1024) unsigned char gsm_raw[];
  // 1024-byte aligned tiles (SWIZZLE_128B atoms are 8 rows x 128 B)
  unsigned char* gsm = reinterpret_cast<unsigned char*>(((uintptr_t)gsm_raw + 1023) & ~(uintptr_t)1023);
  float* a_hi = reinterpret_cast<float*>(gsm);
  float* a_lo = a_hi + GM * GK;
  float* w_hi = a_lo + GM * GK;
  float* w_lo = w_hi + 256 * GK;
  __shared__ uint64_t mma_bar;
  __shared__ uint32_t tmem_base_s;

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int krank = p.ksplit > 1 ? (int)blockIdx.x : 0;
  const int64_t m0 = (int64_t)(p.ksplit > 1 ? blockIdx.y : blockIdx.x) * GM;
  const bool vec_a = (p.lda % 4 == 0) && (((uintptr_t)p.a & 15) == 0);
  const bool vec_w = (p.ldw % 4 == 0) && (((uintptr_t)p.wt & 15) == 0);
  const bool vec_o = (p.ldo % 4 == 0) && (((uintptr_t)p.out & 15) == 0);

  if (warp == 0) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&tmem_base_s)),
                 "r"(p.tmem_cols)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  if (tid == 0) {
    mbar_init(&mma_bar, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  const uint32_t tmem_d = tmem_base_s;
  const uint32_t idesc = make_idesc(p.npad);

  const int nkb = (p.K + GK - 1) / GK;
  uint32_t phase = 0;
  // register staging of the NEXT K block: its global loads are in flight while the tensor core works on
  // the current one (A: 8 x 128-bit per thread; W^T: the first 128 rows, wider tiles load the rest late)
  float4 va[8], vw[8];
  auto load_tiles = [&](int kb) {
    const int k0 = kb * GK;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const int i = tid + j * GTHREADS;
      va[j] = load_row4(p.a, p.lda, m0 + (i >> 3), p.M, k0 + (i & 7) * 4, p.K, vec_a);
    }
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const int i = tid + j * GTHREADS;
      vw[j] = load_row4(p.wt, p.ldw, i < p.npad * 8 ? (i >> 3) : p.Nout, p.Nout, k0 + (i & 7) * 4, p.K, vec_w);
    }
  };
  const int kb_lo = p.ksplit > 1 ? krank * nkb / p.ksplit : 0, kb_hi = p.ksplit > 1 ? (krank + 1) * nkb / p.ksplit : nkb;
  load_tiles(kb_lo);
  for (int kb = kb_lo; kb < kb_hi; ++kb) {
    const int k0 = kb * GK;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const int i = tid + j * GTHREADS;
      put_split(a_hi, a_lo, i >> 3, i & 7, va[j]);
      if (i < p.npad * 8) put_split(w_hi, w_lo, i >> 3, i & 7, vw[j]);
    }
    for (int i0 = 8 * GTHREADS; i0 < p.npad * 8; i0 += 8 * GTHREADS) {  // W^T rows 128.. (Nout > 128)
      float4 v[8];
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const int i = i0 + tid + j * GTHREADS;
        v[j] = load_row4(p.wt, p.ldw, i < p.npad * 8 ? (i >> 3) : p.Nout, p.Nout, k0 + (i & 7) * 4, p.K, vec_w);
      }
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const int i = i0 + tid + j * GTHREADS;
        if (i < p.npad * 8) put_split(w_hi, w_lo, i >> 3, i & 7, v[j]);
      }
    }
    // generic-proxy writes -> visible to the tensor core's async proxy
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    __syncthreads();
    if (warp == 0 && lane == 0) {
      asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
      const uint64_t dah = make_desc(smem_u32(a_hi)), dal = make_desc(smem_u32(a_lo));
      const uint64_t dwh = make_desc(smem_u32(w_hi)), dwl = make_desc(smem_u32(w_lo));
#pragma unroll
      for (int ks = 0; ks < GK / 8; ++ks) {
        const uint64_t adv = (uint64_t)(ks * 2);  // 8 tf32 = 32 bytes = 2 x 16 B along K
        mma_tf32(tmem_d, dah + adv, dwh + adv, idesc, ((kb - kb_lo) | ks) != 0);
        mma_tf32(tmem_d, dal + adv, dwh + adv, idesc, 1);
        mma_tf32(tmem_d, dah + adv, dwl + adv, idesc, 1);
      }
      // arrives on the mbarrier when all MMAs issued so far have completed (implies the fence)
      asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(
                       smem_u32(&mma_bar))
                   : "memory");
    }
    if (kb + 1 < kb_hi) load_tiles(kb + 1);
    // the shared tiles may be overwritten (and, after the last block, TMEM read) once the MMAs are done
    mbar_wait(&mma_bar, phase);
    phase ^= 1;
  }
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");

  // ---- epilogue: warp w owns TMEM lanes (= tile rows) 32w .. 32w+31 -------------------------------------
  // TMEM gives a thread one row x 32 columns; a per-warp shared scratch (pitch 33) transposes that so
  // that every store instruction writes four full 128-byte row segments
  float* scratch = a_hi + warp * (32 * 33);  // the operand tiles are free now
  // split-K (small M, long K: Cora's 2 708 x 1 433 x 16 is 22 row tiles of 45 K blocks): the CTAs of a cluster hold
  // partial accumulators of ONE row tile.  Ranks > 0 write theirs into rank 0's shared memory (DSMEM), rank 0 adds
  // them in rank order -- deterministic -- and runs the epilogue.
  float* part = a_hi + 4 * (32 * 33) + 32;  // [ksplit - 1][128][npad] behind the scratch (rank 0's copy is the target)
  if (p.ksplit > 1) {
    // every CTA of the cluster is done with its MMAs: rank 0's operand tiles may be overwritten
    asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
    if (krank > 0) {
      uint32_t remote;
      asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(remote) : "r"(smem_u32(part)), "r"(0));
      remote += (uint32_t)(((krank - 1) * GM + warp * 32 + lane) * p.npad) * 4u;
      for (int n0 = 0; n0 < p.npad; n0 += 16) {
        uint32_t v[16];
        const uint32_t taddr = tmem_d + ((uint32_t)(warp * 32) << 16) + (uint32_t)n0;
        asm volatile(
            "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
            "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
            : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
              "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
            : "r"(taddr)
            : "memory");
        asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
        for (int j = 0; j < 16; j += 4)
          asm volatile("st.shared::cluster.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(remote + (uint32_t)(n0 + j) * 4u), "r"(v[j]),
                       "r"(v[j + 1]), "r"(v[j + 2]), "r"(v[j + 3])
                       : "memory");
      }
    }
    asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
  }
  const int64_t row = m0 + warp * 32 + lane;
  const float rs = (p.row_scale && row < p.M) ? __ldg(p.row_scale + row) : 1.0f;
  for (int n0 = 0; n0 < p.npad && krank == 0; n0 += 32) {
    uint32_t v[32];
    const uint32_t taddr = tmem_d + ((uint32_t)(warp * 32) << 16) + (uint32_t)n0;
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
          "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]),
          "=r"(v[16]), "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]),
          "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
        : "r"(taddr)
        : "memory");
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
    for (int r = 1; r < p.ksplit; ++r) {   // the other ranks' partial sums of this row, in rank order
      const float* pr = part + (size_t)((r - 1) * GM + warp * 32 + lane) * p.npad + n0;
#pragma unroll
      for (int j = 0; j < 32; j += 4) {
        if (n0 + j < p.npad) {
          const float4 t = *reinterpret_cast<const float4*>(pr + j);
          v[j] = __float_as_uint(__uint_as_float(v[j]) + t.x);
          v[j + 1] = __float_as_uint(__uint_as_float(v[j + 1]) + t.y);
          v[j + 2] = __float_as_uint(__uint_as_float(v[j + 2]) + t.z);
          v[j + 3] = __float_as_uint(__uint_as_float(v[j + 3]) + t.w);
        }
      }
    }
    __syncwarp();  // the previous chunk's readers are done with the scratch
#pragma unroll
    for (int j = 0; j < 32; ++j) {
      float y = __uint_as_float(v[j]) * rs;
      if (p.bias && n0 + j < p.Nout) y += __ldg(p.bias + n0 + j);
      if (p.act == 1) y = relu_keep_nan(y);
      scratch[lane * 33 + j] = y;
    }
    __syncwarp();
    const int cq = (lane & 7) * 4;
#pragma unroll
    for (int r = 0; r < 32; r += 4) {
      const int rr = r + (lane >> 3);
      const int64_t grow = m0 + warp * 32 + rr;
      if (grow < p.M) {
        const float* sp = scratch + rr * 33 + cq;
        float* o = p.out + grow * p.ldo + n0 + cq;
        if (vec_o && n0 + cq + 3 < p.Nout) {
          *reinterpret_cast<float4*>(o) = make_float4(sp[0], sp[1], sp[2], sp[3]);
        } else {
#pragma unroll
          for (int j = 0; j < 4; ++j)
            if (n0 + cq + j < p.Nout) o[j] = sp[j];
        }
      }
    }
  }

  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  if (warp == 0) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_d), "r"(p.tmem_cols) : "memory");
  }
}

// ---- second form: persistent CTAs, W resident in shared memory, A tiles by TMA ------------------------------------
// For the memory-bound layer shapes (arxiv: M = S N = 2.7 M rows, K = N = 128: 1.39 GB in, 1.39 GB out, 0.09 TFLOP) the
// first form re-splits the W tile for every row tile and K block and moves A through registers with one K block in
// flight.  Here a CTA per SM keeps W_hi / W_lo of ALL K blocks in shared memory (swizzled once), and a ring of
// [128 x 32] fp32 A tiles (sized at run time: what fits beside W, 3 at K = N = 128) is filled by TMA
// (cp.async.bulk.tensor.2d, SWIZZLE_128B: the tile lands in the canonical K-major layout the MMA reads) -- roles:
//   warp 0   one thread: waits for a free ring slot, arms its mbarrier with the tile's bytes, issues the TMA load;
//   warps 2-5  when a tile has landed: kind::tf32 reads the upper 19 bits of a 32-bit container, so the tile as delivered
//            IS the hi operand; these warps only make lo = tf32(x - trunc(x)) into a second ring (2-3 tiles),
//            fence.proxy.async, arrive on `ready`;
//   warp 1   one thread: waits for `ready`, issues 4 k-steps x 3 tcgen05.mma (A_hi W_hi + A_lo W_hi + A_hi W_lo) into
//            TMEM accumulator [tile & 1]; tcgen05.commit -> `empty` (raw slot reusable) and `lo_free`, and after the
//            last K block of a row tile -> `acc_full`;
//   warps 6-9  epilogue of a finished row tile from its TMEM accumulator while the other one is being filled: 32x32b
//            loads (the next 32 columns in flight), row scale, XOR-swizzled scratch, bias, relu, STG.128 of four
//            128-byte row segments per instruction; `acc_empty` right after the last TMEM read.
// (With the split warps also running the epilogue the pipeline drained during every epilogue: 1.75 ms; with a thread
// storing its own row: 1.48 ms; now 0.56 - 0.60 ms, profiles/r02_gemm.txt.)
// Out-of-range rows / columns of A are zero-filled by the TMA unit (the tensor map knows M and K).
constexpr int G2_THREADS = 320;  // warp 0 TMA, warp 1 MMA, warps 2-5 split, warps 6-9 epilogue
constexpr int G2_MAXST = 8;      // ring sizes are run-time (what fits beside the resident W): at most 8 raw / 8 lo tiles
constexpr uint32_t G2_TILE = GM * GK * 4;  // 16 KB

struct Gemm2Params {
  const float* wt;  // [Nout, K] row-major (W transposed)
  int64_t ldw;
  int64_t M, ntiles;
  int Nout, K, npad, nkb;
  const float* row_scale;
  const float* bias;
  int act;
  float* out;
  int64_t ldo;
  uint32_t ncol;  // TMEM columns per accumulator (power of two >= npad)
  uint32_t nst, nlo;  // raw-tile ring (TMA targets, hi in place) and lo-tile ring
};

__device__ __forceinline__ void mbar_wait_s(uint32_t bar, uint32_t parity) {
  uint32_t done = 0;
  for (uint32_t spin = 0; !done; ++spin) {
    asm volatile(
        "{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(done)
        : "r"(bar), "r"(parity)
        : "memory");
    if (spin > (1u << 24)) __trap();  // a lost arrival becomes an error, never a hung GPU
  }
}
__device__ __forceinline__ void mbar_arrive_s(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}

__global__ void __launch_bounds__(G2_THREADS, 1) gemm_tma_kernel(const __grid_constant__ CUtensorMap tmap, const Gemm2Params p) {
  extern __shared__ __align__(1024) unsigned char gsm_raw[];
  __shared__ uint64_t bars[4 * G2_MAXST + 4];  // full[], ready[], empty[], lo_free[], acc_full[2], acc_empty[2]
  __shared__ uint32_t tmem_base_s;
  const uint32_t sm0 = (smem_u32(gsm_raw) + 1023u) & ~1023u;
  const uint32_t wtile = (uint32_t)p.npad * 128u;              // one K block of W: npad rows x 128 bytes
  const uint32_t w_hi = sm0, w_lo = sm0 + (uint32_t)p.nkb * wtile;
  const uint32_t st0 = w_lo + (uint32_t)p.nkb * wtile;         // raw / hi tiles: st0 + s TILE (ring of nst, TMA targets)
  const uint32_t lo0 = st0 + p.nst * G2_TILE;                   // lo tiles: lo0 + l TILE (ring of nlo, made just before the MMAs)
  const uint32_t scr0 = lo0 + p.nlo * G2_TILE;                  // epilogue transposition scratch: 4 warps x [32][32] floats
  const uint32_t bar0 = smem_u32(bars);
  auto FULL = [&](int s) { return bar0 + 8u * s; };
  auto READY = [&](int s) { return bar0 + 8u * (G2_MAXST + s); };
  auto EMPTY = [&](int s) { return bar0 + 8u * (2 * G2_MAXST + s); };
  auto LO_FREE = [&](int l) { return bar0 + 8u * (3 * G2_MAXST + l); };
  auto ACC_FULL = [&](int a) { return bar0 + 8u * (4 * G2_MAXST + a); };
  auto ACC_EMPTY = [&](int a) { return bar0 + 8u * (4 * G2_MAXST + 2 + a); };
  // ring cursors: slot + pass parity, advanced without a division
  struct Ring {
    uint32_t i, par, n;
    __device__ void next() { if (++i == n) { i = 0; par ^= 1u; } }
  };
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;

  if (warp == 0) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&tmem_base_s)),
                 "r"(2u * p.ncol)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  if (tid == 0) {
    for (int s = 0; s < G2_MAXST; ++s) {
      asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(FULL(s)) : "memory");
      asm volatile("mbarrier.init.shared::cta.b64 [%0], 4;" ::"r"(READY(s)) : "memory");
      asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(EMPTY(s)) : "memory");
      asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(LO_FREE(s)) : "memory");
    }
    for (int a = 0; a < 2; ++a) {
      asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(ACC_FULL(a)) : "memory");
      asm volatile("mbarrier.init.shared::cta.b64 [%0], 4;" ::"r"(ACC_EMPTY(a)) : "memory");
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  // W^T -> hi / lo, every K block, canonical K-major SWIZZLE_128B tiles (once per CTA)
  {
    const bool vec_w = (p.ldw % 4 == 0) && (((uintptr_t)p.wt & 15) == 0);
    const int per_kb = p.npad * 8;  // 16-byte chunks per K block
    for (int i = tid; i < p.nkb * per_kb; i += G2_THREADS) {
      const int kb = i / per_kb, j = i - kb * per_kb, r = j >> 3, ch = j & 7;
      const float4 v = load_row4(p.wt, p.ldw, r, p.Nout, kb * GK + ch * 4, p.K, vec_w);
      float4 h, l;
      h.x = to_tf32(v.x); h.y = to_tf32(v.y); h.z = to_tf32(v.z); h.w = to_tf32(v.w);
      l.x = to_tf32(v.x - h.x); l.y = to_tf32(v.y - h.y); l.z = to_tf32(v.z - h.z); l.w = to_tf32(v.w - h.w);
      const uint32_t o = (uint32_t)kb * wtile + (uint32_t)r * 128u + (uint32_t)((ch ^ (r & 7)) << 4);
      asm volatile("st.shared.v4.f32 [%0], {%1,%2,%3,%4};" ::"r"(w_hi + o), "f"(h.x), "f"(h.y), "f"(h.z), "f"(h.w) : "memory");
      asm volatile("st.shared.v4.f32 [%0], {%1,%2,%3,%4};" ::"r"(w_lo + o), "f"(l.x), "f"(l.y), "f"(l.z), "f"(l.w) : "memory");
    }
  }
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  const uint32_t tmem_d = tmem_base_s;

  if (warp == 0) {
    // ---------------- TMA producer ----------------
    if (lane == 0) {
      Ring st{0, 0, p.nst};
      bool first_pass = true;
      for (int64_t tile = blockIdx.x; tile < p.ntiles; tile += gridDim.x)
        for (int kb = 0; kb < p.nkb; ++kb) {
          const uint32_t s = st.i;
          if (!first_pass) mbar_wait_s(EMPTY(s), st.par ^ 1u);   // the MMAs of the previous pass over this slot are done
          st.next();
          if (st.i == 0) first_pass = false;
          asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(FULL(s)), "r"(G2_TILE) : "memory");
          asm volatile(
              "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];" ::"r"(
                  st0 + s * G2_TILE),
              "l"(reinterpret_cast<uint64_t>(&tmap)), "r"(kb * GK), "r"((int)(tile * GM)), "r"(FULL(s))
              : "memory");
        }
    }
  } else if (warp == 1) {
    // ---------------- MMA issuer ----------------
    if (lane == 0) {
      const uint32_t idesc = make_idesc(p.npad);
      uint32_t tc = 0;
      Ring st{0, 0, p.nst}, lo{0, 0, p.nlo};
      for (int64_t tile = blockIdx.x; tile < p.ntiles; tile += gridDim.x, ++tc) {
        const uint32_t a = tc & 1u;
        if (tc >= 2) mbar_wait_s(ACC_EMPTY(a), ((tc >> 1) - 1u) & 1u);  // the epilogue has read this accumulator out
        for (int kb = 0; kb < p.nkb; ++kb) {
          const uint32_t s = st.i, l = lo.i;
          mbar_wait_s(READY(s), st.par);
          st.next();
          lo.next();
          asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
          const uint64_t dah = make_desc(st0 + s * G2_TILE), dal = make_desc(lo0 + l * G2_TILE);
          const uint64_t dwh = make_desc(w_hi + (uint32_t)kb * wtile), dwl = make_desc(w_lo + (uint32_t)kb * wtile);
#pragma unroll
          for (int ks = 0; ks < GK / 8; ++ks) {
            const uint64_t adv = (uint64_t)(ks * 2);
            mma_tf32(tmem_d + a * p.ncol, dah + adv, dwh + adv, idesc, (kb | ks) != 0);
            mma_tf32(tmem_d + a * p.ncol, dal + adv, dwh + adv, idesc, 1);
            mma_tf32(tmem_d + a * p.ncol, dah + adv, dwl + adv, idesc, 1);
          }
          asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(EMPTY(s)) : "memory");
          asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(LO_FREE(l)) : "memory");
        }
        asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(ACC_FULL(a)) : "memory");
      }
    }
  } else {
    // ---------------- split warps (2-5) and epilogue warps (6-9) ----------------
    const int q = warp & 3;   // TMEM lane quadrant an epilogue warp may read
    const bool vec_o = (p.ldo % 4 == 0) && (((uintptr_t)p.out & 15) == 0);
    const bool vec_b = (((uintptr_t)p.bias & 15) == 0);
    auto sts128 = [](uint32_t addr, float x, float y, float z, float w) {
      asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "f"(x), "f"(y), "f"(z), "f"(w) : "memory");
    };
    // TMEM hands a thread one row x 32 columns; the per-warp scratch turns that around so that every store
    // instruction writes four full 128-byte row segments (a thread storing its own row touches 32 lines per
    // instruction: the first cut of this kernel spent 1.0 of its 1.48 ms there).  16-byte columns are XORed with
    // the row, so both the row-wise STS.128 and the segment-wise LDS.128 are conflict free.  The TMEM load of the
    // next 32 columns is in flight while this chunk goes through the scratch.
    const uint32_t scr = scr0 + (uint32_t)((warp - 6) & 3) * (32u * 32u * 4u);
    const int c4 = lane & 7, cq = c4 * 4;
    auto ldtm = [&](uint32_t (&v)[32], uint32_t taddr) {
      asm volatile(
          "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
          "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
          "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
          : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
            "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]),
            "=r"(v[16]), "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]),
            "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
          : "r"(taddr)
          : "memory");
    };
    auto chunk_out = [&](const uint32_t (&v)[32], int64_t tile, int n0, float rs) {
      float4 b4 = make_float4(0.f, 0.f, 0.f, 0.f);
      if (p.bias) {
        if (vec_b && n0 + cq + 3 < p.Nout) {
          b4 = __ldg(reinterpret_cast<const float4*>(p.bias + n0 + cq));
        } else {
          if (n0 + cq + 0 < p.Nout) b4.x = __ldg(p.bias + n0 + cq + 0);
          if (n0 + cq + 1 < p.Nout) b4.y = __ldg(p.bias + n0 + cq + 1);
          if (n0 + cq + 2 < p.Nout) b4.z = __ldg(p.bias + n0 + cq + 2);
          if (n0 + cq + 3 < p.Nout) b4.w = __ldg(p.bias + n0 + cq + 3);
        }
      }
      __syncwarp();  // the previous chunk's readers are done with the scratch
#pragma unroll
      for (int c = 0; c < 8; ++c)
        sts128(scr + (uint32_t)(lane * 32 + ((c ^ (lane & 7)) << 2)) * 4u, __uint_as_float(v[4 * c]) * rs,
               __uint_as_float(v[4 * c + 1]) * rs, __uint_as_float(v[4 * c + 2]) * rs, __uint_as_float(v[4 * c + 3]) * rs);
      __syncwarp();
      float4 y[8];
#pragma unroll
      for (int r8 = 0; r8 < 8; ++r8) {
        const int rr = 4 * r8 + (lane >> 3);
        asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];"
                     : "=f"(y[r8].x), "=f"(y[r8].y), "=f"(y[r8].z), "=f"(y[r8].w)
                     : "r"(scr + (uint32_t)(rr * 32 + ((c4 ^ (rr & 7)) << 2)) * 4u));
      }
#pragma unroll
      for (int r8 = 0; r8 < 8; ++r8) {
        const int64_t grow = tile * GM + 32 * q + 4 * r8 + (lane >> 3);
        if (grow < p.M) {
          float4 o4 = make_float4(y[r8].x + b4.x, y[r8].y + b4.y, y[r8].z + b4.z, y[r8].w + b4.w);
          if (p.act == 1) { o4.x = relu_keep_nan(o4.x); o4.y = relu_keep_nan(o4.y); o4.z = relu_keep_nan(o4.z); o4.w = relu_keep_nan(o4.w); }
          float* o = p.out + grow * p.ldo + n0 + cq;
          if (vec_o && n0 + cq + 3 < p.Nout) {
            *reinterpret_cast<float4*>(o) = o4;
          } else {
            if (n0 + cq + 0 < p.Nout) o[0] = o4.x;
            if (n0 + cq + 1 < p.Nout) o[1] = o4.y;
            if (n0 + cq + 2 < p.Nout) o[2] = o4.z;
            if (n0 + cq + 3 < p.Nout) o[3] = o4.w;
          }
        }
      }
    };
    auto epilogue = [&](int64_t tile, uint32_t tc) {
      const uint32_t a = tc & 1u;
      mbar_wait_s(ACC_FULL(a), (tc >> 1) & 1u);
      asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
      const int64_t row = tile * GM + 32 * q + lane;
      const float rs = (p.row_scale && row < p.M) ? __ldg(p.row_scale + row) : 1.0f;
      const uint32_t tbase = tmem_d + ((uint32_t)(32 * q) << 16) + a * p.ncol;
      auto release = [&]() {   // every read of this accumulator has landed: hand it back before the stores
        asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
        __syncwarp();
        if (lane == 0) mbar_arrive_s(ACC_EMPTY(a));
      };
      uint32_t va[32], vb[32];
      ldtm(va, tbase);
      for (int n0 = 0; n0 < p.npad; n0 += 64) {
        asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
        const bool more1 = n0 + 32 < p.npad;
        if (more1) ldtm(vb, tbase + (uint32_t)(n0 + 32)); else release();
        chunk_out(va, tile, n0, rs);
        if (more1) {
          asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
          const bool more2 = n0 + 64 < p.npad;
          if (more2) ldtm(va, tbase + (uint32_t)(n0 + 64)); else release();
          chunk_out(vb, tile, n0 + 32, rs);
        }
      }
    };
    if (warp >= 6) {
      uint32_t tc = 0;
      for (int64_t tile = blockIdx.x; tile < p.ntiles; tile += gridDim.x, ++tc) epilogue(tile, tc);
    } else {
      const int w = warp - 2;   // rows 32 w .. of an A tile
      Ring st{0, 0, p.nst}, lo{0, 0, p.nlo};
      bool lo_first = true;
      for (int64_t tile = blockIdx.x; tile < p.ntiles; tile += gridDim.x) {
        for (int kb = 0; kb < p.nkb; ++kb) {
          const uint32_t s = st.i, l = lo.i;
          mbar_wait_s(FULL(s), st.par);
          if (!lo_first) mbar_wait_s(LO_FREE(l), lo.par ^ 1u);   // the MMAs that read this lo tile one pass ago are done
          st.next();
          lo.next();
          if (lo.i == 0) lo_first = false;
          const uint32_t hi_s = st0 + s * G2_TILE, lo_s = lo0 + l * G2_TILE;
          // kind::tf32 reads the upper 19 bits of each 32-bit container, so the tile as TMA delivered it already IS
          // the hi operand (x with its low 13 mantissa bits dropped); only lo = tf32(x - hi) has to be made.  All
          // eight loads first: the tile is read-only for these warps, nothing orders them behind the stores.
          uint32_t x[8][4];
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            const int idx = lane + 32 * j, r = 32 * w + (idx >> 3), ch = idx & 7;
            const uint32_t o = (uint32_t)r * 128u + (uint32_t)((ch ^ (r & 7)) << 4);
            asm volatile("ld.shared.v4.b32 {%0,%1,%2,%3}, [%4];" : "=r"(x[j][0]), "=r"(x[j][1]), "=r"(x[j][2]), "=r"(x[j][3]) : "r"(hi_s + o));
          }
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            const int idx = lane + 32 * j, r = 32 * w + (idx >> 3), ch = idx & 7;
            const uint32_t o = (uint32_t)r * 128u + (uint32_t)((ch ^ (r & 7)) << 4);
            float l4[4];
#pragma unroll
            for (int t = 0; t < 4; ++t) l4[t] = to_tf32(__uint_as_float(x[j][t]) - __uint_as_float(x[j][t] & 0xFFFFE000u));
            asm volatile("st.shared.v4.f32 [%0], {%1,%2,%3,%4};" ::"r"(lo_s + o), "f"(l4[0]), "f"(l4[1]), "f"(l4[2]), "f"(l4[3]) : "memory");
          }
          asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
          __syncwarp();
          if (lane == 0) mbar_arrive_s(READY(s));
        }
      }
    }
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_d), "r"(2u * p.ncol) : "memory");
}

// cuTensorMapEncodeTiled through the runtime's driver entry point (no link-time dependency on libcuda)
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static EncodeTiledFn encode_tiled() {
  static EncodeTiledFn fn = []() -> EncodeTiledFn {
    void* f = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &f, cudaEnableDefault, &q) != cudaSuccess || q != cudaDriverEntryPointSuccess)
      return nullptr;
    return (EncodeTiledFn)f;
  }();
  return fn;
}

}  // namespace stag

using namespace stag;

extern "C" size_t stag_gemm_workspace_bytes(int64_t M, int32_t Nout, int32_t K) {
  (void)M; (void)Nout; (void)K;
  return 0;
}

extern "C" int stag_gemm_tcgen05(const float* a, int64_t lda, const float* wt, int64_t ldw, int64_t M, int32_t Nout,
                                 int32_t K, const float* row_scale, const float* bias, int act, float* out,
                                 int64_t ldo, void* ws, size_t ws_bytes, void* stream_) {
  (void)ws; (void)ws_bytes;
  cudaStream_t stream = (cudaStream_t)stream_;
  STAG_CHECK_ARG(M >= 0 && Nout > 0 && K > 0, "stag_gemm_tcgen05: bad sizes M=%lld N=%d K=%d", (long long)M, Nout, K);
  if (M == 0) return STAG_OK;
  STAG_CHECK_ARG(a && wt && out, "stag_gemm_tcgen05: null argument");
  STAG_CHECK_ARG(lda >= K && ldw >= K && ldo >= Nout, "stag_gemm_tcgen05: leading dimensions too small");
  STAG_CHECK_ARG(act == 0 || act == 1, "stag_gemm_tcgen05: act must be 0 (none) or 1 (relu)");
  if (Nout > 256) {
    set_error("stag_gemm_tcgen05: Nout=%d > 256 output columns per tile are not supported", Nout);
    return STAG_EUNSUPPORTED;
  }
  {
    // second form (TMA, W resident): 16-byte aligned rows of A, W_hi + W_lo of every K block within 128 KB
    const int npad2 = (Nout + 15) / 16 * 16, nkb2 = (K + GK - 1) / GK;
    static const char* force1 = getenv("STAG_GEMM_FORM");
    const bool ok = lda % 4 == 0 && (((uintptr_t)a) & 15) == 0 && (size_t)npad2 * nkb2 * 128 * 2 <= 128 * 1024 &&
                    M * lda < (1ll << 40) && !(force1 && atoi(force1) == 1) && encode_tiled() != nullptr;
    if (ok) {
      alignas(64) CUtensorMap tmap;
      const cuuint64_t gdim[2] = {(cuuint64_t)K, (cuuint64_t)M};
      const cuuint64_t gstr[1] = {(cuuint64_t)lda * 4};
      const cuuint32_t box[2] = {(cuuint32_t)GK, (cuuint32_t)GM};
      const cuuint32_t estr[2] = {1, 1};
      const CUresult er = encode_tiled()(&tmap, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<float*>(a), gdim, gstr, box, estr,
                                         CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                                         CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
      if (er == CUDA_SUCCESS) {
        Gemm2Params q;
        q.wt = wt; q.ldw = ldw; q.M = M; q.ntiles = (M + GM - 1) / GM; q.Nout = Nout; q.K = K; q.npad = npad2; q.nkb = nkb2;
        q.row_scale = row_scale; q.bias = bias; q.act = act; q.out = out; q.ldo = ldo;
        uint32_t cols = 32;
        while ((int)cols < npad2) cols <<= 1;
        q.ncol = cols;
        // shared memory: W (resident) + scratch + alignment slack, the rest is A tiles: a lo ring of 2-3 and up to
        // G2_MAXST raw tiles in flight (128-column W leaves 3 + 2, the 40-column output layer 7 + 3)
        const size_t fixed = (size_t)npad2 * nkb2 * 128 * 2 + 4 * 32 * 32 * 4 + 1024;
        const int tiles = (int)((227 * 1024 - 1024 - fixed) / G2_TILE);   // 1 KB for the static barriers
        q.nlo = tiles >= 8 ? 3 : 2;
        q.nst = (uint32_t)(tiles - (int)q.nlo < G2_MAXST ? tiles - (int)q.nlo : G2_MAXST);
        static const char* e_nlo = getenv("STAG_G2_NLO");
        static const char* e_nst = getenv("STAG_G2_NST");
        if (e_nlo) { q.nlo = (uint32_t)atoi(e_nlo); q.nst = (uint32_t)(tiles - (int)q.nlo < G2_MAXST ? tiles - (int)q.nlo : G2_MAXST); }
        if (e_nst && (uint32_t)atoi(e_nst) < q.nst) q.nst = (uint32_t)atoi(e_nst);
        const size_t smem2 = fixed + (size_t)(q.nst + q.nlo) * G2_TILE;
        STAG_CUDA(cudaFuncSetAttribute(gemm_tma_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem2));
        const int64_t grid2 = q.ntiles < num_sms() ? q.ntiles : num_sms();
        gemm_tma_kernel<<<(unsigned)grid2, G2_THREADS, smem2, stream>>>(tmap, q);
        STAG_LAUNCH_CHECK();
        return STAG_OK;
      }
    }
  }
  GemmParams p;
  p.a = a; p.lda = lda; p.wt = wt; p.ldw = ldw; p.M = M; p.Nout = Nout; p.K = K;
  p.npad = (Nout + 15) / 16 * 16;
  p.row_scale = row_scale; p.bias = bias; p.act = act; p.out = out; p.ldo = ldo;
  uint32_t cols = 32;
  while ((int)cols < p.npad) cols <<= 1;
  p.tmem_cols = cols;
  const size_t smem = (size_t)(2 * GM * GK + 2 * 256 * GK) * sizeof(float) + 1024;
  STAG_CUDA(cudaFuncSetAttribute(gemm_tcgen05_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  const int64_t grid = (M + GM - 1) / GM;
  STAG_CHECK_ARG(grid < (1ll << 31), "stag_gemm_tcgen05: too many row tiles");
  // few row tiles and a long K: split K over a cluster (at most 8 CTAs, two K blocks or more each, partial tiles
  // within the 79 KB behind the epilogue scratch)
  const int nkb = (K + GK - 1) / GK;
  int ksplit = 1;
  static const char* e_ks = getenv("STAG_GEMM_KSPLIT");
  if (grid * 2 <= num_sms() && nkb >= 4 && grid < 65536) {
    ksplit = (int)(2 * num_sms() / grid);
    if (ksplit > 8) ksplit = 8;
    if (ksplit > nkb / 2) ksplit = nkb / 2;
    if (ksplit > 158 / p.npad + 1) ksplit = 158 / p.npad + 1;
    if (e_ks && atoi(e_ks) >= 1 && atoi(e_ks) < ksplit) ksplit = atoi(e_ks);
  }
  p.ksplit = ksplit;
  if (ksplit > 1) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)ksplit, (unsigned)grid, 1);
    cfg.blockDim = dim3(GTHREADS, 1, 1);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = stream;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeClusterDimension;
    at[0].val.clusterDim.x = (unsigned)ksplit; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
    cfg.attrs = at; cfg.numAttrs = 1;
    STAG_CUDA(cudaLaunchKernelEx(&cfg, gemm_tcgen05_kernel, p));
    STAG_LAUNCH_CHECK();
    return STAG_OK;
  }
  gemm_tcgen05_kernel<<<(unsigned)grid, GTHREADS, smem, stream>>>(p);
  STAG_LAUNCH_CHECK();
  return STAG_OK;
}
