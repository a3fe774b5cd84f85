/* stag_b200 -- C ABI of the B200-native stochastic neighbour aggregation.
 *
 * Drop-in boundary for the ONE hot path of yuanqing-wang/stag (SURVEY.md section 8):
 * the per-edge(-per-channel) multiplicative noise draw + message scaling + segmented
 * reduction that the reference reaches through
 *     StagLayer.forward            stag/layers.py:84-113
 *       -> rsample_noise           stag/layers.py:115-129   (noise [E,K])
 *       -> _in_norm                stag/layers.py:8-36
 *       -> base_layer.forward(graph=, feat=, edge_weight=)   stag/layers.py:109-113
 *            -> graph.update_all(fn.u_mul_e, fn.sum|fn.mean) stag/zoo/gcn.py:63,95
 *                                                            stag/zoo/graph_sage.py:57,72,86
 * and, in training, through autograd of the same (transposed aggregation + SDDMM).
 * The reference has no FFI of its own (pure Python over DGL); these entry points are
 * what a ctypes stub inside stag/zoo/*.py binds instead of graph.update_all -- see
 * INTEGRATION.md.
 *
 * Conventions
 *  - plain C, no torch/CUDA types in signatures: device pointers are passed as raw
 *    pointers, the stream as `void*` (a cudaStream_t; NULL = legacy default stream).
 *  - every buffer is allocated and owned by the caller (PyTorch's caching allocator);
 *    the library never allocates persistent device memory and never frees caller memory.
 *  - every function returns 0 (STAG_OK) or a negative STAG_E* code and never throws;
 *    stag_last_error() returns a thread-local message for the last failure.
 *  - all work is enqueued on the given stream; only stag_csx_build synchronises (it
 *    returns the hub counts to the host), and the *_host convenience entry points.
 *  - features are fp32 row-major; structure is int32 on device (E, N < 2^31); the COO
 *    input is int64 as produced by DGL (g.edges()).
 */
#ifndef STAG_B200_H
#define STAG_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define STAG_ABI_VERSION 2

#if defined(__GNUC__)
#define STAG_API __attribute__((visibility("default")))
#else
#define STAG_API
#endif

enum {
  STAG_OK = 0,
  STAG_EINVAL = -1,       /* bad argument (null pointer, shape mismatch, unsupported combination) */
  STAG_ECUDA = -2,        /* a CUDA runtime call or kernel launch failed */
  STAG_EWORKSPACE = -3,   /* workspace too small; see the *_workspace_bytes query */
  STAG_EUNSUPPORTED = -4  /* valid request that this build does not implement */
};

/* distribution of the multiplicative edge noise (stag/layers.py:115-129) */
enum {
  STAG_NOISE_NONE = 0,      /* w == 1: plain copy_u/sum aggregation (edge_weight=None, stag/zoo/gcn.py:59) */
  STAG_NOISE_EXTERNAL = 1,  /* w read from a caller tensor [S,E,K] in ORIGINAL edge order (parity seam) */
  /* w = loc + scale*eps (torch/distributions/normal.py:82-85).  eps: Box-Muller on the two 16-bit halves of a Philox
   * word, u1 = (h_lo + 1/2) / 65536, u2 = (h_hi + 1/2) / 65536: 65 536 radii x 65 536 angles.  KNOWN LIMIT of this
   * generator: the largest radius is sqrt(2 ln 2^17) = 4.854, so |eps| <= 4.854 -- a true normal puts 1.2e-6 of its
   * mass beyond that (123 of 1e8 draws) and this generator none; within +-4.6 sigma it passes chi-square and KS tests
   * at 1e8 draws (tests/test_gpu_rng_law.py).  STAG_NOISE_NORMAL_HADAMARD has no such cut. */
  STAG_NOISE_NORMAL = 2,
  STAG_NOISE_UNIFORM = 3,   /* w = low + u*(high-low)         torch/distributions/uniform.py:85-88  */
  STAG_NOISE_BERNOULLI = 4, /* w = (u < probs)                torch/distributions/bernoulli.py:116-119 */
  /* w = loc + scale*eps like STAG_NOISE_NORMAL, with eps drawn by the tensor-core generator: the 128 channels of
   * a group are the Walsh-Hadamard mix of 128 masked random FP8 bytes (csrc/spmm_tc.cuh, spmm_wq.cuh; normal to
   * 5.6e-6 in Kolmogorov distance, support to +-24 sigma, tails at the normal rate in tests/test_gpu_rng_law.py).
   * A different stream than STAG_NOISE_NORMAL.  Fused path: K == D, D % 128 == 0, 32-byte aligned rows, scalar or
   * per-edge parameters, no relu / in_norm / parameter gradients; stag_noise_emit: K % 128 == 0. */
  STAG_NOISE_NORMAL_HADAMARD = 5
};

/* shape class of the distribution parameters before `expand([E,K])` (stag/layers.py:117-119) */
enum {
  STAG_PARAM_SCALAR = 0,       /* "r1":  one value                       */
  STAG_PARAM_CHANNEL = 1,      /* "rc":  [K]                             */
  STAG_PARAM_EDGE = 2,         /* "re":  [E,1]  (AmortizedDistribution)  */
  STAG_PARAM_EDGE_CHANNEL = 3  /* "rec": [E,K]  (AmortizedDistribution)  */
};

/* One compressed adjacency (CSC when built by destination, CSR when built by source),
 * as filled in by stag_csx_build.  All pointers are device pointers. */
typedef struct StagGraph {
  int64_t num_rows;          /* N: rows of this structure (dst nodes for CSC, src nodes for CSR) */
  int64_t num_cols;          /* number of nodes on the other side                                */
  int64_t num_edges;         /* E                                                                */
  const int32_t* indptr;     /* [N+1] row pointers                                               */
  const int32_t* indices;    /* [E]   other endpoint of each stored edge                         */
  const int32_t* eid;        /* [E]   original COO position of each stored edge                  */
  /* hub schedule: rows with more than stag_hub_threshold() stored edges are processed as
   * segments of stag_hub_segment() edges and combined in a fixed order (deterministic). */
  int32_t num_hubs;
  int32_t num_hub_segs;
  const int32_t* hub_rows;     /* [num_hubs]   row ids, increasing                */
  const int32_t* hub_seg_ptr;  /* [num_hubs+1] first global segment of each hub   */
  /* processing order of the rows (decreasing stored-edge count) so that rows sharing a warp have
   * equal trip counts; NULL = natural order.  Results do not depend on it, except for the last bits of the summed
   * SCALAR / CHANNEL parameter gradients of stag_spmm_bwd on the row-per-group path (per-CTA partials are added in
   * the order the rows are visited). */
  const int32_t* row_order;    /* [num_rows] or NULL                              */
  /* stream items: consecutive row ranges {row0, row1, e0, e1} holding about 64 stored edges each
   * (e1 = -1: placeholder of a hub row), by decreasing edge count: the unit of work of the
   * streaming kernels */
  const int32_t* items;        /* [num_items][4] or NULL                          */
  int64_t num_items;
  const int32_t* erow;         /* [E] row of every stored edge (the sorted keys) or NULL */
  const int32_t* eidf;         /* [E] eid with bit 31 set on the last stored edge of a row, or NULL */
} StagGraph;

/* Noise specification.  Parameter pointers are DEVICE pointers (they are nn.Parameters /
 * buffers of stag.distributions.ParametrizedDistribution, stag/distributions.py:93-144, or
 * the per-edge outputs of AmortizedDistribution, :221-242), already in natural units
 * (scale, not log_scale). */
typedef struct StagNoise {
  int32_t kind;          /* STAG_NOISE_*                                                        */
  int32_t K;             /* noise width: D (per edge per channel) or 1 (per edge)               */
  int32_t param_shape;   /* STAG_PARAM_*                                                        */
  int32_t relu;          /* stag/layers.py:98-99                                                */
  int32_t in_norm;       /* stag/layers.py:102-105 (_in_norm); forward / CSC pass only          */
  int32_t sample_base;   /* global index of local sample 0 (MC-sample sharding across GPUs)     */
  const float* p0;       /* loc | low | probs                                                   */
  const float* p1;       /* scale | high | NULL                                                 */
  const float* external; /* EXTERNAL: [S,E,K], original edge order                              */
  uint64_t seed;         /* Philox key                                                          */
  uint64_t offset;       /* Philox call counter: one per (layer, forward call)                  */
  /* Optional DEVICE-side addend to the call counter (NULL: none): the kernels add *counter (mod 2^32) to the low
   * word of `offset` when they run.  A training step captured in a CUDA graph bakes `offset` into its kernel
   * parameters; bumping this device word between replays gives every replay fresh noise (ABI version 2). */
  const uint32_t* counter;
} StagNoise;

STAG_API const char* stag_last_error(void);
STAG_API int stag_abi_version(void);
/* number of CUDA kernels this library has launched since it was loaded (process-wide) */
STAG_API long long stag_launch_count(void);
STAG_API int stag_hub_threshold(void);
STAG_API int stag_hub_segment(void);

/* ---- on-device CSC / CSR builder ------------------------------------------------------
 * Replaces DGL's COO->CSC/CSR conversion behind graph.update_all (stag/zoo/gcn.py:95) and
 * graph.in_degrees()/out_degrees() (stag/zoo/gcn.py:68,101; stag/layers.py:21).
 * Stable LSD radix sort by destination (by_dst=1) or source (by_dst=0): bit-exact
 * indptr / indices / eid against a stable sort of the COO list.
 *   hub_rows     capacity  E / stag_hub_threshold() + 1
 *   hub_seg_ptr  capacity  E / stag_hub_threshold() + 2
 *   row_order    [N] rows by decreasing degree (optional, may be NULL)
 *   items        [stag_csx_items_capacity(E, N)][4] stream items (optional, may be NULL)
 *   erow         [E] row of every stored edge (optional, may be NULL)
 *   eidf         [E] eid | (last edge of its row) << 31 (optional, may be NULL)
 *   counts_host  [3] host ints: {num_hubs, num_hub_segs, num_items}  (the call synchronises `stream`)
 */
STAG_API size_t stag_csx_workspace_bytes(int64_t num_edges, int64_t num_nodes);
STAG_API int64_t stag_csx_items_capacity(int64_t num_edges, int64_t num_nodes);
STAG_API int stag_csx_build(const int64_t* src, const int64_t* dst, int64_t num_edges, int64_t num_nodes,
                   int by_dst, int32_t* indptr, int32_t* indices, int32_t* eid,
                   int32_t* hub_rows, int32_t* hub_seg_ptr, int32_t* row_order, int32_t* items,
                   int32_t* erow, int32_t* eidf, int32_t* counts_host, void* ws, size_t ws_bytes, void* stream);

/* ---- fused stochastic aggregation ------------------------------------------------------
 * Forward (CSC graph), replaces rsample_noise + relu + _in_norm + update_all(u_mul_e, sum):
 *
 *   out[s,v,c] = dst_scale[v] * sum_{j in row v} w_s[eid_j, c] * (src_scale[u_j] * x[s,u_j,c])
 *
 * with u_j = indices[j], w drawn inside the kernel (never stored) or read from
 * noise->external.  With in_norm the sum is multiplied by indeg(v) / sum_j w_s[eid_j,c]
 * (1 when that sum is 0) and that factor is written to norm_scale_out [S,N,K] if non-NULL.
 * x_sample_stride = 0 shares one X [N,D] across the S samples (first layer);
 * ld* are row strides in floats.  reduce='mean' is expressed through dst_scale.
 *
 * The same entry point run on the CSR graph with (src_scale, dst_scale) swapped and
 * x := dOut is the transposed aggregation, i.e. dX of the backward pass.
 *
 * The workspace holds per-call state (edge records, hub partial sums, the work-queue counter of the streaming
 * kernels): calls that may run concurrently (different streams) need a workspace each.  Results do not depend on
 * how the queue hands the work out (every output row is summed by one thread group in stored-edge order): bitwise
 * run-to-run.
 */
STAG_API size_t stag_spmm_workspace_bytes(const StagGraph* g, int32_t D, int32_t S);
STAG_API int stag_spmm_fwd(const StagGraph* g, const float* x, int64_t ldx, int64_t x_sample_stride,
                  int32_t D, int32_t S, const StagNoise* noise,
                  const float* src_scale, const float* dst_scale,
                  float* out, int64_t ldo, int64_t out_sample_stride,
                  float* norm_scale_out, void* ws, size_t ws_bytes, void* stream);

/* Backward with noise-parameter gradients (CSR graph; vi=True, stag/layers.py:123-124).
 * One pass over the out-edges of every source node u regenerates w from (seed, offset) and emits
 *   dx[s,u,c]     = src_scale[u] * sum_j w_s[eid_j,c] * g[s,v_j,c],   g = dst_scale[v]*dout[s,v,c]
 *   dw[s,e,c]     = (src_scale[u]*x[s,u,c]) * g[s,v,c]                (SDDMM, never stored unless
 *                                                                     EXTERNAL and dw_external != NULL)
 *   NORMAL : dparam0 = sum dw (d loc), dparam1 = sum dw*eps (d scale)
 *   UNIFORM: dparam0 = sum dw*(1-u) (d low), dparam1 = sum dw*u (d high)
 * reduced to the parameter shape: SCALAR -> [1], CHANNEL -> [K], EDGE -> [E], EDGE_CHANNEL -> [E,K]
 * (EDGE shapes ACCUMULATE into dparam*, summed over the S samples, i.e. the caller zeroes them once; any S when the
 * graph carries erow -- an edge-parallel kernel -- else S == 1).
 * SCALAR / CHANNEL results OVERWRITE dparam* and are summed over the S samples.
 * dx may be NULL (first layer: features need no gradient).  Not valid with in_norm.
 */
STAG_API int stag_spmm_bwd(const StagGraph* csr, const float* x, int64_t ldx, int64_t x_sample_stride,
                  const float* dout, int64_t ldg, int64_t dout_sample_stride,
                  int32_t D, int32_t S, const StagNoise* noise,
                  const float* src_scale, const float* dst_scale,
                  float* dx, int64_t lddx, int64_t dx_sample_stride,
                  float* dparam0, float* dparam1, float* dw_external,
                  void* ws, size_t ws_bytes, void* stream);

/* ---- fused stochastic MAX aggregation ---------------------------------------------------
 * Forward (CSC graph), replaces rsample_noise + relu + update_all(u_mul_e, fn.max) (GraphSAGE 'pool', GIN 'max'):
 *
 *   out[s,v,c] = max_{j in row v} w_s[eid_j, c] * x[s,u_j,c]        (fp32 product, then compare)
 *   arg[s,v,c] = eid_j of the winning edge (ORIGINAL edge id)
 *
 * Ties go to the first edge in stored order, i.e. the smallest edge id (strict >, the CSC is a stable sort); rows
 * without in-edges get out = 0, arg = -1.  arg has the strides of out.  The noise is the stream stag_noise_emit writes
 * for the same spec (every kind; K == 1 or D, STAG_NOISE_NORMAL_HADAMARD with K == D), so the result equals the max over
 * the materialised tensor bit for bit.  No degree scalings; in_norm and STAG_PARAM_EDGE_CHANNEL are rejected
 * (STAG_EINVAL): materialise the noise for those.  Same workspace as stag_spmm_fwd (stag_spmm_workspace_bytes).
 */
STAG_API int stag_spmm_max_fwd(const StagGraph* g, const float* x, int64_t ldx, int64_t x_sample_stride,
                      int32_t D, int32_t S, const StagNoise* noise,
                      float* out, int32_t* arg, int64_t ldo, int64_t out_sample_stride,
                      void* ws, size_t ws_bytes, void* stream);

/* Backward of stag_spmm_max_fwd (CSR graph; arg = the forward's, at the strides of dout).  Only the winner of a
 * (sample, row, channel) receives its gradient:
 *   dx[s,u,c]  = sum_j [arg[s,v_j,c] == eid_j] w_s[eid_j,c] * dout[s,v_j,c]
 *   dw[s,e,c]  = [arg[s,v,c] == e] x[s,u,c] * dout[s,v,c]      (never stored unless EXTERNAL and dw_external != NULL:
 *                                                             K == D per channel, K == 1 summed over the channels)
 *   NORMAL : dparam0 = sum dw (d loc), dparam1 = sum dw*eps (d scale)
 *   UNIFORM: dparam0 = sum dw*(1-u) (d low), dparam1 = sum dw*u (d high)        (relu: masked by w > 0)
 * dx, dparam0/1 and dw_external are each optional (NULL).  SCALAR / CHANNEL parameter gradients OVERWRITE dparam*,
 * EDGE ([E,1]) ones ACCUMULATE (summed over the S samples); per-edge outputs need a graph built with erow.
 * Deterministic: no float atomics.
 */
STAG_API int stag_spmm_max_bwd(const StagGraph* csr, const float* x, int64_t ldx, int64_t x_sample_stride,
                      const float* dout, const int32_t* arg, int64_t ldg, int64_t dout_sample_stride,
                      int32_t D, int32_t S, const StagNoise* noise,
                      float* dx, int64_t lddx, int64_t dx_sample_stride,
                      float* dparam0, float* dparam1, float* dw_external,
                      void* ws, size_t ws_bytes, void* stream);

/* Materialise the noise tensor w [S,E,K] (original edge order) from the same Philox stream
 * the fused kernels use: compatibility path for base layers that are not fused
 * (StagLayer._edge_weight_sample, stag/layers.py:107; KL fallback :141-143) and for RNG tests.
 * eps_out (optional) receives the raw variate (standard normal / uniform) before loc/scale. */
STAG_API int stag_noise_emit(const StagNoise* noise, int64_t num_edges, int32_t S,
                    float* w_out, float* eps_out, void* stream);

/* Sample-based KL terms without the noise tensor: replaces the fallback of StagLayer.kl_divergence
 * (stag/layers.py:139-141: q_a.log_prob(w).sum(-1).mean() - p_a.log_prob(w).sum(-1).mean() on the stored [E,K]
 * sample, used when torch has no analytic KL, e.g. the mixture prior of
 * scripts/citation_rec_contrastive/gcn/run.py:44-52).  The sample is regenerated from `noise` (the spec of the
 * forward: same seed / offset / sample_base / relu) and reduced on the fly:
 *   sums[0] = sum over (sample, edge, channel) of log q(w),  sums[1] = the same of log p(w)   (device, double[2])
 *   dparam0 / dparam1 (optional, device, parameter shape of `noise`): d(sums[0] - sums[1]) / d(p0, p1), the
 *   reparameterisation path w(p0, p1) included.  Deterministic (fixed summation order).
 * q: STAG_NOISE_NORMAL (p0 loc, p1 scale) or STAG_NOISE_UNIFORM (low, high), no in_norm.  The prior is a handful of
 * HOST scalars. */
#define STAG_PRIOR_MAX_COMPONENTS 8
#define STAG_PRIOR_NORMAL_MIXTURE 1
typedef struct StagPrior {
  int32_t kind;                              /* STAG_PRIOR_NORMAL_MIXTURE                                     */
  int32_t M;                                 /* components: 1 = a plain Normal                                */
  float weight[STAG_PRIOR_MAX_COMPONENTS];   /* mixture probabilities (normalised by the library)             */
  float loc[STAG_PRIOR_MAX_COMPONENTS];
  float scale[STAG_PRIOR_MAX_COMPONENTS];
} StagPrior;
STAG_API size_t stag_noise_kl_workspace_bytes(int32_t K);
STAG_API int stag_noise_kl(const StagNoise* noise, int64_t num_edges, int32_t S, const StagPrior* prior, double* sums,
                  float* dparam0, float* dparam1, void* ws, size_t ws_bytes, void* stream);

/* Segmented readout over batch_num_nodes (SumNodes / MeanNodes, stag/layers.py:156-178):
 * out[b,c] = sum (or mean) of feat rows in [node_ptr[b], node_ptr[b+1]). */
STAG_API int stag_segment_reduce(const float* feat, int64_t ldf, const int32_t* node_ptr, int32_t num_graphs,
                        int32_t D, int mean, float* out, int64_t ldo, void* stream);

/* Segmented softmax over the in-edges of every destination (dgl.nn.edge_softmax in the reference's GAT,
 * stag/zoo/gat.py:122): out[e,h] = exp(logits[e,h] - max) / sum over the edges with the same destination.  logits / out
 * [E,H] in ORIGINAL edge order; csc = the graph built by destination.  Backward: dlogits = a * (da - sum_row a * da). */
STAG_API int stag_edge_softmax(const StagGraph* csc, const float* logits, int32_t H, float* out, void* stream);
STAG_API int stag_edge_softmax_bwd(const StagGraph* csc, const float* a, const float* da, int32_t H, float* dlogits,
                          void* stream);

/* The same with GAT's attention logits computed inside (stag/zoo/gat.py:113-122):
 *   logit[e,h] = w[e,h] * leaky_relu(el[u_e,h] + er[v_e,h], slope),   a[e,h] = softmax over the in-edges of v_e
 * el [num_cols,H] (source rows), er [num_rows,H], w [E,H] in original edge order or NULL (no edge noise); a [E,H].
 * Backward from da [E,H]: dw [E,H] (may be NULL), dpre [E,H] = d(el[u] + er[v]) per edge (the caller sums it per SOURCE
 * on the CSR graph: d el), d_er [num_rows,H] = its sum per destination.  No atomics: deterministic. */
STAG_API int stag_attention_softmax(const StagGraph* csc, const float* el, const float* er, const float* w, float slope,
                           int32_t H, float* a, void* stream);
STAG_API int stag_attention_softmax_bwd(const StagGraph* csc, const float* el, const float* er, const float* w, float slope,
                               int32_t H, const float* a, const float* da, float* dw, float* dpre, float* d_er,
                               void* stream);

/* The same over S Monte-Carlo samples in one launch, with the logit noise drawn inside the kernel (stochastic GAT):
 *   logit[s,e,h] = w_s[e,h] * leaky_relu(el[s,u_e,h] + er[s,v_e,h], slope),   a[s,e,h] = softmax over the in-edges of v_e
 * el / er: sample s at el + s * el_sample_stride (0: one [num_cols,H] / [num_rows,H] shared by every sample, the first
 * layer); a [S,E,H] in original edge order.  noise: STAG_NOISE_NONE, EXTERNAL ([S,E,H]) or a generated kind (NORMAL,
 * UNIFORM, BERNOULLI) with K == H, any parameter shape, relu, sample_base and the device counter.  The variate of
 * (edge, head h, sample s) is the one stag_noise_emit writes for channel h of sample sample_base + s, so the result
 * equals the attention over the materialised tensor bit for bit.  STAG_NOISE_NORMAL_HADAMARD -> STAG_EUNSUPPORTED,
 * in_norm -> STAG_EINVAL (materialise the noise for those).
 * Backward from da [S,E,H]: dpre [S,E,H] = d(el[u] + er[v]) per edge (the caller sums it per SOURCE on the CSR graph),
 * d_er [S,num_rows,H] = its sum per destination, dw_external [S,E,H] (EXTERNAL only, may be NULL) and, for Normal /
 * Uniform noise, dparam0 / dparam1 (both or neither) in the parameter shape: d loc / d scale, d low / d high, masked by
 * w > 0 under relu.  SCALAR / CHANNEL results OVERWRITE dparam* and are summed over the S samples; EDGE ([E,1], summed
 * over the heads) and EDGE_CHANNEL ([E,H]) results ACCUMULATE (the caller zeroes them once).  The workspace holds the
 * per-CTA partials of the SCALAR / CHANNEL reduction (stag_attention_workspace_bytes; unused otherwise).  No float
 * atomics: bitwise run-to-run. */
STAG_API size_t stag_attention_workspace_bytes(const StagGraph* csc, int32_t H, int32_t S);
STAG_API int stag_attention_softmax_s(const StagGraph* csc, const float* el, int64_t el_sample_stride,
                             const float* er, int64_t er_sample_stride, int32_t H, int32_t S,
                             const StagNoise* noise, float slope, float* a, void* ws, size_t ws_bytes, void* stream);
STAG_API int stag_attention_softmax_s_bwd(const StagGraph* csc, const float* el, int64_t el_sample_stride,
                                 const float* er, int64_t er_sample_stride, int32_t H, int32_t S,
                                 const StagNoise* noise, float slope, const float* a, const float* da,
                                 float* dpre, float* d_er, float* dparam0, float* dparam1, float* dw_external,
                                 void* ws, size_t ws_bytes, void* stream);

/* Likelihood epilogue (stag/models.py:69-72, stag/likelihoods.py:13-38): for each of the S Monte-Carlo outputs
 *   nll_out[s] = mean over the masked nodes of -log_prob(probs[s], y)
 * kind 0: Categorical(probs=.) -- probs renormalised, clamped to [eps, 1-eps], log, gathered at y (int64 [N]);
 * kind 1: Bernoulli(probs=.)   -- y float [N,C] (row stride ldy), mean over the masked rows x C labels;
 * exactly as torch.distributions evaluates them.  mask: uint8 [N] or NULL.  count_out[0] = number of terms of each
 * mean.  dprobs (optional, same strides as probs) receives d(count * nll_out[s]) / d probs[s] in the same pass. */
STAG_API size_t stag_nll_workspace_bytes(int64_t N, int32_t S);
STAG_API int stag_nll(const float* probs, int64_t ld, int64_t sample_stride, int64_t N, int32_t C, int32_t S,
             int kind, const void* y, int64_t ldy, const uint8_t* mask, float* nll_out, float* count_out,
             float* dprobs, void* ws, size_t ws_bytes, void* stream);

/* Monte-Carlo predictive statistics in bounded memory.  probs[s] (s < S) is the raw [N,C] output of one Monte-Carlo
 * sample (row stride ld, sample stride sample_stride, which may be 0).  acc_sum [N,C] (contiguous) and acc_ent [N] are
 * float64, caller-owned and caller-zeroed; stag_mc_accumulate ADDS to them:
 *   acc_sum += p_s,   acc_ent += H(p_s)
 * in sample order, one row per warp, no atomics: calls over consecutive chunks of samples give the same bits whatever
 * the chunk sizes, and two chunked passes over disjoint sample ranges can be summed (sample sharding).
 * kind 0: H = Categorical(probs=.).entropy() = -sum_c q_c log(clamp(q_c, eps, 1-eps)), q = p / sum(p);
 * kind 1: H = sum over the C labels of Bernoulli(probs=.).entropy(); eps = torch.finfo(float32).eps.
 * A row that sums to zero or holds a NaN gives NaN, as in torch.  C <= 1024 (STAG_EUNSUPPORTED above).
 * stag_mc_finalize, with S_total the number of samples accumulated:
 *   mean = acc_sum / S_total ([N,C] contiguous), pred_entropy = H(mean), exp_entropy = acc_ent / S_total,
 *   mutual_info = pred_entropy - exp_entropy,
 *   loglik (optional, with y) = Categorical(probs=mean).log_prob(y), y int64 [N] (NaN outside [0, C)), or the sum over
 *   the labels of Bernoulli(probs=mean).log_prob(y), y float [N,C] with row stride ldy; y and loglik are both NULL or
 *   both set. */
STAG_API int stag_mc_accumulate(const float* probs, int64_t ld, int64_t sample_stride, int64_t N, int32_t C, int32_t S,
                       int kind, double* acc_sum, double* acc_ent, void* stream);
STAG_API int stag_mc_finalize(const double* acc_sum, const double* acc_ent, int64_t N, int32_t C, int64_t S_total,
                     int kind, const void* y, int64_t ldy, float* mean, float* pred_entropy, float* exp_entropy,
                     float* mutual_info, float* loglik, void* stream);

/* Calibration of [N,C] probabilities (e.g. the Monte-Carlo mean of stag_mc_finalize) as an int64 table of counts and
 * fixed-point sums, fx(x) = x * STAG_CAL_ONE rounded half-to-even.  Integer sums do not depend on their order: the
 * table of a call is the same every run, and the sum of the tables of several calls (row chunks, minibatches, ranks)
 * is the table of one call over all their rows, bit for bit.  ECE, Brier score, accuracy / micro-F1 and reliability
 * diagrams follow from the table (stag_b200/calibration.py).
 *   probs float32 [N,C], row stride ld >= C; mask uint8 [N] or NULL (rows with mask == 0 are not read);
 *   kind 0 (Categorical): y int64 [N]; kind 1 (Bernoulli): y float32 [N,C], row stride ldy >= C (as stag_mc_finalize);
 *   table int64 [stag_calibration_table_len(C, n_bins)], caller-owned and caller-zeroed: the call ADDS to it.
 * Bins (B = n_bins in [1, 64]) are those of sklearn's calibration_curve(strategy="uniform"): interior edges
 * i * (1.0 / B) (double, i = 1 .. B-1, the values of np.linspace(0, 1, B+1)); bin(x) = the number of interior edges
 * strictly below x, so bins are (lo, hi] and 0 falls in bin 0.
 * Layout (int64):
 *   [0] n: valid rows          [1] n_invalid: rows refused (see below)
 *   [2] Categorical: rows whose argmax is the label; Bernoulli: tp      [3] 0 | fp      [4] 0 | fn
 *   [5] brier: sum of fx((q_c - [c == y])^2) over the classes of valid rows (Categorical), of fx((p - y)^2) over the
 *       labels (Bernoulli)
 *   [6 ..)         top-label table [3][B]: count, sum of fx(conf), count of correct rows   (Categorical; 0 for Bernoulli)
 *   [6 + 3B ..)    per-class table [3][C][B]: count, sum of fx(q_c) | fx(p_c), label sum: [c == y] (a count,
 *                  Categorical) | fx(y_c) (Bernoulli)
 * Categorical row m (read as doubles): invalid if any m_c is NaN, infinite or negative, if s = sum m_c is 0 or if
 *   y is outside [0, C).  s is summed as stag_mc_finalize sums a row (lane l of a warp adds classes l, l+32, ... in
 *   order, then an xor butterfly over offsets 16, 8, 4, 2, 1).  q_c = m_c / s; k = the first index of the largest m_c
 *   (torch.argmax); conf = q_k; bin(conf) in the top-label table, bin(q_c) in the table of class c.
 * Bernoulli row: invalid if any p_c or y_c is NaN or outside [0, 1]; tp / fp / fn compare p > 0.5 with y > 0.5;
 *   bin(p_c) in the table of class c.
 * Every fixed-point term is at most STAG_CAL_ONE = 2^32: the caller keeps entries below 2^63 by adding at most 2^31
 * terms to one; one call takes N*C < 2^31 (STAG_EINVAL above).  C <= 1024 (STAG_EUNSUPPORTED above); N = 0 is a no-op.
 * stag_calibration_table_len: 6 + 3B + 3CB, or STAG_EINVAL for C < 1 or n_bins outside [1, 64]. */
#define STAG_CAL_ONE 4294967296.0 /* fixed-point unit of the probability sums: 2^32 */
STAG_API int64_t stag_calibration_table_len(int32_t C, int32_t n_bins);
STAG_API int stag_calibration(const float* probs, int64_t ld, int64_t N, int32_t C, int kind, const void* y,
                              int64_t ldy, const uint8_t* mask, int32_t n_bins, int64_t* table, void* stream);

/* Dense feature transform agg @ W (stag/zoo/gcn.py:97-98) on tcgen05 tensor cores with TMEM
 * accumulators; fp32 in / fp32 out computed as 3xTF32 (fp32-level accuracy), fused epilogue
 *   out[m,n] = act( row_scale[m] * sum_k a[m,k]*w[k,n] + bias[n] ),  act: 0 none, 1 relu.
 * wt is W transposed, [Nout, K] row-major (K-major). */
STAG_API size_t stag_gemm_workspace_bytes(int64_t M, int32_t Nout, int32_t K);
STAG_API int stag_gemm_tcgen05(const float* a, int64_t lda, const float* wt, int64_t ldw,
                      int64_t M, int32_t Nout, int32_t K,
                      const float* row_scale, const float* bias, int act,
                      float* out, int64_t ldo, void* ws, size_t ws_bytes, void* stream);

/* Host-buffer convenience entry point for a non-torch caller (bench.py's e2e leg goes through the Python API instead):
 * COO graph, features and upstream gradient in HOST memory; builds CSC+CSR on the device,
 * runs forward + backward for S samples with generated noise and copies out / dx back.
 * Synchronous.  device = CUDA ordinal. */
STAG_API int stag_aggregate_host(int device, const int64_t* src, const int64_t* dst, int64_t num_edges,
                        int64_t num_nodes, const float* x, const float* dout, int32_t D, int32_t S,
                        const StagNoise* noise_host_params, int gcn_norm_both,
                        float* out, float* dx);

#ifdef __cplusplus
}
#endif
#endif /* STAG_B200_H */
