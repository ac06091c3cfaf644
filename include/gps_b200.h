/*
 * gps_b200.h — C ABI of libgps_b200.so: a B200 (sm_100a) implementation of the GraphGPS
 * `GPSLayer` forward+backward hot path.
 *
 * The reference (rampasek/GraphGPS) is pure Python and has NO FFI of its own (SURVEY.md §8b);
 * the boundary it offers is the Python module `graphgps.layer.gps_layer.GPSLayer`
 * (graphgps/layer/gps_layer.py:16-264).  The entry points below are what a binding for that
 * module calls; each cites the reference lines it replaces.  INTEGRATION.md shows the
 * ctypes binding and the GraphGym-side patch.
 *
 * Conventions
 *   - every pointer is a DEVICE pointer unless the name ends in `_host`;
 *   - the caller (PyTorch) owns every buffer; the library never allocates tensor memory.
 *     Scratch/saved sizes come from gps_layer_plan();
 *   - all work is enqueued on `stream` (a cudaStream_t passed as void*); no hidden
 *     synchronisation, no default-stream use; calls are re-entrant;
 *   - return value: 0 = ok, -1 = bad argument, -2 = unsupported shape/variant,
 *     -3 = CUDA error.  gps_last_error() returns a thread-local message.  No C++ exception
 *     crosses this boundary;
 *   - matrices are row-major float32; weights are `[out, in]` as in torch.nn.Linear
 *     (y = x · Wᵀ + b);
 *   - edge j→i: src = edge_index[0] = j, dst = edge_index[1] = i (PyG source_to_target flow,
 *     graphgps/layer/gatedgcn_layer.py:90-126).
 */
#ifndef GPS_B200_H_
#define GPS_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define GPS_ABI_VERSION 3

enum { GPS_OK = 0, GPS_ERR_ARG = -1, GPS_ERR_UNSUPPORTED = -2, GPS_ERR_CUDA = -3 };

/* local_gnn_type / global_model_type of GPSLayer.__init__ (gps_layer.py:20-24,44-122) */
enum { GPS_LOCAL_NONE = 0, GPS_LOCAL_GATEDGCN = 1, GPS_LOCAL_GINE = 2, GPS_LOCAL_GCN = 3 };
enum { GPS_GLOBAL_NONE = 0, GPS_GLOBAL_TRANSFORMER = 1, GPS_GLOBAL_PERFORMER = 2 };
/* register.act_dict keys used by shipped configs (gps_layer.py:33) */
enum { GPS_ACT_RELU = 0, GPS_ACT_GELU = 1 };
/* arithmetic of the dense products: FP32 = fp32-grade result (split-bf16 x3 on the tensor cores,
 * tolerance 1e-3 vs the reference); BF16 = single bf16 pass, fp32 accumulate (tolerance 1e-2) */
enum { GPS_PREC_FP32 = 0, GPS_PREC_BF16 = 1 };

const char* gps_last_error(void);
int gps_abi_version(void);
/* compiled-for architecture string, e.g. "sm_100a" */
const char* gps_build_arch(void);
/* number of CUDA kernels this library has launched in the calling process (bench.py reports the
 * delta over its timed region as `gpu_launches`) */
unsigned long long gps_launch_count(void);
/* bring-up / tuning hook of the tcgen05 GEMM (tools/gemm_triage.py, tools/gemm_tune.py): low byte = stage
 * switches (1 no global loads, 2 no convert/store, 4 no MMA, 8 no epilogue), bits 8.. = forced tile width. 0 = normal. */
void gps_debug_set(int v);
/* bring-up hook of the TMA-fed GEMM (tools/gemm_trace.py): force_bn = forced tile width (0 = heuristic); trace = device
 * buffer of 256 x 16 uint64 that the first 256 CTAs of each launch fill with globaltimer phase stamps (NULL = off) */
void gps_debug_tma(int force_bn, void* trace);
/* bring-up hook of the tcgen05 attention: device buffer of 3 x 128 x 128 floats that CTA (0,0) fills with its first
 * S tile, P tile and raw O accumulator (NULL = off) */
void gps_debug_attn(void* buf);

/* ------------------------------------------------------------------------------------------
 * Graph structure of one mini-batch (constant across the L layers and across fwd/bwd).
 * Replaces, per layer, PyG `MessagePassing.propagate`'s index handling
 * (gatedgcn_layer.py:67-70), torch_scatter's atomics (gatedgcn_layer.py:118-123) and
 * `to_dense_batch`'s bincount/cumsum/max (gps_layer.py:199).
 * ---------------------------------------------------------------------------------------- */
typedef struct {
  int64_t N, E, B;
  const int32_t* dst_ptr;   /* [N+1] CSR by destination                          */
  const int32_t* dst_src;   /* [E]   source node of the k-th dst-sorted edge      */
  const int32_t* dst_eid;   /* [E]   original edge id of the k-th dst-sorted edge */
  const int32_t* src_ptr;   /* [N+1] CSC by source                               */
  const int32_t* src_dst;   /* [E]   destination node of the k-th src-sorted edge */
  const int32_t* src_eid;   /* [E]   original edge id                            */
  const int32_t* graph_ptr; /* [B+1] node offsets of each graph                  */
} GpsGraph;

/* bytes of int32 scratch the caller must provide to gps_graph_build (all arrays above) */
int64_t gps_graph_bytes(int64_t N, int64_t E, int64_t B);
/* Builds the CSR/CSC/graph_ptr arrays inside `storage` (>= gps_graph_bytes) from int64
 * edge_index [2,E] and sorted int64 batch [N]; fills *out with pointers into storage.
 * Within a node's segment edges are ordered by original edge id, so every reduction over
 * a segment is deterministic. */
int gps_graph_build(const int64_t* edge_index, const int64_t* batch, int64_t N, int64_t E,
                    int64_t B, void* storage, int64_t storage_bytes, GpsGraph* out,
                    void* stream);

/* ------------------------------------------------------------------------------------------
 * One BatchNorm1d (torch.nn.BatchNorm1d: gps_layer.py:136-138,150-151; gatedgcn_layer.py:37-38)
 * ---------------------------------------------------------------------------------------- */
typedef struct {
  const float* weight;       /* gamma [d]                       */
  const float* bias;         /* beta  [d]                       */
  float* running_mean;       /* [d] updated in training mode    */
  float* running_var;        /* [d]                             */
  int64_t* num_batches_tracked; /* [1] or NULL                  */
  float* grad_weight;        /* [d] backward output (may be NULL in forward) */
  float* grad_bias;          /* [d]                             */
} GpsBatchNorm;

/* One Linear (weight [out,in], bias [out] or NULL) with its gradient outputs */
typedef struct {
  const float* weight;
  const float* bias;
  float* grad_weight;
  float* grad_bias;
} GpsLinear;

/* bf16 hi/lo planes of an fp32 [rows, cols] tensor: row-major, pitch ld elements (multiple of 8); lo may be NULL in
 * GPS_PREC_BF16 mode */
typedef struct {
  void* hi;
  void* lo;
  int64_t ld;
} GpsPlanes;

/* ------------------------------------------------------------------------------------------
 * GPSLayer forward / backward  (gps_layer.py:155-257; GatedGCN gatedgcn_layer.py:45-136)
 * state_dict names in comments are the reference's (SURVEY.md §8b).
 * ---------------------------------------------------------------------------------------- */
typedef struct {
  /* configuration */
  int64_t d;                 /* dim_h                                               */
  int64_t heads;             /* num_heads                                           */
  int32_t local_type;        /* GPS_LOCAL_*                                         */
  int32_t global_type;       /* GPS_GLOBAL_*                                        */
  int32_t act;               /* GPS_ACT_*                                           */
  int32_t training;          /* 1: batch statistics + dropout; 0: running stats     */
  int32_t precision;         /* GPS_PREC_*                                          */
  int32_t reserved0;         /* flags; bit 0 (backward): parameter-gradient buffers are already zero; bit 1: gradients are added to the buffers */
  float dropout;             /* cfg.gt.dropout       (gps_layer.py:92-96,139-140,152-153) */
  float attn_dropout;        /* cfg.gt.attn_dropout  (gps_layer.py:105-106,112-114)       */
  uint64_t seed;             /* Philox key for this call's dropout masks            */
  uint64_t offset;           /* Philox counter base (caller advances per call)      */
  float gine_eps;            /* local_model.eps buffer value (GINE)                 */
  int32_t reserved1;         /* flags; bit 0: EquivStableLapPE edge gate (fields pe .. es_r1 at the end)  */

  GpsGraph graph;

  /* inputs / outputs, row-major [N,d] / [E,d] */
  const float* x;            /* batch.x                                             */
  const float* edge_attr;    /* batch.edge_attr                                     */
  float* x_out;              /* new batch.x                                         */
  float* edge_out;           /* new batch.edge_attr (GatedGCN only, else unused)    */

  /* parameters */
  GpsLinear gcn_A, gcn_B, gcn_C, gcn_D, gcn_E;      /* local_model.{A,B,C,D,E}        */
  GpsBatchNorm bn_node_x, bn_edge_e;                /* local_model.bn_node_x / bn_edge_e */
  GpsLinear gine_lin0, gine_lin1;                   /* local_model.nn.0 / nn.2 (GINE) */
  GpsLinear attn_in;                                /* self_attn.in_proj_{weight,bias} [3d,d]   */
  GpsLinear attn_out;                               /* self_attn.out_proj / to_out              */
  GpsLinear perf_q, perf_k, perf_v;                 /* self_attn.to_{q,k,v} (no bias)           */
  const float* perf_proj;                           /* fast_attention.projection_matrix [m,64]  */
  int64_t perf_features;                            /* m (266)                                  */
  int64_t perf_dim_head;                            /* 64                                       */
  GpsBatchNorm norm1_local, norm1_attn, norm2;
  GpsLinear ff1, ff2;                               /* ff_linear1 [2d,d], ff_linear2 [d,2d]     */

  /* gradients w.r.t. outputs (backward input) and inputs (backward output) */
  const float* grad_x_out;   /* [N,d]                                               */
  const float* grad_edge_out;/* [E,d] or NULL (treated as zero)                     */
  float* grad_x;             /* [N,d]                                               */
  float* grad_edge_attr;     /* [E,d]                                               */

  /* caller-owned scratch; sizes from gps_layer_plan() */
  void* saved;   int64_t saved_bytes;     /* written by forward, read by backward   */
  void* workspace; int64_t workspace_bytes; /* transient; may be shared between calls on one stream */

  /* optional device-resident addend for `offset` (uint64 on the device, read by the kernels at run time):
   * lets a captured CUDA graph draw fresh dropout masks on every replay. NULL = use `offset` only. */
  const uint64_t* offset_dev;

  /* ABI 2: PyG GCNConv(dim_h, dim_h) local model (gps_layer.py:49-51): weight = local_model.lin.weight [d,d]
   * (its Linear has no bias), bias = local_model.bias [d], added after the normalised aggregation. */
  GpsLinear gcn_conv;

  /* ABI 3 (backward, optional): a cudaEvent_t the library records as soon as the "early" parameter gradients are
   * final - ff_linear1/2, the attention output projection, norm2, norm1_local, norm1_attn - a few hundred microseconds
   * before the pass ends.  A data-parallel caller makes its communication stream wait on it and all-reduces that
   * part of the gradient bucket under the rest of the backward pass (graphgps_b200/dp.py).  NULL = not recorded. */
  void* ev_grads_early;

  /* ABI 3 (optional): operand-plane hand-off between consecutive layers of a GPSModel (network/gps_model.py:100,105-108)
   * and persistent weight planes.  A plane pair is the bf16 hi/lo image of an fp32 tensor (see gps_to_planes).
   *  x_planes_in / e_planes_in   planes of x / edge_attr written by the previous layer: the layer skips its own
   *                              conversion of the inputs (hi == NULL: convert here, into `saved`);
   *  x_planes_out / e_planes_out caller-owned plane buffers the layer fills next to x_out / edge_out;
   *  wplanes                     caller-owned buffer (GpsLayerPlan.wplanes_bytes) for the planes of every weight;
   *                              wplanes_valid != 0: it already holds this layer's current weights (packed once per
   *                              optimiser step instead of once per forward call). */
  GpsPlanes x_planes_in, e_planes_in, x_planes_out, e_planes_out;
  void* wplanes; int64_t wplanes_bytes; int32_t wplanes_valid; int32_t reserved2;

  /* ABI 3 (backward, optional): two more cudaEvent_t of the same kind as ev_grads_early.  ev_grads_mid: the local
   * model's gradients (A, B, C, D, E / GINE nn / GCN lin, bn_node_x, bn_edge_e) are final - the weight gradient of the
   * fused node projection is computed in two parts for this, the local column block as soon as the message-passing
   * backward is done, the in_proj block at the end.  ev_grads_done: every gradient of this layer is final. */
  void* ev_grads_mid;
  void* ev_grads_done;

  /* EquivStableLapPE edge gate of the GatedGCN local model (GPSLayer(..., equivstable_pe=True): gatedgcn_layer.py:29-35,
   * 63-70, 99-103), switched on by reserved1 bit 0 and read ONLY then, so a zero-initialised caller never reaches these
   * fields.  With the bit set for a local model other than GatedGCN the calls return GPS_ERR_UNSUPPORTED.
   *   r_ij = sum_c (pe_i,c - pe_j,c)^2,  gate_ij = sigmoid(W2 act(W1 r_ij + b1) + b2),  sigma_ij = sigmoid(e_ij) * gate_ij
   * in the aggregation (the edge output e_ij stays ungated).  fp32 in both precision modes.
   *   pe       batch.pe_EquivStableLapPE [N, pe_dim], row-major float32 (the same tensor for every layer);
   *   grad_pe  backward output [N, pe_dim], overwritten (not accumulated); NULL = not computed;
   *   es_r0    local_model.mlp_r_ij.0 (weight [d,1], bias [d]);  es_r1  local_model.mlp_r_ij.2 (weight [1,d], bias [1]).
   * Their gradients follow reserved0 like every other parameter and belong to the ev_grads_mid group. */
  const float* pe;
  int64_t pe_dim;
  float* grad_pe;
  GpsLinear es_r0, es_r1;
} GpsLayerArgs;

typedef struct {
  int64_t saved_bytes;          /* activations kept for backward (0 needed if eval-only) */
  int64_t fwd_workspace_bytes;
  int64_t bwd_workspace_bytes;
  int64_t fwd_launches;         /* kernels the forward enqueues  */
  int64_t bwd_launches;         /* kernels the backward enqueues */
  int64_t wplanes_bytes;        /* ABI 3: size of the optional persistent weight-plane buffer (GpsLayerArgs.wplanes) */
} GpsLayerPlan;

/* Sizes for the given configuration/graph (only sizes and type fields of args are read). */
int gps_layer_plan(const GpsLayerArgs* args, GpsLayerPlan* plan);
int gps_layer_forward(const GpsLayerArgs* args, void* stream);
int gps_layer_backward(const GpsLayerArgs* args, void* stream);

/* ------------------------------------------------------------------------------------------
 * Stage-level entry points (the same kernels the layer calls; exported so the parity tests can
 * pin each stage against the oracle separately).
 * ---------------------------------------------------------------------------------------- */

/* C[M,N] = A[M,K] · W[N,K]ᵀ + bias  — replaces pyg_nn.Linear / nn.Linear (gatedgcn_layer.py:57-61,
 * gps_layer.py:253-257).  precision selects the tensor-core path (GPS_PREC_*). */
int gps_linear_forward(const float* A, int64_t lda, const float* W, int64_t ldw, const float* bias,
                       float* C, int64_t ldc, int64_t M, int64_t N, int64_t K, int32_t act,
                       int32_t precision, void* stream);

/* General dense product used for the data / weight gradients of every Linear:
 *   C[M,N] (+)= Aop[M,K] * Bop[K,N];  ta==0: Aop[m,k]=A[m*lda+k], ta==1: Aop[m,k]=A[k*lda+m];
 *   tb==0: Bop[k,n]=B[n*ldb+k] (an nn.Linear weight), tb==1: Bop[k,n]=B[k*ldb+n].
 * splitk > 1 accumulates atomically into a pre-zeroed C.  impl: 0 = dispatcher (tcgen05 when the
 * shape qualifies), 1 = exact CUDA-core kernel, 2 = tcgen05 kernel (GPS_ERR_UNSUPPORTED if it does
 * not take the shape). */
int gps_gemm(const float* A, int64_t lda, int32_t ta, const float* B, int64_t ldb, int32_t tb, float* C,
             int64_t ldc, int64_t M, int64_t N, int64_t K, int32_t splitk, int32_t precision, int32_t impl,
             void* stream);

/* GatedGCN message+aggregate+update (gatedgcn_layer.py:90-136) given the five projections.
 * Y holds [Ax | Bx | Dx | Ex] columns at the given offsets with row stride ldy; Ce [E,d] is
 * overwritten with e_ij (pre-activation edge output, :106,:134); xt [N,d] = Ax + num/(den+1e-6).
 * stats_x/stats_e: optional double [2][d] column sum / sum of squares accumulators (BatchNorm). */
int gps_gatedgcn_aggregate_forward(const GpsGraph* g, int64_t d, const float* Ax, const float* Bx,
                                   const float* Dx, const float* Ex, int64_t ldy, float* Ce,
                                   float* xt, double* stats_x, double* stats_e, void* stream);

/* EquivStableLapPE edge gate (see GpsLayerArgs.pe): r [E] and gate [E] per original edge id.  w0/b0 = mlp_r_ij.0,
 * w2/b2 = mlp_r_ij.2, act = GPS_ACT_*. */
int gps_es_gate_forward(const GpsGraph* g, const float* pe, int64_t pe_dim, int64_t d, int32_t act,
                        const float* w0, const float* b0, const float* w2, const float* b2, float* r, float* gate,
                        void* stream);
/* gps_gatedgcn_aggregate_forward with sigma_ij = sigmoid(e_ij) * gate[edge id]. */
int gps_gatedgcn_es_aggregate_forward(const GpsGraph* g, int64_t d, const float* Ax, const float* Bx,
                                      const float* Dx, const float* Ex, int64_t ldy, float* Ce, float* xt,
                                      double* stats_x, double* stats_e, const float* gate, void* stream);
/* Backward of the gate MLP: given g_gate [E] = d loss / d gate, writes g_r [E] = d loss / d r and the four
 * mlp_r_ij gradients (overwritten).  Deterministic (per-block partials in `workspace`, fixed-order final sum);
 * workspace_bytes >= gps_es_gate_backward_workspace_bytes(E, d). */
int64_t gps_es_gate_backward_workspace_bytes(int64_t E, int64_t d);
int gps_es_gate_backward(int64_t E, int64_t d, int32_t act, const float* w0, const float* b0, const float* w2,
                         const float* b2, const float* r, const float* gate, const float* g_gate, float* g_r,
                         float* grad_w0, float* grad_b0, float* grad_w2, float* grad_b2, void* workspace,
                         int64_t workspace_bytes, void* stream);
/* d loss / d pe from g_r: grad_pe_n = sum_{e: dst=n} 2 g_r_e (pe_n - pe_src(e)) + sum_{e: src=n} 2 g_r_e (pe_n - pe_dst(e)) */
int gps_es_pe_backward(const GpsGraph* g, const float* pe, int64_t pe_dim, const float* g_r, float* grad_pe,
                       void* stream);

/* GINE aggregate: out_i = (1+eps)·x_i + Σ_{j→i} relu(x_j + e_ij)  (gine_conv_layer.py:56-84) */
int gps_gine_aggregate_forward(const GpsGraph* g, int64_t d, const float* x, const float* e,
                               float eps, float* out, void* stream);

/* Dense softmax attention over each graph's own nodes — replaces to_dense_batch +
 * nn.MultiheadAttention core + [mask] (gps_layer.py:199-201,234-241) without padding.
 * Q,K,V: [N, heads*hd] slices with row stride ld; O [N, heads*hd] (row stride ldo); lse [N,heads]. */
int gps_attention_forward(const GpsGraph* g, int64_t heads, int64_t hd, const float* Q,
                          const float* K, const float* V, int64_t ld, float* O, int64_t ldo,
                          float* lse, float p_drop, uint64_t seed, uint64_t offset, void* stream);
/* ABI 3: the same forward on the tensor cores (csrc/attention_tc.cu: tcgen05 S = QK^T and O += PV, TMA-staged tiles,
 * block-diagonal graph mask applied in-kernel).  qkv_hi/qkv_lo: bf16 hi/lo planes [N, ld] holding Q | K | V per head in
 * the padded layout column (which * heads + h) * hd_pad + k with hd_pad = round_up(hd, 16) and zero pad columns
 * (qkv_lo NULL for GPS_PREC_BF16).  Same O / lse conventions as gps_attention_forward, so either backward applies. */
int gps_attention_forward_tc(const GpsGraph* g, int64_t heads, int64_t hd, const void* qkv_hi, const void* qkv_lo,
                             int64_t ld, float* O, int64_t ldo, float* lse, float p_drop, uint64_t seed,
                             uint64_t offset, int32_t precision, void* stream);
/* (the layer-level calls additionally honour GpsLayerArgs.offset_dev) */
int gps_attention_backward(const GpsGraph* g, int64_t heads, int64_t hd, const float* Q,
                           const float* K, const float* V, int64_t ld, const float* O,
                           const float* dO, int64_t ldo, const float* lse, float* delta,
                           float* dQ, float* dK, float* dV, int64_t ldg, float p_drop,
                           uint64_t seed, uint64_t offset, void* stream);

/* ABI 3: operand "planes" of the TMA-fed tcgen05 GEMM (csrc/gemm_tma.cu).  A plane pair is the bf16 image of an
 * fp32 matrix: hi = bf16(v), lo = bf16(v - hi), both plain row-major with pitch ldp (elements, multiple of 8); lo may
 * be NULL for GPS_PREC_BF16.  gps_to_planes converts; gps_gemm_planes multiplies plane operands stored as
 * A: [M,K] (ta = 0) or [K,M] (ta = 1), B: [N,K] (tb = 0, an nn.Linear weight) or [K,N] (tb = 1), writes fp32 C
 * (may be NULL) and/or the planes of C, optionally adds the row sums of Aop into colsum_a[M] (ta = 1: the bias
 * gradient of dW = G^T X).  splitk > 1 accumulates atomically into a pre-zeroed fp32 C. */
int gps_to_planes(const float* src, int64_t ld, int64_t rows, int64_t cols, void* hi, void* lo, int64_t ldp,
                  void* stream);
int gps_gemm_planes(const void* A_hi, const void* A_lo, int64_t lda, int32_t ta, const void* B_hi, const void* B_lo,
                    int64_t ldb, int32_t tb, float* C, int64_t ldc, void* C_hi, void* C_lo, int64_t ldcp, int64_t M,
                    int64_t N, int64_t K, int32_t splitk, int32_t precision, float* colsum_a, void* stream);
/* number of dense products that fell back from the tensor-core kernels to the exact CUDA-core kernel
 * (unaligned / odd shapes) in this process; with GPS_B200_STRICT=1 in the environment such a fallback is an error */
unsigned long long gps_fallback_count(void);

/* Dropout keep-mask generator used by every dropout site (tests replay it): writes 1/0 floats. */
int gps_dropout_mask(float* mask, int64_t rows, int64_t cols, float p, uint64_t seed,
                     uint64_t offset, int32_t site, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* GPS_B200_H_ */
