// layer.cu — host-side orchestration of one GPSLayer forward / backward and the C ABI.
//
// Follows graphgps/layer/gps_layer.py:155-232 (composition), :234-257 (attention / FFN blocks) and
// graphgps/layer/gatedgcn_layer.py:45-88 (GatedGCN with residual=True as built at gps_layer.py:92-96).
// Stage list (training mode, CustomGatedGCN+Transformer):
//   pack W -> [Ax|Bx|Dx|Ex|Q|K|V] = x Wcat^T -> Ce = e C^T -> segmented gather-reduce (+BN stats)
//   -> x_loc = x + act(BN(x~)) (+stats), e_out = e + act(BN(e^)) -> attention -> hA = x + O Wo^T (+stats)
//   -> s = BN(x_loc) + BN(hA) -> FFN (+stats) -> BN.
// Training-mode BatchNorm is "producer accumulates column sums, tiny finalize, consumer normalises".
#include <stdarg.h>
#include <string.h>

#include <algorithm>
#include <atomic>

#include "gemm.cuh"
#include "kernels.cuh"

namespace gps {

// performer.cu
int perf_supported(int64_t dim_head, int64_t features);
int64_t perf_mp();
int perf_prep(const float* P, int64_t m, float* Pn, const GpsGraph& g, int64_t H, int* nmax, float* gmax, int* argk,
              cudaStream_t st);
int perf_features_fwd(float* fq, float* fk, const float* Q, const float* K, const GpsGraph& g, int64_t H, int64_t m,
                      float* gmax, int* argq, int* argk, cudaStream_t st);
int perf_linattn_fwd(const GpsGraph& g, int64_t H, int64_t m, const int* nmax, const float* qf, const float* kf,
                     const float* V, const float* gmax, float* O, cudaStream_t st);
int perf_linattn_bwd(const GpsGraph& g, int64_t H, int64_t m, const int* nmax, const float* qf, const float* kf,
                     const float* V, const float* gmax, const float* gO, float* g_qf, float* g_kf, float* gV,
                     float* ggmax, cudaStream_t st);
int perf_features_bwd(float* g_fq, float* g_fk, const float* fq, const float* fk, const float* Q, const float* K,
                      float* gQ, float* gK, const GpsGraph& g, int64_t H, int64_t m, const int* argq, const int* argk,
                      float* ggmax, cudaStream_t st);

// performer_quad.cu (pairwise form for batches of small graphs)
int perf_quad_fwd(const GpsGraph& g, int64_t H, int64_t m, const int* nmax, const float* qf, const float* kf,
                  const float* V, const float* gmax, float* O, float* den, cudaStream_t st);
int perf_quad_bwd(const GpsGraph& g, int64_t H, int64_t m, const int* nmax, const float* qf, const float* kf,
                  const float* V, const float* gmax, const float* O, const float* den, const float* gO, float* gden,
                  float* g_qf, float* g_kf, float* gV, float* ggmax, cudaStream_t st);

// ------------------------------------------------------------------------------- error plumbing
static thread_local char g_err[512] = "";
static std::atomic<unsigned long long> g_launches{0};

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}
int cuda_fail(cudaError_t e, const char* what, const char* file, int line) {
  set_error("CUDA error %d (%s) at %s:%d: %s", (int)e, cudaGetErrorString(e), file, line, what);
  return GPS_ERR_CUDA;
}
void count_launch() { g_launches.fetch_add(1, std::memory_order_relaxed); }

static std::atomic<unsigned long long> g_fallbacks{0};

// Dispatcher: TMA-fed tcgen05 kernel when the caller supplies operand planes, else the register-staged tcgen05 kernel
// on the fp32 operands, else (odd shapes / alignment) the exact CUDA-core kernel - counted, and an error under
// GPS_B200_STRICT=1 so that a 10x slower path can never be taken silently.
int gemm(const GemmParams& p, cudaStream_t stream) {
  static const int mode = [] {   // GPS_B200_GEMM: "simt" = CUDA-core only, "tc" = no TMA kernel, default = all
    const char* e = getenv("GPS_B200_GEMM");
    return e && strcmp(e, "simt") == 0 ? 2 : (e && strcmp(e, "tc") == 0 ? 1 : 0);
  }();
  static const bool strict = [] {
    const char* e = getenv("GPS_B200_STRICT");
    return e && e[0] == '1';
  }();
  if (mode == 0 && p.Ap.hi && p.Bp.hi) {
    int rc = gemm_tma(p, stream);
    if (rc != GPS_ERR_UNSUPPORTED) return rc;
  }
  GPS_REQUIRE(p.A && p.B && p.C, GPS_ERR_UNSUPPORTED, "gemm: plane operands rejected and no fp32 operands to fall back to");
  GPS_REQUIRE(!p.bnred[0].sums && !p.bnred[1].sums, GPS_ERR_UNSUPPORTED,
              "gemm: fused BatchNorm-backward reductions exist in the TMA kernel only");
  GemmParams q = p;
  if (q.Cp.hi) {   // the fp32 kernels do not write planes: convert afterwards
    q.Cp = Planes();
  }
  int rc = GPS_ERR_UNSUPPORTED;
  if (mode != 2) rc = gemm_tc(q, stream);
  if (rc == GPS_ERR_UNSUPPORTED) {
    if (mode != 2) {
      g_fallbacks.fetch_add(1, std::memory_order_relaxed);
      GPS_REQUIRE(!strict, GPS_ERR_UNSUPPORTED,
                  "GPS_B200_STRICT: dense product M=%d N=%d K=%d (ta=%d tb=%d) would fall back to the CUDA-core kernel",
                  p.M, p.N, p.K, p.ta, p.tb);
    }
    rc = gemm_simt(q, stream);
  }
  if (rc == GPS_OK && p.Cp.hi) {
    ToPlanesItem it{p.C, p.ldc, p.M, p.N, p.Cp};
    rc = to_planes(&it, 1, stream);
  }
  return rc;
}

namespace {

// ------------------------------------------------------------------------------- side stream (fork / join)
// Independent stages run concurrently with the main chain: the edge projection next to the node projections, the
// attention branch next to the message-passing branch (gps_layer.py:161-218 computes both from the same h_in1),
// and every weight-gradient GEMM next to the data-gradient chain.  Fork = event on the caller's stream that the
// side stream waits on; join = the reverse.  All of it is capturable into a CUDA graph.
struct Side {
  cudaStream_t s = nullptr;    // weight gradients / edge projection / forward attention branch
  cudaStream_t s3 = nullptr;   // backward attention branch (next to the message-passing backward)
  cudaStream_t s4 = nullptr;   // edge-side BatchNorm backward (depends on grad_edge_out only, so it starts at once)
  cudaEvent_t ev[32];
  int next = 0;
  bool ok = false;
  int init() {
    if (ok) return GPS_OK;
    GPS_CUDA(cudaStreamCreateWithFlags(&s, cudaStreamNonBlocking));
    GPS_CUDA(cudaStreamCreateWithFlags(&s3, cudaStreamNonBlocking));
    GPS_CUDA(cudaStreamCreateWithFlags(&s4, cudaStreamNonBlocking));
    for (int i = 0; i < 32; ++i) GPS_CUDA(cudaEventCreateWithFlags(&ev[i], cudaEventDisableTiming));
    ok = true;
    return GPS_OK;
  }
  int order(cudaStream_t from, cudaStream_t to) {   // `to` waits for everything enqueued on `from` so far
    cudaEvent_t e = ev[next++ & 31];
    GPS_CUDA(cudaEventRecord(e, from));
    GPS_CUDA(cudaStreamWaitEvent(to, e, 0));
    return GPS_OK;
  }
  int fork(cudaStream_t main) { return order(main, s); }
  int join(cudaStream_t main) { return order(s, main); }
};

// A/B switches (GPS_B200_OPT): 1 MN-major weight planes, 2 merged attention backward, 4 early edge BN backward,
// 8 projection gradients split into the message-passing and attention column blocks
static int opt_flags() {
  static const int v = [] {
    const char* e = getenv("GPS_B200_OPT");
    return e ? atoi(e) : 7;   // Measured slower on B200 and therefore off (same-box A/B, profiles/r2_ab_switches.txt):
                              // 8 (split dgrad+wgrad tail) 0.478 vs 0.465; 16 (two-part Wcat wgrad) 0.476 vs 0.465;
                              // 32 + 64 (bn_node_x reduce inside the norm1_local apply pass, norm1_local / norm1_attn
                              // reduces in the epilogue of the GEMM producing g_s) 0.4946 vs 0.4856: three launches
                              // fewer, but the fused kernels run as few fat CTAs and delay the branches behind them on B200 (0.478 vs 0.465 ms/step in round 2 as well); 16 (two-part Wcat
                              // weight gradient) too: 0.476 vs 0.465 on one GPU and no gain at N = 2
  }();
  return v;
}

static Side* side_stream() {
  static const bool enabled = [] {
    const char* e = getenv("GPS_B200_STREAMS");
    return !(e && e[0] == '0');
  }();
  if (!enabled) return nullptr;
  static thread_local Side sides[64];
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return nullptr;
  if (sides[dev].init() != GPS_OK) return nullptr;
  return &sides[dev];
}

// ------------------------------------------------------------------------------- weight packing
struct PackSeg {
  const float* w; const float* b; float* gw; float* gb; int rows;
};
struct PackDesc {
  PackSeg seg[5];
  int nseg; int d; int total_rows;
};

// cat[r, :] = seg.w[r - row0, :], bcat[r] = seg.b[...] (0 when the Linear has no bias).  One row per blockIdx.x.
__global__ void k_pack(PackDesc pd, float* __restrict__ Wcat, float* __restrict__ bcat) {
  const int r = blockIdx.x;
  int row0 = 0, s = 0;
  while (s < pd.nseg - 1 && r >= row0 + pd.seg[s].rows) row0 += pd.seg[s++].rows;
  const float* src = pd.seg[s].w + (int64_t)(r - row0) * pd.d;
  float* dst = Wcat + (int64_t)r * pd.d;
  for (int c = threadIdx.x * 4; c < pd.d; c += blockDim.x * 4) st4(dst + c, ld4(src + c));
  if (threadIdx.x == 0) bcat[r] = pd.seg[s].b ? pd.seg[s].b[r - row0] : 0.f;
}
__global__ void k_unpack(PackDesc pd, const float* __restrict__ gWcat, const float* __restrict__ gbcat, int accumulate,
                         int row_begin) {
  const int r = blockIdx.x + row_begin;
  int row0 = 0, s = 0;
  while (s < pd.nseg - 1 && r >= row0 + pd.seg[s].rows) row0 += pd.seg[s++].rows;
  if (pd.seg[s].gw) {
    float* dst = pd.seg[s].gw + (int64_t)(r - row0) * pd.d;
    const float* src = gWcat + (int64_t)r * pd.d;
    for (int c = threadIdx.x * 4; c < pd.d; c += blockDim.x * 4)
      st4(dst + c, accumulate ? f4add(ld4(dst + c), ld4(src + c)) : ld4(src + c));
  }
  if (threadIdx.x == 0 && pd.seg[s].gb) pd.seg[s].gb[r - row0] = (accumulate ? pd.seg[s].gb[r - row0] : 0.f) + gbcat[r];
}

enum { BN_X = 0, BN_E = 1, BN_L = 2, BN_A = 3, BN_2 = 4, BN_COUNT = 5 };

struct Plan {
  int64_t N, E, d, H, hd, Wy, qkv_off;
  bool gated, gine, gcn, attn, perf;
  int64_t inner, mp, m;   // Performer: H*64, padded / real feature count
  float *pQ, *pK, *pV, *pfq, *pfk, *pPn, *pgmax;   // saved (Performer)
  int *pargq, *pargk, *pnmax;
  float *pden, *g_pden;   // pairwise form: denominators (saved) and their gradients
  bool perf_pairwise;     // mean graph size <= 48: n^2 (m+64) < 2 n m 64
  float *g_pfq, *g_pfk, *g_pQ, *g_pK, *g_pV, *g_pgmax, *g_xp;   // backward workspace (Performer)
  // saved
  float *Wcat, *bcat, *Y1, *ehat, *xt, *xloc, *O, *lse, *hA, *s, *hid, *hid_pre, *t, *bnbuf;
  float *agg, *h1, *h1_pre;
  float* dinv;   // GCN: deg^-1/2 per node
  // EquivStableLapPE edge gate (GpsLayerArgs.reserved1 bit 0, GatedGCN only): saved r_e, gate_e; backward workspace
  // d loss / d gate shares [E, es_nw], d loss / d r [E] and the per-block partials of the mlp_r_ij gradients
  bool es;
  int es_nw;
  float *es_r, *es_g, *es_ggate, *es_gr;
  void* es_work;
  int64_t es_work_bytes;
  // pre-packed bf16 hi/lo weight planes for the forward GEMMs (bulk-TMA B operand)
  uint8_t *pk_cat, *pk_C, *pk_out, *pk_ff1, *pk_ff2, *pk_g0, *pk_g1;
  // the same weights as MN-major planes for the data-gradient GEMMs of the backward pass (training only)
  uint8_t *pt_cat, *pt_C, *pt_out, *pt_ff1, *pt_ff2, *pt_g0, *pt_g1;
  bool prepack;
  // bf16 hi/lo operand planes of the TMA-fed GEMM (gemm_tma.cu).  Saved: layer inputs, weights and the forward
  // activations the weight gradients re-read; workspace: the backward gradients that feed GEMMs.
  bool use_planes;
  Planes x_p, e_p, O_p, s_p, hid_p, agg_p, h1_p, Wcat_p, C_p, out_p, ff1_p, ff2_p, g0_p, g1_p, pq_p, pk_p, pv_p;
  Planes gt_p, ghid_p, ghA_p, ge_p, gY1_p, gtmp_p, gtmp2_p, gtmp3_p, gl1_p, gh1_p;
  Planes qkv_p;        // Q | K | V per head, padded to hd_pad columns: operands of the tcgen05 attention
  bool attn_tc;        // softmax attention on the tensor cores (attention_tc.cu)
  int64_t saved_bytes;
  int64_t wplanes_bytes;
  // forward workspace
  double* fstats;
  int64_t fwd_bytes;
  // backward workspace
  double* bsums;
  float *g_t, *g_hid, *g_s, *g_xloc, *g_hA, *g_O, *gY1, *g_e, *g_num, *delta, *g_tmp, *g_tmp2, *g_tmp3, *g_h1, *g_agg, *gWcat,
      *gbcat, *g_xl;
  int64_t bwd_bytes;
  int64_t fwd_launches, bwd_launches;
};

// GPS_B200_GEMM=tc|simt keeps the round-1 operand path (register-staged conversion per consuming CTA)
static bool planes_enabled() {
  static const bool v = [] {
    const char* e = getenv("GPS_B200_GEMM");
    return !(e && (strcmp(e, "tc") == 0 || strcmp(e, "simt") == 0));
  }();
  return v;
}

// Forward softmax attention on the tensor cores (attention_tc.cu) when the batch's graphs are large enough for 128 x 128
// tiles to pay: measured on B200 (round 2) the tcgen05 kernel needs 57 us at the PCQM4M shape (mean 14 nodes per graph:
// a 128-row tile sees ~45 useful keys of 256, one latency-bound wave of 116 CTAs) against 25 us for the CUDA-core kernel,
// and wins once a graph fills a tile (ogbg-code2 shape, mean 125 / max ~1000 nodes).  GPS_B200_ATTN=simt | tc overrides.
static bool attn_tc_enabled(int64_t N, int64_t B) {
  static const int mode = [] {
    const char* e = getenv("GPS_B200_ATTN");
    return e && strcmp(e, "simt") == 0 ? 0 : (e && strcmp(e, "tc") == 0 ? 2 : 1);
  }();
  if (mode != 1) return mode == 2;
  return B > 0 && N >= 64 * B;
}

static int make_plan(const GpsLayerArgs* a, Plan* P, bool bind) {
  memset(P, 0, sizeof(*P));
  GPS_REQUIRE(a, GPS_ERR_ARG, "null args");
  P->N = a->graph.N;
  P->E = a->graph.E;
  P->d = a->d;
  P->H = a->heads;
  GPS_REQUIRE(a->d > 0 && a->d % 4 == 0, GPS_ERR_UNSUPPORTED, "dim_h must be a positive multiple of 4 (got %lld)",
              (long long)a->d);
  P->gated = a->local_type == GPS_LOCAL_GATEDGCN;
  P->gine = a->local_type == GPS_LOCAL_GINE;
  P->gcn = a->local_type == GPS_LOCAL_GCN;
  P->es = (a->reserved1 & 1) != 0;
  GPS_REQUIRE(!P->es || P->gated, GPS_ERR_UNSUPPORTED,
              "equivstable_pe (reserved1 bit 0) is built for the GatedGCN local model only (local_type %d)", a->local_type);
  GPS_REQUIRE(!P->es || a->d <= 1023, GPS_ERR_UNSUPPORTED, "equivstable_pe supports dim_h <= 1023 (got %lld)",
              (long long)a->d);
  GPS_REQUIRE(a->local_type == GPS_LOCAL_NONE || P->gated || P->gine || P->gcn, GPS_ERR_ARG, "unknown local_type %d",
              a->local_type);
  GPS_REQUIRE(a->global_type == GPS_GLOBAL_NONE || a->global_type == GPS_GLOBAL_TRANSFORMER ||
                  a->global_type == GPS_GLOBAL_PERFORMER,
              GPS_ERR_ARG, "unknown global_type %d", a->global_type);
  P->attn = a->global_type == GPS_GLOBAL_TRANSFORMER;
  P->perf = a->global_type == GPS_GLOBAL_PERFORMER;
  if (P->perf) {
    GPS_TRY(perf_supported(a->perf_dim_head, a->perf_features));
    GPS_REQUIRE(a->heads > 0, GPS_ERR_ARG, "num_heads must be positive");
    P->inner = a->heads * a->perf_dim_head;
    P->mp = perf_mp();
    P->m = a->perf_features;
  }
  GPS_REQUIRE(a->local_type != GPS_LOCAL_NONE || P->attn || P->perf, GPS_ERR_ARG,
              "GPSLayer needs a local model or a global model");
  if (P->attn) {
    GPS_REQUIRE(a->heads > 0 && a->d % a->heads == 0, GPS_ERR_ARG, "dim_h %% num_heads != 0");
    P->hd = a->d / a->heads;
    GPS_REQUIRE(P->hd % 4 == 0, GPS_ERR_UNSUPPORTED, "head dim %lld must be a multiple of 4", (long long)P->hd);
  }
  GPS_REQUIRE(a->act == GPS_ACT_RELU || a->act == GPS_ACT_GELU, GPS_ERR_ARG, "unknown activation %d", a->act);
  GPS_REQUIRE(a->dropout >= 0.f && a->dropout < 1.f && a->attn_dropout >= 0.f && a->attn_dropout < 1.f,
              GPS_ERR_ARG, "dropout probabilities must be in [0,1)");
  const int64_t N = P->N, E = P->E, d = P->d;
  P->qkv_off = P->gated ? 4 * d : (P->gcn ? d : 0);
  P->Wy = P->qkv_off + (P->attn ? 3 * d : 0);
  const bool gelu = a->act == GPS_ACT_GELU;

  Arena S(bind ? a->saved : nullptr, a->saved_bytes);
  P->bnbuf = S.alloc<float>(BN_COUNT * 2 * d);
  if (P->Wy) {
    P->Wcat = S.alloc<float>(P->Wy * d);
    P->bcat = S.alloc<float>(P->Wy);
    P->Y1 = S.alloc<float>(N * P->Wy);
  }
  if (P->gated) {
    P->ehat = S.alloc<float>(E * d);
    P->xt = S.alloc<float>(N * d);
    if (P->es) {
      P->es_r = S.alloc<float>(E);
      P->es_g = S.alloc<float>(E);
    }
  }
  if (P->gine) {
    P->agg = S.alloc<float>(N * d);
    P->h1 = S.alloc<float>(N * d);
    if (gelu) P->h1_pre = S.alloc<float>(N * d);
  }
  if (P->gcn) P->dinv = S.alloc<float>(N);
  if (P->gated || P->gine || P->gcn) P->xloc = S.alloc<float>(N * d);
  if (P->attn) {
    P->O = S.alloc<float>(N * d);
    P->lse = S.alloc<float>(N * P->H);
    P->hA = S.alloc<float>(N * d);
  }
  if (P->perf) {
    const int64_t NH = N * P->H, BH = a->graph.B * P->H;
    P->pQ = S.alloc<float>(N * P->inner);
    P->pK = S.alloc<float>(N * P->inner);
    P->pV = S.alloc<float>(N * P->inner);
    P->pfq = S.alloc<float>(NH * P->mp);
    P->pfk = S.alloc<float>(NH * P->mp);
    P->pPn = S.alloc<float>(P->mp * a->perf_dim_head);
    P->pgmax = S.alloc<float>(BH);
    P->pargq = S.alloc<int>(NH);
    P->pargk = S.alloc<int>(BH);
    P->pnmax = S.alloc<int>(1);
    P->pden = S.alloc<float>(NH);
    P->perf_pairwise = a->graph.B > 0 && N <= 48 * a->graph.B;
    P->O = S.alloc<float>(N * P->inner);
    P->hA = S.alloc<float>(N * d);
  }
  P->s = S.alloc<float>(N * d);
  P->hid = S.alloc<float>(N * 2 * d);
  if (gelu) P->hid_pre = S.alloc<float>(N * 2 * d);
  P->t = S.alloc<float>(N * d);
  P->prepack = (d % 8 == 0) && (!P->perf || P->inner % 8 == 0);
  P->use_planes = P->prepack && planes_enabled();
  const bool lo = a->precision == GPS_PREC_FP32;
  auto mkplanes = [&](Arena& A, int64_t rows, int64_t cols) {
    Planes q;
    q.ld = round_up(cols, 8);
    q.hi = A.alloc<__nv_bfloat16>(rows * q.ld + 8);
    q.lo = lo ? A.alloc<__nv_bfloat16>(rows * q.ld + 8) : nullptr;
    return q;
  };
  if (P->use_planes) {
    const int64_t kout = P->perf ? P->inner : d;
    auto handed = [&](const GpsPlanes& g) {   // planes written by the previous layer of the stack
      Planes q;
      q.hi = (__nv_bfloat16*)g.hi; q.lo = lo ? (__nv_bfloat16*)g.lo : nullptr; q.ld = g.ld;
      return q;
    };
    const bool x_in = a->x_planes_in.hi && (!lo || a->x_planes_in.lo) && a->x_planes_in.ld >= d && a->x_planes_in.ld % 8 == 0;
    const bool e_in = a->e_planes_in.hi && (!lo || a->e_planes_in.lo) && a->e_planes_in.ld >= d && a->e_planes_in.ld % 8 == 0;
    P->x_p = x_in ? handed(a->x_planes_in) : mkplanes(S, N, d);
    if (P->gated || P->gine) P->e_p = e_in ? handed(a->e_planes_in) : mkplanes(S, E, d);
    if (P->attn || P->perf) P->O_p = mkplanes(S, N, kout);
    P->attn_tc = P->attn && attention_tc_supported(P->hd) && attn_tc_enabled(N, a->graph.B);
    if (P->attn_tc) P->qkv_p = mkplanes(S, N, 3 * P->H * attention_tc_hd_pad(P->hd));
    P->s_p = mkplanes(S, N, d);
    P->hid_p = mkplanes(S, N, 2 * d);
    if (P->gine) {
      P->agg_p = mkplanes(S, N, d);
      P->h1_p = mkplanes(S, N, d);
    }
    // weight planes: in the caller's persistent buffer when one is given (packed once per optimiser step), else in `saved`
    Arena Wa(bind ? a->wplanes : nullptr, a->wplanes_bytes);
    const bool persistent = bind && a->wplanes != nullptr;
    Arena& WA = persistent ? Wa : S;
    Arena Wc(nullptr, 0);            // size of the persistent buffer, counted independently of `saved`
    for (int pass = 0; pass < 2; ++pass) {
      Arena& A = pass == 0 ? Wc : WA;
      Planes wcat, cp, outp, f1, f2, g0, g1, pq, pk, pv;
      if (P->Wy) wcat = mkplanes(A, P->Wy, d);
      if (P->gated) cp = mkplanes(A, d, d);
      if (P->attn || P->perf) outp = mkplanes(A, d, kout);
      f1 = mkplanes(A, 2 * d, d);
      f2 = mkplanes(A, d, 2 * d);
      if (P->gine) {
        g0 = mkplanes(A, d, d);
        g1 = mkplanes(A, d, d);
      }
      if (P->perf) {
        pq = mkplanes(A, P->inner, d);
        pk = mkplanes(A, P->inner, d);
        pv = mkplanes(A, P->inner, d);
      }
      if (pass == 1) {
        P->Wcat_p = wcat; P->C_p = cp; P->out_p = outp; P->ff1_p = f1; P->ff2_p = f2; P->g0_p = g0; P->g1_p = g1;
        P->pq_p = pq; P->pk_p = pk; P->pv_p = pv;
      }
    }
    P->wplanes_bytes = Wc.used;
    GPS_REQUIRE(!Wa.overflow, GPS_ERR_ARG, "wplanes buffer too small (%lld < %lld)", (long long)a->wplanes_bytes,
                (long long)Wc.used);
  }
  if (P->prepack && !P->use_planes) {
    const int64_t kout = P->perf ? P->inner : d;
    if (P->Wy) P->pk_cat = S.alloc<uint8_t>(prepack_bytes((int)P->Wy, (int)d));
    if (P->gated) P->pk_C = S.alloc<uint8_t>(prepack_bytes((int)d, (int)d));
    if (P->attn || P->perf) P->pk_out = S.alloc<uint8_t>(prepack_bytes((int)d, (int)kout));
    P->pk_ff1 = S.alloc<uint8_t>(prepack_bytes((int)(2 * d), (int)d));
    P->pk_ff2 = S.alloc<uint8_t>(prepack_bytes((int)d, (int)(2 * d)));
    if (P->gine) {
      P->pk_g0 = S.alloc<uint8_t>(prepack_bytes((int)d, (int)d));
      P->pk_g1 = S.alloc<uint8_t>(prepack_bytes((int)d, (int)d));
    }
    if (a->training) {   // W as [K = out features] x [N = in features]
      if (P->Wy) P->pt_cat = S.alloc<uint8_t>(prepack_bytes_mn((int)d, (int)P->Wy));
      if (P->gated) P->pt_C = S.alloc<uint8_t>(prepack_bytes_mn((int)d, (int)d));
      if (P->attn || P->perf) P->pt_out = S.alloc<uint8_t>(prepack_bytes_mn((int)kout, (int)d));
      P->pt_ff1 = S.alloc<uint8_t>(prepack_bytes_mn((int)d, (int)(2 * d)));
      P->pt_ff2 = S.alloc<uint8_t>(prepack_bytes_mn((int)(2 * d), (int)d));
      if (P->gine) {
        P->pt_g0 = S.alloc<uint8_t>(prepack_bytes_mn((int)d, (int)d));
        P->pt_g1 = S.alloc<uint8_t>(prepack_bytes_mn((int)d, (int)d));
      }
    }
  }
  P->saved_bytes = S.used;
  GPS_REQUIRE(!S.overflow, GPS_ERR_ARG, "saved buffer too small (%lld < %lld)", (long long)a->saved_bytes,
              (long long)S.used);

  // forward and backward share the caller's workspace (never live at the same time)
  Arena F(bind ? a->workspace : nullptr, a->workspace_bytes);
  P->fstats = F.alloc<double>(BN_COUNT * 2 * d);
  P->fwd_bytes = F.used;

  Arena Bk(bind ? a->workspace : nullptr, a->workspace_bytes);
  P->bsums = Bk.alloc<double>(BN_COUNT * 2 * d);
  P->g_t = Bk.alloc<float>(N * d);
  P->g_hid = Bk.alloc<float>(N * 2 * d);
  P->g_s = Bk.alloc<float>(N * d);
  P->g_tmp = Bk.alloc<float>(N * d);
  if (a->dropout > 0.f || (P->perf && a->attn_dropout > 0.f)) {   // separate dropout temporaries: side-stream weight
    P->g_tmp2 = Bk.alloc<float>(N * d);                            // gradients still read the earlier ones
    P->g_tmp3 = Bk.alloc<float>(N * d);
  }
  if (P->gated || P->gine || P->gcn) P->g_xloc = Bk.alloc<float>(N * d);
  if (P->attn) {
    P->g_hA = Bk.alloc<float>(N * d);
    P->g_O = Bk.alloc<float>(N * d);
    P->delta = Bk.alloc<float>(N * P->H);
  }
  if (P->perf) {
    const int64_t NH = N * P->H, BH = a->graph.B * P->H;
    P->g_hA = Bk.alloc<float>(N * d);
    P->g_O = Bk.alloc<float>(N * P->inner);
    P->g_pfq = Bk.alloc<float>(NH * P->mp);
    P->g_pfk = Bk.alloc<float>(NH * P->mp);
    P->g_pQ = Bk.alloc<float>(N * P->inner);
    P->g_pK = Bk.alloc<float>(N * P->inner);
    P->g_pV = Bk.alloc<float>(N * P->inner);
    P->g_pgmax = Bk.alloc<float>(BH);
    P->g_pden = Bk.alloc<float>(NH);
    P->g_xp = Bk.alloc<float>(N * d);
  }
  if (P->Wy) {
    P->gY1 = Bk.alloc<float>(N * P->Wy);
    P->gWcat = Bk.alloc<float>(P->Wy * d + P->Wy);   // [gWcat | gbcat] contiguous: one memset
    P->gbcat = P->gWcat ? P->gWcat + P->Wy * d : nullptr;
  }
  if (P->gated) {
    P->g_e = Bk.alloc<float>(E * d);
    P->g_num = Bk.alloc<float>(N * d);
    if (P->es) {
      P->es_nw = gatedgcn_es_nwarps(d);
      P->es_ggate = Bk.alloc<float>(E * P->es_nw);
      P->es_gr = Bk.alloc<float>(E);
      P->es_work_bytes = es_gate_bwd_bytes(E, d);
      P->es_work = Bk.alloc<uint8_t>(P->es_work_bytes);
    }
  }
  if (P->gine) {
    P->g_h1 = Bk.alloc<float>(N * d);
    P->g_agg = Bk.alloc<float>(N * d);
    P->g_xl = Bk.alloc<float>(N * d);
  }
  if (P->use_planes) {
    P->gt_p = mkplanes(Bk, N, d);
    P->ghid_p = mkplanes(Bk, N, 2 * d);
    if (P->attn || P->perf) P->ghA_p = mkplanes(Bk, N, d);
    if (P->gated) P->ge_p = mkplanes(Bk, E, d);
    if (P->Wy) P->gY1_p = mkplanes(Bk, N, P->Wy);
    if (a->dropout > 0.f || (P->perf && a->attn_dropout > 0.f)) {
      P->gtmp_p = mkplanes(Bk, N, d);
      P->gtmp2_p = mkplanes(Bk, N, d);
      P->gtmp3_p = mkplanes(Bk, N, d);
    }
    if (P->gine) {
      P->gl1_p = mkplanes(Bk, N, d);
      P->gh1_p = mkplanes(Bk, N, d);
    }
  }
  P->bwd_bytes = Bk.used;
  return GPS_OK;
}

static BnView bn_view(const Plan& P, int which, const GpsBatchNorm& bn) {
  BnView v;
  v.mean = P.bnbuf + (int64_t)which * 2 * P.d;
  v.invstd = v.mean + P.d;
  v.gamma = bn.weight;
  v.beta = bn.bias;
  return v;
}

// forward view: the consumer kernel finalises the statistics itself (BnView mode 1 / 2)
static BnView bn_view_fwd(const Plan& P, const GpsLayerArgs* a, int which, const GpsBatchNorm& bn, int64_t n) {
  BnView v = bn_view(P, which, bn);
  v.d = P.d;
  v.running_mean = bn.running_mean;
  v.running_var = bn.running_var;
  if (a->training) {
    v.mode = 1;
    v.sums = P.fstats + (int64_t)which * 2 * P.d;
    v.inv_n = 1.0 / (double)(n > 0 ? n : 1);
    v.unbias = n > 1 ? (double)n / (double)(n - 1) : 1.0;
    v.save_mean = P.bnbuf + (int64_t)which * 2 * P.d;
    v.save_invstd = v.save_mean + P.d;
    v.nbt = (long long*)bn.num_batches_tracked;
  } else {
    v.mode = 2;
  }
  return v;
}

static PackDesc pack_desc(const GpsLayerArgs* a, const Plan& P) {
  PackDesc pd;
  memset(&pd, 0, sizeof(pd));
  pd.d = (int)P.d;
  auto add = [&](const GpsLinear& l, int rows) {
    pd.seg[pd.nseg++] = PackSeg{l.weight, l.bias, l.grad_weight, l.grad_bias, rows};
    pd.total_rows += rows;
  };
  if (P.gated) {
    add(a->gcn_A, (int)P.d);
    add(a->gcn_B, (int)P.d);
    add(a->gcn_D, (int)P.d);
    add(a->gcn_E, (int)P.d);
  }
  if (P.gcn) {   // GCNConv.lin has no bias; GCNConv.bias is added after the aggregation (scatter.cu)
    pd.seg[pd.nseg++] = PackSeg{a->gcn_conv.weight, nullptr, a->gcn_conv.grad_weight, nullptr, (int)P.d};
    pd.total_rows += (int)P.d;
  }
  if (P.attn) add(a->attn_in, (int)(3 * P.d));
  return pd;
}

static int check_linear(const GpsLinear& l, const char* name, bool need_bias) {
  GPS_REQUIRE(l.weight, GPS_ERR_ARG, "missing parameter %s.weight", name);
  GPS_REQUIRE(!need_bias || l.bias, GPS_ERR_ARG, "missing parameter %s.bias", name);
  return GPS_OK;
}
static int check_bn(const GpsBatchNorm& b, const char* name) {
  GPS_REQUIRE(b.weight && b.bias, GPS_ERR_ARG, "missing parameter %s.{weight,bias}", name);
  return GPS_OK;
}

static EsMlp es_mlp(const GpsLayerArgs* a) {
  return EsMlp{a->es_r0.weight, a->es_r0.bias, a->es_r1.weight, a->es_r1.bias,
               a->es_r0.grad_weight, a->es_r0.grad_bias, a->es_r1.grad_weight, a->es_r1.grad_bias};
}

static int check_params(const GpsLayerArgs* a, const Plan& P) {
  GPS_REQUIRE(a->x && (P.E == 0 || a->edge_attr || !(P.gated || P.gine)), GPS_ERR_ARG,
              "missing x / edge_attr");
  if (P.gated) {
    GPS_TRY(check_linear(a->gcn_A, "local_model.A", true));
    GPS_TRY(check_linear(a->gcn_B, "local_model.B", true));
    GPS_TRY(check_linear(a->gcn_C, "local_model.C", true));
    GPS_TRY(check_linear(a->gcn_D, "local_model.D", true));
    GPS_TRY(check_linear(a->gcn_E, "local_model.E", true));
    GPS_TRY(check_bn(a->bn_node_x, "local_model.bn_node_x"));
    GPS_TRY(check_bn(a->bn_edge_e, "local_model.bn_edge_e"));
  }
  if (P.es) {
    GPS_REQUIRE(a->pe && a->pe_dim > 0, GPS_ERR_ARG, "equivstable_pe: missing pe_EquivStableLapPE (pe / pe_dim)");
    GPS_TRY(check_linear(a->es_r0, "local_model.mlp_r_ij.0", true));
    GPS_TRY(check_linear(a->es_r1, "local_model.mlp_r_ij.2", true));
  }
  if (P.gine) {
    GPS_TRY(check_linear(a->gine_lin0, "local_model.nn.0", true));
    GPS_TRY(check_linear(a->gine_lin1, "local_model.nn.2", true));
  }
  if (P.gcn) GPS_TRY(check_linear(a->gcn_conv, "local_model.lin / local_model.bias", true));
  if (P.gated || P.gine || P.gcn) GPS_TRY(check_bn(a->norm1_local, "norm1_local"));
  if (P.attn) {
    GPS_TRY(check_linear(a->attn_in, "self_attn.in_proj", true));
    GPS_TRY(check_linear(a->attn_out, "self_attn.out_proj", true));
    GPS_TRY(check_bn(a->norm1_attn, "norm1_attn"));
  }
  if (P.perf) {
    GPS_TRY(check_linear(a->perf_q, "self_attn.to_q", false));
    GPS_TRY(check_linear(a->perf_k, "self_attn.to_k", false));
    GPS_TRY(check_linear(a->perf_v, "self_attn.to_v", false));
    GPS_TRY(check_linear(a->attn_out, "self_attn.to_out", true));
    GPS_REQUIRE(a->perf_proj, GPS_ERR_ARG, "missing buffer self_attn.fast_attention.projection_matrix");
    GPS_TRY(check_bn(a->norm1_attn, "norm1_attn"));
  }
  GPS_TRY(check_linear(a->ff1, "ff_linear1", true));
  GPS_TRY(check_linear(a->ff2, "ff_linear2", true));
  GPS_TRY(check_bn(a->norm2, "norm2"));
  return GPS_OK;
}

// set per call from GpsLayerArgs.reserved0 bit 0: the caller already zeroed every parameter-gradient buffer
// (one multi-tensor fill instead of a memset per weight and bias)
static thread_local bool g_grads_prezeroed = false;
// GpsLayerArgs.reserved0 bit 1: parameter gradients are ADDED to the caller's buffers (torch's .grad accumulation
// semantics on a static gradient bucket: graphgps_b200/dp.py); implies bit 0
static thread_local bool g_grads_accumulate = false;

static int splitk_for(int64_t rows, int64_t out = 304, int64_t in = 304) {
  // Weight gradients reduce over `rows` (nodes/edges) into a small [out, in] tile grid: split the reduction so
  // that tiles x splits ~ 300 CTAs (two per SM), at least 4 k-blocks of 64 rows per CTA (tools/gemm_tune.py).
  const int64_t tiles = ceil_div(out, 128) * ceil_div(in, in >= 160 ? 160 : 64);
  int64_t s = ceil_div(300, tiles > 0 ? tiles : 1);
  const int64_t max_s = rows / 256;
  if (s > max_s) s = max_s;
  if (s < 1) s = 1;
  if (s > 64) s = 64;
  return (int)s;
}

// weight gradient of a Linear: dW[out,in] = G[rows,out]^T X[rows,in], db[out] = colsum(G)
static int linear_wgrad(const float* G, int64_t ldg, const float* X, int64_t ldx, int64_t rows, int64_t out,
                        int64_t in, float* dW, float* db, int precision, cudaStream_t st, Planes Gp = Planes(),
                        Planes Xp = Planes()) {
  if (!dW) return GPS_OK;
  if (!g_grads_prezeroed) {
    GPS_CUDA(cudaMemsetAsync(dW, 0, (size_t)(out * in) * sizeof(float), st));
    if (db) GPS_CUDA(cudaMemsetAsync(db, 0, (size_t)out * sizeof(float), st));
  }
  if (rows == 0) return GPS_OK;
  GemmParams p;
  p.M = (int)out; p.N = (int)in; p.K = (int)rows;
  p.A = G; p.lda = (int)ldg; p.ta = 1;
  p.B = X; p.ldb = (int)ldx; p.tb = 1;
  p.C = dW; p.ldc = (int)in;
  p.splitk = splitk_for(rows, out, in);
  if (p.splitk == 1) p.splitk = 2;  // accumulate path (C pre-zeroed) also for tiny inputs
  p.colsum_a = db;
  p.precision = precision;
  p.Ap = Gp; p.Bp = Xp;
  if (precision == GPS_PREC_BF16 && Gp.hi && db) {
    // bf16 mode stores no lo plane: summing ~N bf16-rounded rows would put ~sqrt(N) 2^-9 of noise on a bias gradient
    // that is often a near-cancelling sum (every Linear here feeds a BatchNorm) -> exact fp32 column sum instead
    p.colsum_a = nullptr;
    GPS_TRY(colsum(G, ldg, rows, out, db, st));
  }
  return gemm(p, st);
}

}  // namespace

// =================================================================================== forward
static int layer_forward(const GpsLayerArgs* a, cudaStream_t st) {
  Plan P;
  GPS_TRY(make_plan(a, &P, true));
  GPS_REQUIRE(a->saved && a->workspace, GPS_ERR_ARG, "saved/workspace buffers are required");
  GPS_REQUIRE(a->workspace_bytes >= P.fwd_bytes, GPS_ERR_ARG, "workspace too small (%lld < %lld)",
              (long long)a->workspace_bytes, (long long)P.fwd_bytes);
  GPS_TRY(check_params(a, P));
  GPS_REQUIRE(a->x_out, GPS_ERR_ARG, "x_out is null");
  const int64_t N = P.N, E = P.E, d = P.d;
  const int act = a->act;
  const bool train = a->training != 0;
  const float pd = train ? a->dropout : 0.f;
  const float pa = train ? a->attn_dropout : 0.f;
  auto drop = [&](int site) {
    DropCfg c;
    c.p = pd; c.seed = a->seed; c.offset = a->offset; c.site = site;
    c.offset_dev = (const unsigned long long*)a->offset_dev;
    return c;
  };
  auto stats = [&](int which) -> double* { return train ? P.fstats + (int64_t)which * 2 * d : nullptr; };
  auto out_planes = [&](const GpsPlanes& g) {   // planes of this layer's outputs for the next layer of the stack
    Planes q;
    if (P.use_planes && g.hi && g.ld >= d && g.ld % 8 == 0) {
      q.hi = (__nv_bfloat16*)g.hi;
      q.lo = a->precision == GPS_PREC_FP32 ? (__nv_bfloat16*)g.lo : nullptr;
      q.ld = g.ld;
      if (a->precision == GPS_PREC_FP32 && !q.lo) q = Planes();
    }
    return q;
  };

  if (train) GPS_CUDA(cudaMemsetAsync(P.fstats, 0, (size_t)BN_COUNT * 2 * d * sizeof(double), st));
  Side* sd = side_stream();
  cudaStream_t s2 = sd ? sd->s : st;
  const bool two_branches = (P.gated || P.gine || P.gcn) && (P.attn || P.perf);

  // weights: concatenate the node projections, then pre-pack every forward weight into the tcgen05 kernel's
  // shared-memory tile image (bf16 hi/lo planes) so its B operand arrives by bulk TMA
  if (P.Wy) {
    PackDesc pdsc0 = pack_desc(a, P);
    k_pack<<<(unsigned)pdsc0.total_rows, 128, 0, st>>>(pdsc0, P.Wcat, P.bcat);
    GPS_LAUNCH_CHECK();
  }
  auto set_bpk = [&](GemmParams& g, const uint8_t* pk, int64_t rows, int64_t K, int64_t row0) {
    if (!P.prepack || !pk) return;
    g.bpk = pk;
    g.bpk_lo_off = prepack_plane_bytes((int)rows, (int)K);
    g.bpk_groups = prepack_groups((int)rows);
    g.bpk_row0 = (int)row0;
  };
  // Weight planes: the ones the first GEMMs need are packed on the caller's stream; the rest (output projection,
  // FFN, and the MN-major images the backward pass reads) are packed next to those GEMMs on their own stream.
  cudaStream_t sp = sd ? sd->s4 : st;
  if (P.use_planes) {
    // layer inputs and every weight -> bf16 hi/lo planes, one launch (the producers inside the layer write the
    // planes of their outputs themselves).  Wcat_p rows follow pack_desc(): [A;B;D;E | conv] then in_proj.
    ToPlanesItem it[16];
    int ni = 0;
    auto add = [&](const float* src, int64_t ld, int64_t rows, int64_t cols, Planes dst) {
      if (src && dst.hi && rows > 0) it[ni++] = ToPlanesItem{src, ld, (int)rows, (int)cols, dst};
    };
    const int64_t kout = P.perf ? P.inner : d;
    if (P.x_p.hi != (__nv_bfloat16*)a->x_planes_in.hi) add(a->x, d, N, d, P.x_p);
    if ((P.gated || P.gine) && P.e_p.hi != (__nv_bfloat16*)a->e_planes_in.hi) add(a->edge_attr, d, E, d, P.e_p);
    const bool wvalid = a->wplanes && a->wplanes_valid;
    if (wvalid) goto weights_done;
    if (P.gated) {
      add(a->gcn_A.weight, d, d, d, P.Wcat_p.rows(0));
      add(a->gcn_B.weight, d, d, d, P.Wcat_p.rows(d));
      add(a->gcn_D.weight, d, d, d, P.Wcat_p.rows(2 * d));
      add(a->gcn_E.weight, d, d, d, P.Wcat_p.rows(3 * d));
      add(a->gcn_C.weight, d, d, d, P.C_p);
    }
    if (P.gcn) add(a->gcn_conv.weight, d, d, d, P.Wcat_p.rows(0));
    if (P.attn) add(a->attn_in.weight, d, 3 * d, d, P.Wcat_p.rows(P.qkv_off));
    if (P.gine) {
      add(a->gine_lin0.weight, d, d, d, P.g0_p);
      add(a->gine_lin1.weight, d, d, d, P.g1_p);
    }
    if (P.attn || P.perf) add(a->attn_out.weight, kout, d, kout, P.out_p);
    add(a->ff1.weight, d, 2 * d, d, P.ff1_p);
    add(a->ff2.weight, 2 * d, d, 2 * d, P.ff2_p);
    if (P.perf) {
      add(a->perf_q.weight, d, P.inner, d, P.pq_p);
      add(a->perf_k.weight, d, P.inner, d, P.pk_p);
      add(a->perf_v.weight, d, P.inner, d, P.pv_p);
    }
  weights_done:
    GPS_TRY(to_planes(it, ni, st));
  }
  if (P.prepack && !P.use_planes) {
    PrepackItem items[16];
    int ni = 0;
    const int64_t kout = P.perf ? P.inner : d;
    if (P.Wy) items[ni++] = PrepackItem{P.Wcat, (int)P.Wy, (int)d, (int)d, P.pk_cat};
    if (P.gated) items[ni++] = PrepackItem{a->gcn_C.weight, (int)d, (int)d, (int)d, P.pk_C};
    if (P.gine) {
      items[ni++] = PrepackItem{a->gine_lin0.weight, (int)d, (int)d, (int)d, P.pk_g0};
      items[ni++] = PrepackItem{a->gine_lin1.weight, (int)d, (int)d, (int)d, P.pk_g1};
    }
    GPS_TRY(prepack_weights(items, ni, st));
    ni = 0;
    if (sp != st) GPS_TRY(sd->order(st, sp));
    if (P.attn || P.perf) items[ni++] = PrepackItem{a->attn_out.weight, (int)d, (int)kout, (int)kout, P.pk_out};
    items[ni++] = PrepackItem{a->ff1.weight, (int)(2 * d), (int)d, (int)d, P.pk_ff1};
    items[ni++] = PrepackItem{a->ff2.weight, (int)d, (int)(2 * d), (int)(2 * d), P.pk_ff2};
    if (a->training && (opt_flags() & 1)) {   // MN-major images for the backward data gradients: W is [K x N] there
      if (P.Wy) items[ni++] = PrepackItem{P.Wcat, (int)d, (int)P.Wy, (int)d, P.pt_cat, 1};
      if (P.gated) items[ni++] = PrepackItem{a->gcn_C.weight, (int)d, (int)d, (int)d, P.pt_C, 1};
      if (P.attn || P.perf) items[ni++] = PrepackItem{a->attn_out.weight, (int)kout, (int)d, (int)kout, P.pt_out, 1};
      items[ni++] = PrepackItem{a->ff1.weight, (int)d, (int)(2 * d), (int)d, P.pt_ff1, 1};
      items[ni++] = PrepackItem{a->ff2.weight, (int)(2 * d), (int)d, (int)(2 * d), P.pt_ff2, 1};
      if (P.gine) {
        items[ni++] = PrepackItem{a->gine_lin0.weight, (int)d, (int)d, (int)d, P.pt_g0, 1};
        items[ni++] = PrepackItem{a->gine_lin1.weight, (int)d, (int)d, (int)d, P.pt_g1, 1};
      }
    }
    GPS_TRY(prepack_weights(items, ni, sp));
  }
  if (P.gated) {   // edge projection has no dependency on the node side: run it next to the node projections
    GPS_REQUIRE(a->edge_out, GPS_ERR_ARG, "edge_out is null");
    if (sd) GPS_TRY(sd->fork(st));
    GemmParams g;  // Ce = e C^T + bC (gatedgcn_layer.py:59)
    g.M = (int)E; g.N = (int)d; g.K = (int)d;
    g.A = a->edge_attr; g.lda = (int)d; g.B = a->gcn_C.weight; g.ldb = (int)d; g.C = P.ehat; g.ldc = (int)d;
    g.bias = a->gcn_C.bias; g.precision = a->precision;
    set_bpk(g, P.pk_C, d, d, 0);
    g.Ap = P.e_p; g.Bp = P.C_p;
    GPS_TRY(gemm(g, s2));
    // EquivStableLapPE gate: PE and mlp_r_ij only, next to the edge projection (joined before the aggregation)
    if (P.es) GPS_TRY(es_gate_fwd(a->graph, a->pe, a->pe_dim, d, act, es_mlp(a), P.es_r, P.es_g, s2));
  }

  // ---- node projections: [Ax|Bx|Dx|Ex|Q|K|V] = x Wcat^T + bcat  (gatedgcn_layer.py:57-61, MHA in_proj)
  // The two consumers of the projections get their own GEMM: [Ax|Bx|Dx|Ex] on the main stream for the
  // message-passing branch, [Q|K|V] on the attention branch's stream, so both branches start ~25 us after the
  // pack instead of after one 50 us GEMM.
  cudaStream_t sg = st;   // stream of the global-attention branch
  if (two_branches && sd) {
    GPS_TRY(sd->order(st, sd->s3));
    sg = sd->s3;
  }
  if (P.Wy) {
    const int64_t wl = P.qkv_off, wg = P.Wy - P.qkv_off;   // local / global column blocks
    if (wg > 0) {
      GemmParams g;
      g.M = (int)N; g.N = (int)wg; g.K = (int)d;
      g.A = a->x; g.lda = (int)d; g.B = P.Wcat + wl * d; g.ldb = (int)d; g.C = P.Y1 + wl; g.ldc = (int)P.Wy;
      g.bias = P.bcat + wl; g.precision = a->precision;
      set_bpk(g, P.pk_cat, P.Wy, d, wl);
      g.Ap = P.x_p; g.Bp = P.Wcat_p.rows(wl);
      if (P.attn_tc) {   // Q | K | V additionally as padded per-head operand planes for the tcgen05 attention
        g.Cp = P.qkv_p; g.cp_hd = (int)P.hd; g.cp_hd_pad = (int)attention_tc_hd_pad(P.hd); g.cp_col0 = 0;
      }
      GPS_TRY(gemm(g, sg));
    }
    if (wl > 0) {
      GemmParams g;
      g.M = (int)N; g.N = (int)wl; g.K = (int)d;
      g.A = a->x; g.lda = (int)d; g.B = P.Wcat; g.ldb = (int)d; g.C = P.Y1; g.ldc = (int)P.Wy;
      g.bias = P.bcat; g.precision = a->precision;
      set_bpk(g, P.pk_cat, P.Wy, d, 0);
      g.Ap = P.x_p; g.Bp = P.Wcat_p;
      GPS_TRY(gemm(g, st));
    }
  }

  // main waits for the edge projection
  if (P.gated && sd) GPS_TRY(sd->join(st));

  // ---- local model
  if (P.gated) {
    GPS_TRY(gatedgcn_fwd(a->graph, d, P.Y1, P.Y1 + d, P.Y1 + 2 * d, P.Y1 + 3 * d, P.Wy, P.ehat, P.xt,
                         stats(BN_X), stats(BN_E), st, P.es ? P.es_g : nullptr));
    // x_loc = x + drop(act(BN(x~)));  e_out = e + drop(act(BN(e^)))   (gatedgcn_layer.py:72-83)
    GPS_TRY(bn_act_residual2(P.xt, a->x, P.xloc, N, bn_view_fwd(P, a, BN_X, a->bn_node_x, N), drop(GPS_SITE_GCN_X), stats(BN_L),
                             P.ehat, a->edge_attr, a->edge_out, E, bn_view_fwd(P, a, BN_E, a->bn_edge_e, E),
                             drop(GPS_SITE_GCN_E), out_planes(a->e_planes_out), d, act, st));
  } else if (P.gine) {
    GPS_TRY(gine_fwd(a->graph, d, a->x, a->edge_attr, a->gine_eps, P.agg, st, P.agg_p));
    GemmParams g;  // h1 = act(agg W0^T + b0)
    g.M = (int)N; g.N = (int)d; g.K = (int)d;
    g.A = P.agg; g.lda = (int)d; g.B = a->gine_lin0.weight; g.ldb = (int)d; g.C = P.h1; g.ldc = (int)d;
    g.bias = a->gine_lin0.bias; g.act = act; g.C_pre = P.h1_pre; g.ldpre = (int)d; g.precision = a->precision;
    set_bpk(g, P.pk_g0, d, d, 0);
    g.Ap = P.agg_p; g.Bp = P.g0_p; g.Cp = P.h1_p;
    GPS_TRY(gemm(g, st));
    GemmParams g2;  // x_loc = x + drop(h1 W1^T + b1)  (gps_layer.py:188-189)
    g2.M = (int)N; g2.N = (int)d; g2.K = (int)d;
    g2.A = P.h1; g2.lda = (int)d; g2.B = a->gine_lin1.weight; g2.ldb = (int)d; g2.C = P.xloc; g2.ldc = (int)d;
    g2.bias = a->gine_lin1.bias; g2.R1 = a->x; g2.ldr1 = (int)d; g2.stats = stats(BN_L);
    g2.p_drop = pd; g2.seed = a->seed; g2.offset = a->offset; g2.site = GPS_SITE_LOCAL;
    g2.offset_dev = (const unsigned long long*)a->offset_dev;
    g2.precision = a->precision;
    set_bpk(g2, P.pk_g1, d, d, 0);
    g2.Ap = P.h1_p; g2.Bp = P.g1_p;
    GPS_TRY(gemm(g2, st));
  } else if (P.gcn) {
    // x_loc = x + drop(GCNConv(x))  (gps_layer.py:49-51,186-189); Y = x W^T is column block 0 of Y1
    GPS_TRY(gcn_dinv(a->graph, P.dinv, st));
    GPS_TRY(gcn_fwd(a->graph, d, P.Y1, P.Wy, P.dinv, a->gcn_conv.bias, a->x, P.xloc, drop(GPS_SITE_LOCAL), stats(BN_L), st));
  }

  // ---- global attention  (gps_layer.py:198-218, 234-241)
  if (P.attn) {
    const float* Q = P.Y1 + P.qkv_off;
    if (P.attn_tc)
      GPS_TRY(attention_tc_fwd(a->graph, P.H, P.hd, P.qkv_p, P.O, d, P.O_p, P.lse, pa, a->seed, a->offset,
                               (const unsigned long long*)a->offset_dev, a->precision, sg));
    else
      GPS_TRY(attention_fwd(a->graph, P.H, P.hd, Q, Q + d, Q + 2 * d, P.Wy, P.O, d, P.lse, pa, a->seed, a->offset, sg,
                            (const unsigned long long*)a->offset_dev, P.O_p));
    GemmParams g;  // hA = x + drop(O Wo^T + bo)
    g.M = (int)N; g.N = (int)d; g.K = (int)d;
    g.A = P.O; g.lda = (int)d; g.B = a->attn_out.weight; g.ldb = (int)d; g.C = P.hA; g.ldc = (int)d;
    g.bias = a->attn_out.bias; g.R1 = a->x; g.ldr1 = (int)d; g.stats = stats(BN_A);
    g.p_drop = pd; g.seed = a->seed; g.offset = a->offset; g.site = GPS_SITE_ATTN_OUT;
    g.offset_dev = (const unsigned long long*)a->offset_dev;
    g.precision = a->precision;
    set_bpk(g, P.pk_out, d, d, 0);
    g.Ap = P.O_p; g.Bp = P.out_p;
    if (P.prepack && !P.use_planes && sp != st) GPS_TRY(sd->order(sp, sg));
    GPS_TRY(gemm(g, sg));
  }

  // ---- Performer global attention (gps_layer.py:205-206; performer_layer.py:476-503)
  if (P.perf) {
    const int64_t inner = P.inner, NH = N * P.H, dh = a->perf_dim_head;
    const GpsLinear* lin[3] = {&a->perf_q, &a->perf_k, &a->perf_v};
    float* dst[3] = {P.pQ, P.pK, P.pV};
    for (int i = 0; i < 3; ++i) {   // q, k, v = x W^T (no bias)
      GemmParams g;
      g.M = (int)N; g.N = (int)inner; g.K = (int)d;
      g.A = a->x; g.lda = (int)d; g.B = lin[i]->weight; g.ldb = (int)d; g.C = dst[i]; g.ldc = (int)inner;
      g.precision = a->precision;
      g.Ap = P.x_p; g.Bp = i == 0 ? P.pq_p : (i == 1 ? P.pk_p : P.pv_p);
      GPS_TRY(gemm(g, sg));
    }
    GPS_TRY(perf_prep(a->perf_proj, P.m, P.pPn, a->graph, P.H, P.pnmax, P.pgmax, P.pargk, sg));
    float* ddst[2] = {P.pfq, P.pfk};
    for (int i = 0; i < 2; ++i) {   // dd = (x dn) P^T for every (node, head) row
      GemmParams g;
      g.M = (int)NH; g.N = (int)P.mp; g.K = (int)dh;
      g.A = dst[i]; g.lda = (int)dh; g.B = P.pPn; g.ldb = (int)dh; g.C = ddst[i]; g.ldc = (int)P.mp;
      g.precision = a->precision;
      GPS_TRY(gemm(g, sg));
    }
    GPS_TRY(perf_features_fwd(P.pfq, P.pfk, P.pQ, P.pK, a->graph, P.H, P.m, P.pgmax, P.pargq, P.pargk, sg));
    if (P.perf_pairwise)
      GPS_TRY(perf_quad_fwd(a->graph, P.H, P.m, P.pnmax, P.pfq, P.pfk, P.pV, P.pgmax, P.O, P.pden, sg));
    else
      GPS_TRY(perf_linattn_fwd(a->graph, P.H, P.m, P.pnmax, P.pfq, P.pfk, P.pV, P.pgmax, P.O, sg));
    GemmParams g;  // hA = x + drop(to_out(O))
    g.M = (int)N; g.N = (int)d; g.K = (int)inner;
    g.A = P.O; g.lda = (int)inner; g.B = a->attn_out.weight; g.ldb = (int)inner; g.C = P.hA; g.ldc = (int)d;
    g.bias = a->attn_out.bias; g.R1 = a->x; g.ldr1 = (int)d; g.stats = stats(BN_A);
    // SelfAttention ends with dropout(p = attn_dropout) on to_out(O) (performer_layer.py:501-503, built with
    // dropout=self.attn_dropout at gps_layer.py:112-114); GPSLayer.dropout_attn (p = dropout) follows (:212)
    g.p_drop = pd > 0.f ? pd : 0.f; g.seed = a->seed; g.offset = a->offset; g.site = GPS_SITE_ATTN_OUT;
    g.p_drop2 = pa; g.site2 = GPS_SITE_PERF_OUT;
    g.offset_dev = (const unsigned long long*)a->offset_dev;
    g.precision = a->precision;
    GPS_TRY(gemm(g, sg));
  }

  if (two_branches && sd) GPS_TRY(sd->order(sd->s3, st));

  // ---- s = norm1_local(x_loc) + norm1_attn(hA)   (gps_layer.py:194,217,222)
  {
    const bool loc = P.gated || P.gine || P.gcn;
    const float* first = loc ? P.xloc : P.hA;
    BnView bf = loc ? bn_view_fwd(P, a, BN_L, a->norm1_local, N) : bn_view_fwd(P, a, BN_A, a->norm1_attn, N);
    const float* second = (loc && (P.attn || P.perf)) ? P.hA : nullptr;
    BnView bs = bn_view_fwd(P, a, BN_A, a->norm1_attn, N);
    GPS_TRY(bn_combine(first, bf, second, bs, P.s, N, d, st, P.s_p));
  }

  // ---- FFN: t = s + drop(W2 drop(act(W1 s + b1)) + b2)   (gps_layer.py:225, 253-257)
  {
    if (P.prepack && !P.use_planes && sp != st) GPS_TRY(sd->order(sp, st));
    GemmParams g;
    g.M = (int)N; g.N = (int)(2 * d); g.K = (int)d;
    g.A = P.s; g.lda = (int)d; g.B = a->ff1.weight; g.ldb = (int)d; g.C = P.hid; g.ldc = (int)(2 * d);
    g.bias = a->ff1.bias; g.act = act; g.C_pre = P.hid_pre; g.ldpre = (int)(2 * d);
    g.p_drop = pd; g.seed = a->seed; g.offset = a->offset; g.site = GPS_SITE_FF1; g.precision = a->precision;
    g.offset_dev = (const unsigned long long*)a->offset_dev;
    set_bpk(g, P.pk_ff1, 2 * d, d, 0);
    g.Ap = P.s_p; g.Bp = P.ff1_p; g.Cp = P.hid_p;
    GPS_TRY(gemm(g, st));
    GemmParams g2;
    g2.M = (int)N; g2.N = (int)d; g2.K = (int)(2 * d);
    g2.A = P.hid; g2.lda = (int)(2 * d); g2.B = a->ff2.weight; g2.ldb = (int)(2 * d); g2.C = P.t; g2.ldc = (int)d;
    g2.bias = a->ff2.bias; g2.R1 = P.s; g2.ldr1 = (int)d; g2.stats = stats(BN_2);
    g2.p_drop = pd; g2.seed = a->seed; g2.offset = a->offset; g2.site = GPS_SITE_FF2; g2.precision = a->precision;
    g2.offset_dev = (const unsigned long long*)a->offset_dev;
    set_bpk(g2, P.pk_ff2, d, 2 * d, 0);
    g2.Ap = P.hid_p; g2.Bp = P.ff2_p;
    GPS_TRY(gemm(g2, st));
    GPS_TRY(bn_combine(P.t, bn_view_fwd(P, a, BN_2, a->norm2, N), nullptr, BnView(), a->x_out, N, d, st,
                       out_planes(a->x_planes_out)));  // :229
  }
  return GPS_OK;
}

// =================================================================================== backward
// out = a * dropout_scale(site)  (only launched when p > 0)
static int dropmul(const float* src, float* dst, int64_t rows, int64_t d, const Plan& P, const GpsLayerArgs* a,
                   int site, cudaStream_t st, float p2 = 0.f, int site2 = 0, Planes dstp = Planes());

static int layer_backward(const GpsLayerArgs* a, cudaStream_t st) {
  Plan P;
  GPS_TRY(make_plan(a, &P, true));
  GPS_REQUIRE(a->saved && a->workspace, GPS_ERR_ARG, "saved/workspace buffers are required");
  GPS_REQUIRE(a->workspace_bytes >= P.bwd_bytes, GPS_ERR_ARG, "workspace too small (%lld < %lld)",
              (long long)a->workspace_bytes, (long long)P.bwd_bytes);
  GPS_TRY(check_params(a, P));
  // eval mode (running statistics, no dropout): BatchNorm is a per-column affine map, its backward has no batch terms
  g_grads_accumulate = (a->reserved0 & 2) != 0;
  g_grads_prezeroed = (a->reserved0 & 1) != 0 || g_grads_accumulate;
  GPS_REQUIRE(a->grad_x_out && a->grad_x, GPS_ERR_ARG, "grad_x_out / grad_x are required");
  const int64_t N = P.N, E = P.E, d = P.d;
  const int act = a->act, prec = a->precision;
  const float pd = a->training ? a->dropout : 0.f, pa = a->training ? a->attn_dropout : 0.f;
  const bool relu = act == GPS_ACT_RELU;
  auto drop = [&](int site) {
    DropCfg c;
    c.p = pd; c.seed = a->seed; c.offset = a->offset; c.site = site;
    c.offset_dev = (const unsigned long long*)a->offset_dev;
    return c;
  };
  DropCfg nodrop;
  // training: the batch statistics saved by the forward pass; eval: the running statistics the forward pass used
  auto bview = [&](int which, const GpsBatchNorm& bn) {
    BnView v = bn_view(P, which, bn);
    if (!a->training) {
      v.mode = 2;
      v.running_mean = bn.running_mean;
      v.running_var = bn.running_var;
    }
    return v;
  };
  auto sums = [&](int which) { return P.bsums + (int64_t)which * 2 * d; };
  GPS_CUDA(cudaMemsetAsync(P.bsums, 0, (size_t)BN_COUNT * 2 * d * sizeof(double), st));
  // weight-gradient GEMMs run on the side stream, each forked where its operands become final
  Side* sd = side_stream();
  cudaStream_t s2 = sd ? sd->s : st;
  auto wfork = [&](cudaStream_t from) -> int { return sd ? sd->order(from, s2) : GPS_OK; };
  const bool two_branches = (P.gated || P.gine || P.gcn) && (P.attn || P.perf);
  cudaStream_t sa = (two_branches && sd) ? sd->s3 : st;   // stream of the attention-branch backward
  const int opt = opt_flags();
  const bool early_edge = (opt & 4) != 0;
  // data-parallel hook: the caller's event is recorded on the weight-gradient stream once the early gradient group
  // (FFN, attention output projection, norm2 / norm1_local / norm1_attn) has been enqueued there
  // (recorded as EXTERNAL events under stream capture, so that collectives enqueued outside the captured graph can wait
  // on them after each replay: NCCL kernels inside a graph cost ~0.5 ms of host time per launch on this stack)
  auto record_ev = [&](void* ev, cudaStream_t s) -> int {
    if (!ev) return GPS_OK;
    cudaStreamCaptureStatus cs = cudaStreamCaptureStatusNone;
    GPS_CUDA(cudaStreamIsCapturing(s, &cs));
    GPS_CUDA(cudaEventRecordWithFlags((cudaEvent_t)ev, s, cs == cudaStreamCaptureStatusActive ? cudaEventRecordExternal
                                                                                               : cudaEventRecordDefault));
    return GPS_OK;
  };
  auto early_done = [&]() -> int { return record_ev(a->ev_grads_early, s2); };
  // accumulators of the last two GEMMs of the pass are zeroed now, while their streams are idle, instead of on the tail
  const bool gx_splitk = P.Wy >= 1024 && N > 0 && !((opt & 8) && P.gated && P.attn && sd && P.qkv_off > 0 && P.qkv_off < P.Wy);
  if (P.Wy) {
    if (sd) GPS_TRY(sd->order(st, s2));
    GPS_CUDA(cudaMemsetAsync(P.gWcat, 0, (size_t)(P.Wy * d + P.Wy) * sizeof(float), s2));
  }
  if (gx_splitk) GPS_CUDA(cudaMemsetAsync(a->grad_x, 0, (size_t)(N * d) * sizeof(float), st));
  // [Ax|Bx|Dx|Ex] gradients are final long before [Q|K|V]'s: their share of dWcat and of g_x = gY1 Wcat is
  // computed under the attention backward, leaving only the [Q|K|V] share for the tail of the pass
  const bool split_tail = (opt & 8) && P.gated && P.attn && sd && P.qkv_off > 0 && P.qkv_off < P.Wy && N > 0;
  auto wcat_wgrad = [&](int64_t r0, int64_t rows) -> int {   // d Wcat[r0 : r0 + rows] (+ bias gradient) on s2
    GemmParams w;
    w.M = (int)rows; w.N = (int)d; w.K = (int)N;
    w.A = P.gY1 + r0; w.lda = (int)P.Wy; w.ta = 1; w.B = a->x; w.ldb = (int)d; w.tb = 1;
    w.C = P.gWcat + r0 * d; w.ldc = (int)d;
    w.splitk = splitk_for(N, rows, d) < 2 ? 2 : splitk_for(N, rows, d);
    w.colsum_a = P.gbcat + r0; w.precision = prec;
    w.Ap = P.gY1_p.cols(r0); w.Bp = P.x_p;
    if (prec == GPS_PREC_BF16 && w.Ap.hi && N > 0) {
      w.colsum_a = nullptr;
      GPS_TRY(colsum(P.gY1 + r0, P.Wy, N, rows, P.gbcat + r0, s2));
    }
    return N > 0 ? gemm(w, s2) : GPS_OK;
  };
  // The weight gradient of the fused node projection in two parts (GPS_B200_OPT bit 16, default on): rows [0, qkv_off)
  // (A, B, D, E / GCN lin) as soon as the message-passing backward has produced their gY1 columns - under the attention
  // backward - and the in_proj rows at the end.  Shortens the tail of the pass and lets a data-parallel caller reduce
  // the local model's gradients early (ev_grads_mid).
  const bool wgrad_split = (opt & 16) && sd && !((opt & 8) && P.gated && P.attn) && P.qkv_off > 0 && P.qkv_off < P.Wy && N > 0;
  auto unpack_rows = [&](int64_t r0, int64_t rows) -> int {
    PackDesc pdsc = pack_desc(a, P);
    k_unpack<<<(unsigned)rows, 128, 0, s2>>>(pdsc, P.gWcat, P.gbcat, g_grads_accumulate ? 1 : 0, (int)r0);
    GPS_LAUNCH_CHECK();
    return GPS_OK;
  };
  auto mid_done = [&]() -> int {   // on s2, after the local model's weight gradients
    if (wgrad_split) {
      GPS_TRY(wcat_wgrad(0, P.qkv_off));
      GPS_TRY(unpack_rows(0, P.qkv_off));
    }
    return record_ev(a->ev_grads_mid, s2);
  };

  cudaStream_t se = (P.gated && sd && early_edge) ? sd->s4 : st;   // stream of the edge BatchNorm backward
  // data gradients g_in = g_out W read W through the MN-major planes packed by the forward pass
  auto set_bpt = [&](GemmParams& g, const uint8_t* pt, int64_t cols, int64_t K) {
    if (!P.prepack || !pt || !(opt & 1)) return;
    g.bpk = pt;
    g.bpk_mn = 1;
    g.bpk_lo_off = prepack_plane_bytes_mn((int)cols, (int)K);
    g.bpk_groups = prepack_groups_mn((int)cols);
    g.bpk_row0 = 0;
  };

  auto edge_bn_bwd = [&]() -> int {
    // e_out = e + drop(act(BN_e(e^))) (gatedgcn_layer.py:76-83): g_e^ needs grad_edge_out alone -> off the critical path
    if (se != st) GPS_TRY(sd->order(st, se));
    BnView ve = bview(BN_E, a->bn_edge_e);
    if (a->grad_edge_out && E > 0) {
      GPS_TRY(bn_bwd_reduce(a->grad_edge_out, d, P.ehat, d, E, d, ve, act, drop(GPS_SITE_GCN_E), sums(BN_E), se));
      GPS_TRY(bn_bwd_apply(a->grad_edge_out, d, P.ehat, d, E, d, ve, act, drop(GPS_SITE_GCN_E), sums(BN_E), P.g_e, d,
                           a->bn_edge_e.grad_weight, a->bn_edge_e.grad_bias, se, g_grads_accumulate));
    } else {
      if (E > 0) GPS_CUDA(cudaMemsetAsync(P.g_e, 0, (size_t)(E * d) * sizeof(float), se));
      if (a->bn_edge_e.grad_weight && !g_grads_prezeroed)
        GPS_CUDA(cudaMemsetAsync(a->bn_edge_e.grad_weight, 0, d * sizeof(float), se));
      if (a->bn_edge_e.grad_bias && !g_grads_prezeroed)
        GPS_CUDA(cudaMemsetAsync(a->bn_edge_e.grad_bias, 0, d * sizeof(float), se));
    }
    return GPS_OK;
  };
  if (P.gated && early_edge) GPS_TRY(edge_bn_bwd());

  // ---- norm2 (gps_layer.py:229): g_t
  BnView v2 = bview(BN_2, a->norm2);
  GPS_TRY(bn_bwd_reduce(a->grad_x_out, d, P.t, d, N, d, v2, -1, nodrop, sums(BN_2), st));
  GPS_TRY(bn_bwd_apply(a->grad_x_out, d, P.t, d, N, d, v2, -1, nodrop, sums(BN_2), P.g_t, d, a->norm2.grad_weight,
                       a->norm2.grad_bias, st, g_grads_accumulate, P.gt_p));

  bool fused_la = false;
  // ---- FFN (gps_layer.py:253-257)
  const float* g_ff2 = P.g_t;  // gradient at the output of ff_linear2 (after ff_dropout2)
  Planes g_ff2_p = P.gt_p;
  if (pd > 0.f) {
    GPS_TRY(dropmul(P.g_t, P.g_tmp, N, d, P, a, GPS_SITE_FF2, st, 0.f, 0, P.gtmp_p));
    g_ff2 = P.g_tmp;
    g_ff2_p = P.gtmp_p;
  }
  {
    GemmParams g;  // g_hid = (g_ff2 W2) * act'(pre) * drop1
    g.M = (int)N; g.N = (int)(2 * d); g.K = (int)d;
    g.A = g_ff2; g.lda = (int)d; g.B = a->ff2.weight; g.ldb = (int)(2 * d); g.tb = 1; g.C = P.g_hid; g.ldc = (int)(2 * d);
    if (relu) { g.mask_src = P.hid; g.mask_is_post = 1; } else { g.mask_src = P.hid_pre; g.mask_act = act; }
    g.ldmask = (int)(2 * d);
    g.p_drop = pd; g.seed = a->seed; g.offset = a->offset; g.site = GPS_SITE_FF1; g.precision = prec;
    g.offset_dev = (const unsigned long long*)a->offset_dev;
    set_bpt(g, P.pt_ff2, 2 * d, d);
    g.Ap = g_ff2_p; g.Bp = P.ff2_p; g.Cp = P.ghid_p;
    GPS_TRY(gemm(g, st));
    GPS_TRY(wfork(st));
    GPS_TRY(linear_wgrad(g_ff2, d, P.hid, 2 * d, N, d, 2 * d, a->ff2.grad_weight, a->ff2.grad_bias, prec, s2, g_ff2_p, P.hid_p));
    GPS_TRY(linear_wgrad(P.g_hid, 2 * d, P.s, d, N, 2 * d, d, a->ff1.grad_weight, a->ff1.grad_bias, prec, s2, P.ghid_p, P.s_p));
    GemmParams g2;  // g_s = g_t + g_hid W1
    g2.M = (int)N; g2.N = (int)d; g2.K = (int)(2 * d);
    g2.A = P.g_hid; g2.lda = (int)(2 * d); g2.B = a->ff1.weight; g2.ldb = (int)d; g2.tb = 1; g2.C = P.g_s; g2.ldc = (int)d;
    g2.R1 = P.g_t; g2.ldr1 = (int)d; g2.precision = prec;
    set_bpt(g2, P.pt_ff1, d, 2 * d);
    g2.Ap = P.ghid_p; g2.Bp = P.ff1_p;
    // norm1_local and norm1_attn both take g_s as their upstream gradient (gps_layer.py:194,217,222): their backward
    // reductions ride this GEMM's epilogue instead of two more passes over g_s (GPS_B200_OPT bit 64)
    fused_la = (opt & 64) && P.use_planes && g2.Ap.hi && g2.Bp.hi && N > 0 && a->training;
    if (fused_la) {
      if (P.gated || P.gine || P.gcn) {
        BnView v = bview(BN_L, a->norm1_local);
        g2.bnred[0].z = P.xloc; g2.bnred[0].ldz = (int)d; g2.bnred[0].mean = v.mean; g2.bnred[0].invstd = v.invstd;
        g2.bnred[0].sums = sums(BN_L);
      }
      if (P.attn || P.perf) {
        BnView v = bview(BN_A, a->norm1_attn);
        g2.bnred[1].z = P.hA; g2.bnred[1].ldz = (int)d; g2.bnred[1].mean = v.mean; g2.bnred[1].invstd = v.invstd;
        g2.bnred[1].sums = sums(BN_A);
      }
    }
    GPS_TRY(gemm(g2, st));
  }

  const bool loc = P.gated || P.gine || P.gcn;
  bool chain_x = false;
  // ---- norm1_local / norm1_attn (gps_layer.py:194,217): g_xloc, g_hA
  if (loc) {
    BnView v = bview(BN_L, a->norm1_local);
    if (!fused_la) GPS_TRY(bn_bwd_reduce(P.g_s, d, P.xloc, d, N, d, v, -1, nodrop, sums(BN_L), st));
    chain_x = P.gated && N > 0 && (opt & 32) && a->training;
    if (chain_x)   // ... and the reduction of local_model.bn_node_x's backward in the same pass (one launch less)
      GPS_TRY(bn_bwd_apply_chain(P.g_s, d, P.xloc, d, N, d, v, sums(BN_L), P.g_xloc, d, a->norm1_local.grad_weight,
                                 a->norm1_local.grad_bias, g_grads_accumulate, P.gl1_p, P.xt, d,
                                 bview(BN_X, a->bn_node_x), act, drop(GPS_SITE_GCN_X), sums(BN_X), st));
    else
      GPS_TRY(bn_bwd_apply(P.g_s, d, P.xloc, d, N, d, v, -1, nodrop, sums(BN_L), P.g_xloc, d,
                           a->norm1_local.grad_weight, a->norm1_local.grad_bias, st, g_grads_accumulate, P.gl1_p));
  }
  if (!P.attn && !P.perf) {   // no global model: the early group ends with norm1_local's gradients (stream st)
    GPS_TRY(wfork(st));
    GPS_TRY(early_done());
  }
  if (two_branches && sd) GPS_TRY(sd->order(st, sa));   // attention-branch backward runs next to the local-model backward
  if (P.attn) {
    BnView v = bview(BN_A, a->norm1_attn);
    if (!fused_la) GPS_TRY(bn_bwd_reduce(P.g_s, d, P.hA, d, N, d, v, -1, nodrop, sums(BN_A), sa));
    GPS_TRY(bn_bwd_apply(P.g_s, d, P.hA, d, N, d, v, -1, nodrop, sums(BN_A), P.g_hA, d, a->norm1_attn.grad_weight,
                         a->norm1_attn.grad_bias, sa, g_grads_accumulate, P.ghA_p));
    // hA = x + drop(O Wo^T + bo)
    const float* g_ao = P.g_hA;
    Planes g_ao_p = P.ghA_p;
    if (pd > 0.f) {
      GPS_TRY(dropmul(P.g_hA, P.g_tmp2, N, d, P, a, GPS_SITE_ATTN_OUT, sa, 0.f, 0, P.gtmp2_p));
      g_ao = P.g_tmp2;
      g_ao_p = P.gtmp2_p;
    }
    GemmParams g;  // g_O = g_ao Wo
    g.M = (int)N; g.N = (int)d; g.K = (int)d;
    g.A = g_ao; g.lda = (int)d; g.B = a->attn_out.weight; g.ldb = (int)d; g.tb = 1; g.C = P.g_O; g.ldc = (int)d;
    g.precision = prec;
    set_bpt(g, P.pt_out, d, d);
    g.Ap = g_ao_p; g.Bp = P.out_p;
    GPS_TRY(gemm(g, sa));
    GPS_TRY(wfork(sa));
    GPS_TRY(linear_wgrad(g_ao, d, P.O, d, N, d, d, a->attn_out.grad_weight, a->attn_out.grad_bias, prec, s2, g_ao_p, P.O_p));
    GPS_TRY(early_done());
    const float* Q = P.Y1 + P.qkv_off;
    float* gQ = P.gY1 + P.qkv_off;
    GPS_TRY(attention_bwd(a->graph, P.H, P.hd, Q, Q + d, Q + 2 * d, P.Wy, P.O, P.g_O, d, P.lse, P.delta, gQ, gQ + d,
                          gQ + 2 * d, P.Wy, pa, a->seed, a->offset, sa, (const unsigned long long*)a->offset_dev,
                          P.gY1_p.cols(P.qkv_off), P.gY1_p.cols(P.qkv_off + d), P.gY1_p.cols(P.qkv_off + 2 * d)));
  }

  if (P.perf) {
    const int64_t inner = P.inner, NH = N * P.H, dh = a->perf_dim_head;
    BnView v = bview(BN_A, a->norm1_attn);
    if (!fused_la) GPS_TRY(bn_bwd_reduce(P.g_s, d, P.hA, d, N, d, v, -1, nodrop, sums(BN_A), sa));
    GPS_TRY(bn_bwd_apply(P.g_s, d, P.hA, d, N, d, v, -1, nodrop, sums(BN_A), P.g_hA, d, a->norm1_attn.grad_weight,
                         a->norm1_attn.grad_bias, sa, g_grads_accumulate));
    const float* g_ao = P.g_hA;   // hA = x + drop_pd(drop_pa(to_out(O)))
    if (pd > 0.f || pa > 0.f) {
      GPS_TRY(dropmul(P.g_hA, P.g_tmp2, N, d, P, a, GPS_SITE_ATTN_OUT, sa, pa, GPS_SITE_PERF_OUT));
      g_ao = P.g_tmp2;
    }
    GemmParams g;  // g_O = g_ao Wout   [N, inner]
    g.M = (int)N; g.N = (int)inner; g.K = (int)d;
    g.A = g_ao; g.lda = (int)d; g.B = a->attn_out.weight; g.ldb = (int)inner; g.tb = 1; g.C = P.g_O; g.ldc = (int)inner;
    g.precision = prec;
    set_bpt(g, P.pt_out, inner, d);
    GPS_TRY(gemm(g, sa));
    GPS_TRY(wfork(sa));
    GPS_TRY(linear_wgrad(g_ao, d, P.O, inner, N, d, inner, a->attn_out.grad_weight, a->attn_out.grad_bias, prec, s2));
    GPS_TRY(early_done());
    // linear attention and feature maps (performer_layer.py:200-205, 119-144)
    if (P.perf_pairwise)
      GPS_TRY(perf_quad_bwd(a->graph, P.H, P.m, P.pnmax, P.pfq, P.pfk, P.pV, P.pgmax, P.O, P.pden, P.g_O, P.g_pden,
                            P.g_pfq, P.g_pfk, P.g_pV, P.g_pgmax, sa));
    else
      GPS_TRY(perf_linattn_bwd(a->graph, P.H, P.m, P.pnmax, P.pfq, P.pfk, P.pV, P.pgmax, P.g_O, P.g_pfq, P.g_pfk, P.g_pV,
                               P.g_pgmax, sa));
    GPS_TRY(perf_features_bwd(P.g_pfq, P.g_pfk, P.pfq, P.pfk, P.pQ, P.pK, P.g_pQ, P.g_pK, a->graph, P.H, P.m, P.pargq,
                              P.pargk, P.g_pgmax, sa));
    float* gdd[2] = {P.g_pfq, P.g_pfk};
    float* gqk[2] = {P.g_pQ, P.g_pK};
    for (int i = 0; i < 2; ++i) {   // g_q += g_dd Pn   (dd = q Pn^T)
      GemmParams h;
      h.M = (int)NH; h.N = (int)dh; h.K = (int)P.mp;
      h.A = gdd[i]; h.lda = (int)P.mp; h.B = P.pPn; h.ldb = (int)dh; h.tb = 1; h.C = gqk[i]; h.ldc = (int)dh;
      h.R1 = gqk[i]; h.ldr1 = (int)dh; h.precision = prec;
      GPS_TRY(gemm(h, sa));
    }
    // projections: dW = g^T x ;  g_xp = g_hA + gQ Wq + gK Wk + gV Wv
    const GpsLinear* lin[3] = {&a->perf_q, &a->perf_k, &a->perf_v};
    const float* gsrc[3] = {P.g_pQ, P.g_pK, P.g_pV};
    GPS_TRY(wfork(sa));
    for (int i = 0; i < 3; ++i) {
      GPS_TRY(linear_wgrad(gsrc[i], inner, a->x, d, N, inner, d, lin[i]->grad_weight, nullptr, prec, s2));
      GemmParams h;
      h.M = (int)N; h.N = (int)d; h.K = (int)inner;
      h.A = gsrc[i]; h.lda = (int)inner; h.B = lin[i]->weight; h.ldb = (int)d; h.tb = 1; h.C = P.g_xp; h.ldc = (int)d;
      h.R1 = i == 0 ? P.g_hA : P.g_xp; h.ldr1 = (int)d; h.precision = prec;
      GPS_TRY(gemm(h, sa));
    }
  }

  // ---- local model backward
  const float* g_x_local = nullptr;  // direct gradient paths into x besides the projections
  if (P.gated) {
    // x_loc = x + drop(act(BN_x(x~))): g_x~ -> gY1[:, 0:d]  (gatedgcn_layer.py:72-83)
    BnView vx = bview(BN_X, a->bn_node_x);
    if (!chain_x) GPS_TRY(bn_bwd_reduce(P.g_xloc, d, P.xt, d, N, d, vx, act, drop(GPS_SITE_GCN_X), sums(BN_X), st));
    GPS_TRY(bn_bwd_apply(P.g_xloc, d, P.xt, d, N, d, vx, act, drop(GPS_SITE_GCN_X), sums(BN_X), P.gY1, P.Wy,
                         a->bn_node_x.grad_weight, a->bn_node_x.grad_bias, st, g_grads_accumulate, P.gY1_p));
    if (!early_edge) GPS_TRY(edge_bn_bwd());
    if (se != st) GPS_TRY(sd->order(se, st));
    // message/aggregate backward (SURVEY Appendix C)
    GPS_TRY(gatedgcn_bwd_dst(a->graph, d, P.gY1, P.Wy, P.ehat, P.Y1 + d, P.Wy, P.g_e, P.g_num, P.gY1 + 2 * d, st, P.ge_p,
                             P.gY1_p.cols(2 * d), P.es ? P.es_g : nullptr, P.es_ggate));
    GPS_TRY(gatedgcn_bwd_src(a->graph, d, P.g_e, P.ehat, P.g_num, P.gY1 + 3 * d, P.gY1 + d, P.Wy, st, P.gY1_p.cols(3 * d),
                             P.gY1_p.cols(d), P.es ? P.es_g : nullptr));
    // C: dC = g_e^T e ; g_edge_attr = grad_edge_out + g_e C
    GPS_TRY(wfork(st));
    GPS_TRY(linear_wgrad(P.g_e, d, a->edge_attr, d, E, d, d, a->gcn_C.grad_weight, a->gcn_C.grad_bias, prec, s2, P.ge_p, P.e_p));
    if (P.es) {   // EquivStableLapPE gate: mlp_r_ij gradients (MID group, final before ev_grads_mid) and d loss / d PE
      GPS_TRY(es_gate_bwd(E, d, act, es_mlp(a), P.es_r, P.es_g, P.es_ggate, P.es_nw, P.es_gr, P.es_work, P.es_work_bytes,
                          g_grads_accumulate, s2));
      if (a->grad_pe) GPS_TRY(es_pe_bwd(a->graph, a->pe, a->pe_dim, P.es_gr, a->grad_pe, s2));
    }
    GPS_TRY(mid_done());
    if (a->grad_edge_attr && E > 0) {
      GemmParams g;
      g.M = (int)E; g.N = (int)d; g.K = (int)d;
      g.A = P.g_e; g.lda = (int)d; g.B = a->gcn_C.weight; g.ldb = (int)d; g.tb = 1; g.C = a->grad_edge_attr; g.ldc = (int)d;
      g.R1 = a->grad_edge_out; g.ldr1 = (int)d; g.precision = prec;
      set_bpt(g, P.pt_C, d, d);
      g.Ap = P.ge_p; g.Bp = P.C_p;
      GPS_TRY(gemm(g, st));
    }
    if (split_tail) {
      const int64_t wl = P.qkv_off;
      GPS_TRY(wcat_wgrad(0, wl));
      GemmParams g;   // g_x = g_xloc + gY1[:, :wl] Wcat[:wl]
      g.M = (int)N; g.N = (int)d; g.K = (int)wl;
      g.A = P.gY1; g.lda = (int)P.Wy; g.B = P.Wcat; g.ldb = (int)d; g.tb = 1; g.C = a->grad_x; g.ldc = (int)d;
      g.R1 = P.g_xloc; g.ldr1 = (int)d; g.precision = prec;
      set_bpt(g, P.pt_cat, d, P.Wy);
      g.Ap = P.gY1_p; g.Bp = P.Wcat_p;
      GPS_TRY(gemm(g, st));
    }
    g_x_local = P.g_xloc;  // residual x_in + ...
  } else if (P.gine) {
    // x_loc = x + drop(h1 W1^T + b1)
    const float* g_l1 = P.g_xloc;
    Planes g_l1_p = P.gl1_p;
    if (pd > 0.f) {
      GPS_TRY(dropmul(P.g_xloc, P.g_tmp3, N, d, P, a, GPS_SITE_LOCAL, st, 0.f, 0, P.gtmp3_p));
      g_l1 = P.g_tmp3;
      g_l1_p = P.gtmp3_p;
    }
    GemmParams g;  // g_h1 = (g_l1 W1) * act'(pre)
    g.M = (int)N; g.N = (int)d; g.K = (int)d;
    g.A = g_l1; g.lda = (int)d; g.B = a->gine_lin1.weight; g.ldb = (int)d; g.tb = 1; g.C = P.g_h1; g.ldc = (int)d;
    if (relu) { g.mask_src = P.h1; g.mask_is_post = 1; } else { g.mask_src = P.h1_pre; g.mask_act = act; }
    g.ldmask = (int)d; g.precision = prec;
    set_bpt(g, P.pt_g1, d, d);
    g.Ap = g_l1_p; g.Bp = P.g1_p; g.Cp = P.gh1_p;
    GPS_TRY(gemm(g, st));
    GPS_TRY(wfork(st));
    GPS_TRY(linear_wgrad(g_l1, d, P.h1, d, N, d, d, a->gine_lin1.grad_weight, a->gine_lin1.grad_bias, prec, s2, g_l1_p, P.h1_p));
    GPS_TRY(linear_wgrad(P.g_h1, d, P.agg, d, N, d, d, a->gine_lin0.grad_weight, a->gine_lin0.grad_bias, prec, s2, P.gh1_p, P.agg_p));
    GPS_TRY(mid_done());
    GemmParams g2;  // g_agg = g_h1 W0
    g2.M = (int)N; g2.N = (int)d; g2.K = (int)d;
    g2.A = P.g_h1; g2.lda = (int)d; g2.B = a->gine_lin0.weight; g2.ldb = (int)d; g2.tb = 1; g2.C = P.g_agg; g2.ldc = (int)d;
    g2.precision = prec;
    set_bpt(g2, P.pt_g0, d, d);
    g2.Ap = P.gh1_p; g2.Bp = P.g0_p;
    GPS_TRY(gemm(g2, st));
    GPS_REQUIRE(a->grad_edge_attr || E == 0, GPS_ERR_ARG, "grad_edge_attr is required for GINE");
    GPS_TRY(gine_bwd_dst(a->graph, d, a->x, a->edge_attr, P.g_agg, a->grad_edge_attr, st));
    GPS_TRY(gine_bwd_src(a->graph, d, a->grad_edge_attr, P.g_agg, a->gine_eps, P.g_xloc, P.g_xl, st));
    g_x_local = P.g_xl;
  } else if (P.gcn) {
    // x_loc = x + drop(b + A_hat Y): g_h = drop * g_xloc; g_b = colsum(g_h); gY = A_hat^T g_h -> gY1[:, 0:d]
    const float* g_h = P.g_xloc;
    if (pd > 0.f) {
      GPS_TRY(dropmul(P.g_xloc, P.g_tmp3, N, d, P, a, GPS_SITE_LOCAL, st));
      g_h = P.g_tmp3;
    }
    if (a->gcn_conv.grad_bias) {
      if (!g_grads_prezeroed) GPS_CUDA(cudaMemsetAsync(a->gcn_conv.grad_bias, 0, (size_t)d * sizeof(float), st));
      GPS_TRY(colsum(g_h, d, N, d, a->gcn_conv.grad_bias, st));
    }
    GPS_TRY(gcn_bwd(a->graph, d, g_h, P.dinv, P.gY1, P.Wy, st, P.gY1_p));
    GPS_TRY(wfork(st));
    GPS_TRY(mid_done());
    g_x_local = P.g_xloc;
  }

  if (two_branches && sd) GPS_TRY(sd->order(sa, st));

  // ---- g_x = [local paths] + [attention residual] + gY1 Wcat ;  d{A,B,D,E,in_proj}
  if (P.Wy && split_tail) {
    const int64_t wl = P.qkv_off, wg = P.Wy - P.qkv_off;
    GPS_TRY(wfork(st));
    GPS_TRY(wcat_wgrad(wl, wg));
    GPS_TRY(unpack_rows(0, P.Wy));
    GemmParams g;   // g_x += g_hA + gY1[:, wl:] Wcat[wl:]  (accumulated onto the first share)
    g.M = (int)N; g.N = (int)d; g.K = (int)wg;
    g.A = P.gY1 + wl; g.lda = (int)P.Wy; g.B = P.Wcat + wl * d; g.ldb = (int)d; g.tb = 1; g.C = a->grad_x; g.ldc = (int)d;
    g.R1 = P.g_hA; g.ldr1 = (int)d; g.precision = prec;
    g.splitk = 2;
    if (wl % 64 == 0) {
      set_bpt(g, P.pt_cat, d, P.Wy);
      g.bpk_kb0 = (int)(wl / 64);
    }
    g.Ap = P.gY1_p.cols(wl); g.Bp = P.Wcat_p.rows(wl);
    GPS_TRY(gemm(g, st));
  } else if (P.Wy) {
    GPS_TRY(wfork(st));
    if (wgrad_split) {
      GPS_TRY(wcat_wgrad(P.qkv_off, P.Wy - P.qkv_off));
      GPS_TRY(unpack_rows(P.qkv_off, P.Wy - P.qkv_off));
    } else {
      GemmParams w;
      w.M = (int)P.Wy; w.N = (int)d; w.K = (int)N;
      w.A = P.gY1; w.lda = (int)P.Wy; w.ta = 1; w.B = a->x; w.ldb = (int)d; w.tb = 1; w.C = P.gWcat; w.ldc = (int)d;
      w.splitk = splitk_for(N, P.Wy, d) < 2 ? 2 : splitk_for(N, P.Wy, d);
      w.colsum_a = P.gbcat; w.precision = prec;
      w.Ap = P.gY1_p; w.Bp = P.x_p;
      if (prec == GPS_PREC_BF16 && w.Ap.hi && N > 0) {   // exact bias gradients in bf16 mode (see linear_wgrad)
        w.colsum_a = nullptr;
        GPS_TRY(colsum(P.gY1, P.Wy, N, P.Wy, P.gbcat, s2));
      }
      if (N > 0) GPS_TRY(gemm(w, s2));
      GPS_TRY(unpack_rows(0, P.Wy));
    }
    GemmParams g;
    g.M = (int)N; g.N = (int)d; g.K = (int)P.Wy;
    g.A = P.gY1; g.lda = (int)P.Wy; g.B = P.Wcat; g.ldb = (int)d; g.tb = 1; g.C = a->grad_x; g.ldc = (int)d;
    g.R1 = g_x_local; g.ldr1 = (int)d;
    g.R2 = P.attn ? P.g_hA : (P.perf ? P.g_xp : nullptr); g.ldr2 = (int)d;
    g.precision = prec;
    if (gx_splitk) g.splitk = 4;   // long reduction, few output tiles: split-K fills the machine (grad_x zeroed above)
    set_bpt(g, P.pt_cat, d, P.Wy);
    g.Ap = P.gY1_p; g.Bp = P.Wcat_p;
    GPS_TRY(gemm(g, st));
  } else if (g_x_local) {
    GPS_TRY(add3(g_x_local, d, P.perf ? P.g_xp : nullptr, d, nullptr, 0, a->grad_x, d, N, d, st));
  } else {
    GPS_TRY(add3(P.g_xp, d, nullptr, 0, nullptr, 0, a->grad_x, d, N, d, st));   // Performer only
  }
  if (sd) GPS_TRY(sd->join(st));
  GPS_TRY(record_ev(a->ev_grads_done, st));
  return GPS_OK;
}

// ---- dropout-only pass: reuse the BN-apply skeleton with an identity BatchNorm is overkill; a
// dedicated tiny kernel keeps it explicit.
namespace {
__global__ void k_dropmul(const float* __restrict__ src, float* __restrict__ dst, int64_t n4, int64_t c4n, float p,
                          uint64_t seed, uint64_t offset, int site, const unsigned long long* offset_dev, float p2,
                          int site2, Planes dstp) {
  if (offset_dev) offset += *offset_dev;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n4; i += (int64_t)gridDim.x * blockDim.x) {
    float4 v = ld4(src + i * 4);
    if (p > 0.f) v = f4mul(v, dropout_scale4(p, seed, offset, site, (uint64_t)i));
    if (p2 > 0.f) v = f4mul(v, dropout_scale4(p2, seed, offset, site2, (uint64_t)i));
    st4(dst + i * 4, v);
    if (dstp.hi) planes_store4(dstp, i / c4n, (i % c4n) * 4, v);
  }
}
__global__ void k_dropmask(float* __restrict__ dst, int64_t n4, float p, uint64_t seed, uint64_t offset, int site) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n4; i += (int64_t)gridDim.x * blockDim.x) {
    float4 s = dropout_scale4(p, seed, offset, site, (uint64_t)i);
    st4(dst + i * 4, make_float4(s.x > 0.f ? 1.f : 0.f, s.y > 0.f ? 1.f : 0.f, s.z > 0.f ? 1.f : 0.f,
                                 s.w > 0.f ? 1.f : 0.f));
  }
}
}  // namespace

static int dropmul(const float* src, float* dst, int64_t rows, int64_t d, const Plan&, const GpsLayerArgs* a, int site,
                   cudaStream_t st, float p2, int site2, Planes dstp) {
  int64_t n4 = rows * d / 4;
  if (n4 == 0) return GPS_OK;
  k_dropmul<<<(unsigned)std::min<int64_t>(ceil_div(n4, 256), kNumSMs * 8), 256, 0, st>>>(src, dst, n4, d / 4, a->dropout,
                                                                                        a->seed, a->offset, site,
                                                                                        (const unsigned long long*)a->offset_dev,
                                                                                        p2, site2, dstp);
  GPS_LAUNCH_CHECK();
  return GPS_OK;
}

}  // namespace gps

// =================================================================================== C ABI
using namespace gps;

extern "C" const char* gps_last_error(void) { return g_err; }
extern "C" int gps_abi_version(void) { return GPS_ABI_VERSION; }
extern "C" const char* gps_build_arch(void) { return "sm_100a"; }
extern "C" unsigned long long gps_launch_count(void) { return g_launches.load(); }
extern "C" unsigned long long gps_fallback_count(void) { return g_fallbacks.load(); }

extern "C" int gps_to_planes(const float* src, int64_t ld, int64_t rows, int64_t cols, void* hi, void* lo, int64_t ldp,
                             void* stream) {
  GPS_REQUIRE(src && hi, GPS_ERR_ARG, "gps_to_planes: null argument");
  ToPlanesItem it{src, ld, (int)rows, (int)cols, Planes{(__nv_bfloat16*)hi, (__nv_bfloat16*)lo, ldp}};
  return to_planes(&it, 1, (cudaStream_t)stream);
}

extern "C" int gps_gemm_planes(const void* A_hi, const void* A_lo, int64_t lda, int32_t ta, const void* B_hi,
                               const void* B_lo, int64_t ldb, int32_t tb, float* C, int64_t ldc, void* C_hi, void* C_lo,
                               int64_t ldcp, int64_t M, int64_t N, int64_t K, int32_t splitk, int32_t precision,
                               float* colsum_a, void* stream) {
  GemmParams g;
  g.M = (int)M; g.N = (int)N; g.K = (int)K;
  g.ta = ta; g.tb = tb; g.C = C; g.ldc = (int)ldc;
  g.Ap = Planes{(__nv_bfloat16*)A_hi, (__nv_bfloat16*)A_lo, lda};
  g.Bp = Planes{(__nv_bfloat16*)B_hi, (__nv_bfloat16*)B_lo, ldb};
  g.Cp = Planes{(__nv_bfloat16*)C_hi, (__nv_bfloat16*)C_lo, ldcp};
  g.splitk = splitk < 1 ? 1 : splitk; g.precision = precision; g.colsum_a = colsum_a;
  int rc = gemm_tma(g, (cudaStream_t)stream);
  if (rc == GPS_ERR_UNSUPPORTED) set_error("gps_gemm_planes: the TMA kernel does not take this shape/alignment");
  return rc;
}
extern "C" void gps_debug_set(int v) { gemm_tc_set_debug(v); }
// bring-up hooks of the TMA GEMM: forced tile width (0 = heuristic) and a device buffer of 256 x 16 uint64 phase stamps
extern "C" void gps_debug_tma(int force_bn, void* trace) {
  gemm_tma_set_force_bn(force_bn);
  gemm_tma_set_trace((unsigned long long*)trace);
}
extern "C" void gps_debug_attn(void* buf) { attention_tc_set_debug((float*)buf); }

extern "C" int gps_layer_plan(const GpsLayerArgs* args, GpsLayerPlan* plan) {
  GPS_REQUIRE(args && plan, GPS_ERR_ARG, "gps_layer_plan: null argument");
  Plan P;
  GPS_TRY(make_plan(args, &P, false));
  plan->saved_bytes = P.saved_bytes;
  plan->fwd_workspace_bytes = P.fwd_bytes;
  plan->bwd_workspace_bytes = P.bwd_bytes;
  plan->fwd_launches = 0;
  plan->bwd_launches = 0;
  plan->wplanes_bytes = P.wplanes_bytes;
  return GPS_OK;
}

extern "C" int gps_layer_forward(const GpsLayerArgs* args, void* stream) {
  GPS_REQUIRE(args, GPS_ERR_ARG, "gps_layer_forward: null args");
  return layer_forward(args, (cudaStream_t)stream);
}

extern "C" int gps_layer_backward(const GpsLayerArgs* args, void* stream) {
  GPS_REQUIRE(args, GPS_ERR_ARG, "gps_layer_backward: null args");
  return layer_backward(args, (cudaStream_t)stream);
}

extern "C" int gps_linear_forward(const float* A, int64_t lda, const float* W, int64_t ldw, const float* bias,
                                  float* C, int64_t ldc, int64_t M, int64_t N, int64_t K, int32_t act,
                                  int32_t precision, void* stream) {
  GemmParams g;
  g.M = (int)M; g.N = (int)N; g.K = (int)K;
  g.A = A; g.lda = (int)lda; g.B = W; g.ldb = (int)ldw; g.C = C; g.ldc = (int)ldc; g.bias = bias; g.act = act;
  g.precision = precision;
  return gemm(g, (cudaStream_t)stream);
}

extern "C" int gps_gemm(const float* A, int64_t lda, int32_t ta, const float* B, int64_t ldb, int32_t tb, float* C,
                        int64_t ldc, int64_t M, int64_t N, int64_t K, int32_t splitk, int32_t precision, int32_t impl,
                        void* stream) {
  GemmParams g;
  g.M = (int)M; g.N = (int)N; g.K = (int)K;
  g.A = A; g.lda = (int)lda; g.ta = ta; g.B = B; g.ldb = (int)ldb; g.tb = tb; g.C = C; g.ldc = (int)ldc;
  g.splitk = splitk < 1 ? 1 : splitk; g.precision = precision;
  if (impl == 1) return gemm_simt(g, (cudaStream_t)stream);
  if (impl == 2) {
    int rc = gemm_tc(g, (cudaStream_t)stream);
    if (rc == GPS_ERR_UNSUPPORTED) set_error("gps_gemm: the tcgen05 kernel does not take this shape/alignment");
    return rc;
  }
  return gemm(g, (cudaStream_t)stream);
}

extern "C" int gps_gatedgcn_aggregate_forward(const GpsGraph* g, int64_t d, const float* Ax, const float* Bx,
                                              const float* Dx, const float* Ex, int64_t ldy, float* Ce, float* xt,
                                              double* stats_x, double* stats_e, void* stream) {
  GPS_REQUIRE(g && Ax && Bx && Dx && Ex && (Ce || g->E == 0) && xt, GPS_ERR_ARG, "gatedgcn_aggregate: null argument");
  return gatedgcn_fwd(*g, d, Ax, Bx, Dx, Ex, ldy, Ce, xt, stats_x, stats_e, (cudaStream_t)stream);
}

extern "C" int gps_es_gate_forward(const GpsGraph* g, const float* pe, int64_t pe_dim, int64_t d, int32_t act,
                                   const float* w0, const float* b0, const float* w2, const float* b2, float* r, float* gate,
                                   void* stream) {
  GPS_REQUIRE(g && (act == GPS_ACT_RELU || act == GPS_ACT_GELU), GPS_ERR_ARG, "es_gate_forward: bad argument");
  EsMlp m{w0, b0, w2, b2, nullptr, nullptr, nullptr, nullptr};
  return es_gate_fwd(*g, pe, pe_dim, d, act, m, r, gate, (cudaStream_t)stream);
}

extern "C" int gps_gatedgcn_es_aggregate_forward(const GpsGraph* g, int64_t d, const float* Ax, const float* Bx,
                                                 const float* Dx, const float* Ex, int64_t ldy, float* Ce, float* xt,
                                                 double* stats_x, double* stats_e, const float* gate, void* stream) {
  GPS_REQUIRE(g && Ax && Bx && Dx && Ex && (Ce || g->E == 0) && xt && (gate || g->E == 0), GPS_ERR_ARG,
              "gatedgcn_es_aggregate: null argument");
  return gatedgcn_fwd(*g, d, Ax, Bx, Dx, Ex, ldy, Ce, xt, stats_x, stats_e, (cudaStream_t)stream, gate);
}

extern "C" int64_t gps_es_gate_backward_workspace_bytes(int64_t E, int64_t d) { return es_gate_bwd_bytes(E, d); }

extern "C" int gps_es_gate_backward(int64_t E, int64_t d, int32_t act, const float* w0, const float* b0, const float* w2,
                                    const float* b2, const float* r, const float* gate, const float* g_gate, float* g_r,
                                    float* grad_w0, float* grad_b0, float* grad_w2, float* grad_b2, void* workspace,
                                    int64_t workspace_bytes, void* stream) {
  GPS_REQUIRE(act == GPS_ACT_RELU || act == GPS_ACT_GELU, GPS_ERR_ARG, "es_gate_backward: unknown activation %d", act);
  EsMlp m{w0, b0, w2, b2, grad_w0, grad_b0, grad_w2, grad_b2};
  return es_gate_bwd(E, d, act, m, r, gate, g_gate, 1, g_r, workspace, workspace_bytes, false, (cudaStream_t)stream);
}

extern "C" int gps_es_pe_backward(const GpsGraph* g, const float* pe, int64_t pe_dim, const float* g_r, float* grad_pe,
                                  void* stream) {
  GPS_REQUIRE(g, GPS_ERR_ARG, "es_pe_backward: null graph");
  return es_pe_bwd(*g, pe, pe_dim, g_r, grad_pe, (cudaStream_t)stream);
}

extern "C" int gps_gine_aggregate_forward(const GpsGraph* g, int64_t d, const float* x, const float* e, float eps,
                                          float* out, void* stream) {
  GPS_REQUIRE(g && x && out, GPS_ERR_ARG, "gine_aggregate: null argument");
  return gine_fwd(*g, d, x, e, eps, out, (cudaStream_t)stream);
}

extern "C" int gps_attention_forward(const GpsGraph* g, int64_t heads, int64_t hd, const float* Q, const float* K,
                                     const float* V, int64_t ld, float* O, int64_t ldo, float* lse, float p_drop,
                                     uint64_t seed, uint64_t offset, void* stream) {
  GPS_REQUIRE(g && Q && K && V && O && lse, GPS_ERR_ARG, "attention_forward: null argument");
  return attention_fwd(*g, heads, hd, Q, K, V, ld, O, ldo, lse, p_drop, seed, offset, (cudaStream_t)stream);
}

extern "C" int gps_attention_forward_tc(const GpsGraph* g, int64_t heads, int64_t hd, const void* qkv_hi, const void* qkv_lo,
                                        int64_t ld, float* O, int64_t ldo, float* lse, float p_drop, uint64_t seed,
                                        uint64_t offset, int32_t precision, void* stream) {
  GPS_REQUIRE(g && qkv_hi && O && lse, GPS_ERR_ARG, "attention_forward_tc: null argument");
  Planes q{(__nv_bfloat16*)qkv_hi, (__nv_bfloat16*)qkv_lo, ld};
  return attention_tc_fwd(*g, heads, hd, q, O, ldo, Planes(), lse, p_drop, seed, offset, nullptr, precision,
                          (cudaStream_t)stream);
}

extern "C" int gps_attention_backward(const GpsGraph* g, int64_t heads, int64_t hd, const float* Q, const float* K,
                                      const float* V, int64_t ld, const float* O, const float* dO, int64_t ldo,
                                      const float* lse, float* delta, float* dQ, float* dK, float* dV, int64_t ldg,
                                      float p_drop, uint64_t seed, uint64_t offset, void* stream) {
  GPS_REQUIRE(g && Q && K && V && O && dO && lse && delta && dQ && dK && dV, GPS_ERR_ARG,
              "attention_backward: null argument");
  return attention_bwd(*g, heads, hd, Q, K, V, ld, O, dO, ldo, lse, delta, dQ, dK, dV, ldg, p_drop, seed, offset,
                       (cudaStream_t)stream);
}

extern "C" int gps_dropout_mask(float* mask, int64_t rows, int64_t cols, float p, uint64_t seed, uint64_t offset,
                                int32_t site, void* stream) {
  GPS_REQUIRE(mask && cols % 4 == 0, GPS_ERR_ARG, "dropout_mask: cols must be a multiple of 4");
  int64_t n4 = rows * cols / 4;
  if (n4 == 0) return GPS_OK;
  k_dropmask<<<(unsigned)std::min<int64_t>(ceil_div(n4, 256), kNumSMs * 8), 256, 0, (cudaStream_t)stream>>>(
      mask, n4, p, seed, offset, site);
  GPS_LAUNCH_CHECK();
  return GPS_OK;
}
