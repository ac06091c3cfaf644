// kernels.cuh — internal launch API of the non-GEMM stages (implemented in elementwise.cu,
// scatter.cu, attention.cu).  All functions enqueue on `stream` and return GPS_* codes.
#pragma once
#include "common.cuh"

namespace gps {

// Per-column BatchNorm view used by consumers: y = gamma * (z - mean) * invstd + beta
// mode 0: mean/invstd arrays are final (backward, or after an explicit bn_finalize)
// mode 1: training forward — the consumer derives mean/invstd from the producer's double column sums itself and
//         its first CTA stores them (for backward) and applies torch.nn.BatchNorm1d's running-stat update, so no
//         separate finalize launch sits between producer and consumer
// mode 2: eval forward — running statistics
struct BnView {
  const float* mean = nullptr;
  const float* invstd = nullptr;
  const float* gamma = nullptr;
  const float* beta = nullptr;
  int mode = 0;
  const double* sums = nullptr;   // [2][d]
  double inv_n = 0.0, unbias = 1.0;
  int64_t d = 0;
  float* save_mean = nullptr;
  float* save_invstd = nullptr;
  float* running_mean = nullptr;
  float* running_var = nullptr;
  long long* nbt = nullptr;
};

struct DropCfg {
  float p = 0.f;
  uint64_t seed = 0, offset = 0;
  int site = 0;
  const unsigned long long* offset_dev = nullptr;  // optional device-resident addend (CUDA-graph replays)
};

// ---- forward row-wise stages ----------------------------------------------------------------
// out = R + dropout(act(BN(z)))  [+ column sums of out into stats]   (gatedgcn_layer.py:72-83)
int bn_act_residual(const float* z, int64_t ldz, const float* R, float* out, int64_t rows, int64_t d,
                    BnView bn, int act, DropCfg drop, double* stats, cudaStream_t stream, Planes outp = Planes());
int bn_act_residual2(const float* zx, const float* Rx, float* outx, int64_t N, BnView bnx, DropCfg dropx, double* statsx,
                     const float* ze, const float* Re, float* oute, int64_t E, BnView bne, DropCfg drope, Planes outep,
                     int64_t d, int act, cudaStream_t stream);
// out = BN_a(a) [+ BN_b(b)]   (gps_layer.py:194,217,222 and :229)
int bn_combine(const float* a, BnView bna, const float* b, BnView bnb, float* out, int64_t rows, int64_t d,
               cudaStream_t stream, Planes outp = Planes());

// ---- backward row-wise stages ---------------------------------------------------------------
// g' = g * [act'(BN(z))] * [dropout scale];  sums[0][c] += sum_r g', sums[1][c] += sum_r g' * zhat
int bn_bwd_reduce(const float* g, int64_t ldg, const float* z, int64_t ldz, int64_t rows, int64_t d, BnView bn,
                  int act /* -1: none */, DropCfg drop, double* sums, cudaStream_t stream);
// out = gamma*invstd*(g' - S1/n - zhat*S2/n) (+ add); also writes grad_gamma = S2, grad_beta = S1
int bn_bwd_apply(const float* g, int64_t ldg, const float* z, int64_t ldz, int64_t rows, int64_t d, BnView bn,
                 int act, DropCfg drop, const double* sums, float* out, int64_t ldo, float* grad_gamma,
                 float* grad_beta, cudaStream_t stream, bool accumulate = false, Planes outp = Planes());
// bn_bwd_apply of one BatchNorm (no activation / dropout in front of it) fused with the bn_bwd_reduce of the NEXT
// BatchNorm down the backward chain, which consumes this one's output: sums2 gets what
// bn_bwd_reduce(out, z2, bn2, act2, drop2) would have produced.
int bn_bwd_apply_chain(const float* g, int64_t ldg, const float* z, int64_t ldz, int64_t rows, int64_t d, BnView bn,
                       const double* sums, float* out, int64_t ldo, float* grad_gamma, float* grad_beta, bool accumulate,
                       Planes outp, const float* z2, int64_t ldz2, BnView bn2, int act2, DropCfg drop2, double* sums2,
                       cudaStream_t stream);
// out = a + b (+ c)   row-wise with independent leading dimensions
int add3(const float* a, int64_t lda, const float* b, int64_t ldb, const float* c, int64_t ldc, float* out,
         int64_t ldo, int64_t rows, int64_t d, cudaStream_t stream);
// out[c] = sum_r a[r, c]  (float atomics into pre-zeroed out)
int colsum(const float* a, int64_t lda, int64_t rows, int64_t d, float* out, cudaStream_t stream);
// dst[r, :] = src[r, :] for a [rows, d] block with leading dimensions
int copy2d(const float* src, int64_t lds, float* dst, int64_t ldd, int64_t rows, int64_t d, cudaStream_t stream);

// ---- sparse (message passing) stages -------------------------------------------------------
// gate != nullptr: EquivStableLapPE-gated aggregation, sigma_ij = sigmoid(e_ij) * gate[eid] (gate from es_gate_fwd)
int gatedgcn_fwd(const GpsGraph& g, int64_t d, const float* Ax, const float* Bx, const float* Dx,
                 const float* Ex, int64_t ldy, float* Ce, float* xt, double* stats_x, double* stats_e,
                 cudaStream_t stream, const float* gate = nullptr);
// dst-ordered backward pass: reads g_xt (ld ldg), ehat, Bx; g_e holds the BN_e-path gradient on entry
// and the total gradient w.r.t. e_ij on exit; writes g_num [N,d] and g_Dx (ld ldg).
// gate != nullptr: the gated pass; it also writes the per-warp shares of d loss / d gate[eid] to
// g_gate [E, gatedgcn_es_nwarps(d)]
int gatedgcn_bwd_dst(const GpsGraph& g, int64_t d, const float* g_xt, int64_t ldg, const float* ehat,
                     const float* Bx, int64_t ldy, float* g_e, float* g_num, float* g_Dx,
                     cudaStream_t stream, Planes g_e_p = Planes(), Planes g_Dx_p = Planes(),
                     const float* gate = nullptr, float* g_gate = nullptr);
int gatedgcn_es_nwarps(int64_t d);
// src-ordered backward pass: g_Ex_j = sum g_e_k, g_Bx_j = sum g_num[dst(k)] * sigmoid(ehat_k) [* gate_k]
int gatedgcn_bwd_src(const GpsGraph& g, int64_t d, const float* g_e, const float* ehat, const float* g_num,
                     float* g_Ex, float* g_Bx, int64_t ldg, cudaStream_t stream, Planes g_Ex_p = Planes(),
                     Planes g_Bx_p = Planes(), const float* gate = nullptr);

// ---- EquivStableLapPE edge gate (eslappe.cu; gatedgcn_layer.py:29-35, 99-103)
// r_e = sum_c (PE_dst - PE_src)_c^2 ;  gate_e = sigmoid(W2 act(W1 r_e + b1) + b2)   (W1 [d,1], W2 [1,d])
struct EsMlp {
  const float *w1, *b1, *w2, *b2;
  float *gw1, *gb1, *gw2, *gb2;
};
int es_gate_fwd(const GpsGraph& g, const float* pe, int64_t k, int64_t d, int act, const EsMlp& m, float* r, float* gate,
                cudaStream_t stream);
// workspace of es_gate_bwd: per-block partial sums of the mlp_r_ij gradients
int64_t es_gate_bwd_bytes(int64_t E, int64_t d);
// g_gate [E, nshare]: shares of d loss / d gate_e (summed in order).  Writes g_r [E] and the four parameter gradients
// (added to the buffers when accumulate), deterministic: per-block partials, then a fixed-order final sum.
int es_gate_bwd(int64_t E, int64_t d, int act, const EsMlp& m, const float* r, const float* gate, const float* g_gate,
                int nshare, float* g_r, void* work, int64_t work_bytes, bool accumulate, cudaStream_t stream);
// grad_pe_n = sum_{e in dst(n)} 2 g_r_e (PE_n - PE_src(e)) + sum_{e in src(n)} 2 g_r_e (PE_n - PE_dst(e))
int es_pe_bwd(const GpsGraph& g, const float* pe, int64_t k, const float* g_r, float* grad_pe, cudaStream_t stream);
int gine_fwd(const GpsGraph& g, int64_t d, const float* x, const float* e, float eps, float* out,
             cudaStream_t stream, Planes outp = Planes());
// g_e[k] = g_o[dst(k)] * [x_src + e_k > 0];  (dst ordered)
int gine_bwd_dst(const GpsGraph& g, int64_t d, const float* x, const float* e, const float* g_o, float* g_e,
                 cudaStream_t stream);
// g_x[j] = (1+eps) g_o[j] + sum_{k: src=j} g_e[k]  (+ add[j])
int gine_bwd_src(const GpsGraph& g, int64_t d, const float* g_e, const float* g_o, float eps, const float* add,
                 float* g_x, cudaStream_t stream);

// GCN (PyG GCNConv): dinv_i = (1 + #non-self in-edges)^-1/2; x_loc = x + drop(b + A_hat Y) [+ column sums of x_loc];
// backward gY = A_hat^T g_h
int gcn_dinv(const GpsGraph& g, float* dinv, cudaStream_t stream);
int gcn_fwd(const GpsGraph& g, int64_t d, const float* Y, int64_t ldy, const float* dinv, const float* bias,
            const float* x, float* xloc, DropCfg drop, double* stats, cudaStream_t stream);
int gcn_bwd(const GpsGraph& g, int64_t d, const float* g_h, const float* dinv, float* gY, int64_t ldg,
            cudaStream_t stream, Planes gYp = Planes());

// ---- attention ------------------------------------------------------------------------------
int attention_fwd(const GpsGraph& g, int64_t heads, int64_t hd, const float* Q, const float* K, const float* V,
                  int64_t ld, float* O, int64_t ldo, float* lse, float p_drop, uint64_t seed, uint64_t offset,
                  cudaStream_t stream, const unsigned long long* offset_dev = nullptr, Planes Op = Planes());
int attention_bwd(const GpsGraph& g, int64_t heads, int64_t hd, const float* Q, const float* K, const float* V,
                  int64_t ld, const float* O, const float* dO, int64_t ldo, const float* lse, float* delta,
                  float* dQ, float* dK, float* dV, int64_t ldg, float p_drop, uint64_t seed, uint64_t offset,
                  cudaStream_t stream, const unsigned long long* offset_dev = nullptr, Planes dQp = Planes(),
                  Planes dKp = Planes(), Planes dVp = Planes());

// tcgen05 version (attention_tc.cu): Q, K, V from bf16 hi/lo planes in the per-head padded layout
// column (which * H + h) * hd_pad + k, hd_pad = attention_tc_hd_pad(hd), pad columns zero
void attention_tc_set_debug(float* buf);   // bring-up: 3 x 128 x 128 floats (S, P, raw O of CTA (0,0))
bool attention_tc_supported(int64_t hd);
int64_t attention_tc_hd_pad(int64_t hd);
int attention_tc_fwd(const GpsGraph& g, int64_t heads, int64_t hd, Planes qkv, float* O, int64_t ldo, Planes Op, float* lse,
                     float p_drop, uint64_t seed, uint64_t offset, const unsigned long long* offset_dev, int precision,
                     cudaStream_t stream);

}  // namespace gps
