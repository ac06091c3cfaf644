// eslappe.cu — EquivStableLapPE edge gate of the GatedGCN local model (Wang et al., ICLR 2022, "Equivariant and Stable
// Positional Encoding for More Powerful Graph Neural Networks"), as the reference builds it:
// graphgps/layer/gatedgcn_layer.py:29-35 (mlp_r_ij = Linear(1,d), act, Linear(d,1), Sigmoid) and :99-103
//   r_ij    = sum_c (PE_i,c - PE_j,c)^2            (edge j -> i: src = j, dst = i)
//   gate_ij = sigmoid(W2 act(W1 r_ij + b1) + b2)
//   sigma_ij = sigmoid(e_ij) * gate_ij             (applied inside the aggregation, scatter.cu GATED variants)
// The gate depends on PE and mlp_r_ij only, so the layer computes it on the edge-projection side stream.  Everything
// here is fp32 on the CUDA cores, one warp per edge (forward, gate backward) or per node (PE gradient); every
// reduction runs in a fixed order, so results are bitwise reproducible.
#include <algorithm>

#include "kernels.cuh"

namespace gps {

namespace {

constexpr int kEsWarps = 4;   // warps per CTA of the gate backward (shared-memory partials: 3 d floats per warp)

__device__ __forceinline__ float es_sigmoid(float z) { return 1.f / (1.f + expf(-z)); }

// one warp per destination node, each of its in-edges in turn: r_e (k-wide distance) and gate_e (d-wide MLP)
template <int ACT>
__global__ void k_es_gate_fwd(GpsGraph g, const float* __restrict__ pe, int k, int d, EsMlp m, float* __restrict__ r,
                              float* __restrict__ gate) {
  const int lane = threadIdx.x & 31;
  const int64_t w0 = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5, nw = ((int64_t)gridDim.x * blockDim.x) >> 5;
  const float b2 = m.b2[0];
  for (int64_t i = w0; i < g.N; i += nw) {
    const float* pi = pe + i * k;
    for (int q = g.dst_ptr[i]; q < g.dst_ptr[i + 1]; ++q) {
      const float* pj = pe + (int64_t)g.dst_src[q] * k;
      float acc = 0.f;
      for (int c = lane; c < k; c += 32) {
        const float t = pi[c] - pj[c];
        acc = fmaf(t, t, acc);
      }
      const float rr = warp_sum(acc);
      float z = 0.f;
      for (int h = lane; h < d; h += 32) z = fmaf(m.w2[h], act_fwd<ACT>(fmaf(m.w1[h], rr, m.b1[h])), z);
      z = warp_sum(z) + b2;
      if (lane == 0) {
        const int64_t eid = g.dst_eid[q];
        r[eid] = rr;
        gate[eid] = es_sigmoid(z);
      }
    }
  }
}

// one warp per edge (edge-id order, fixed grid): d loss / d gate -> d loss / d r and the mlp_r_ij gradients.  Lane l owns
// hidden units h = l + 32 t and accumulates their gradients in its warp's shared-memory slice; the CTA sums its warps
// in order and writes one partial row [gW1 | gb1 | gW2 | gb2] per CTA.
template <int ACT>
__global__ void k_es_gate_bwd(int64_t E, int d, EsMlp m, const float* __restrict__ r, const float* __restrict__ gate,
                              const float* __restrict__ g_gate, int nshare, float* __restrict__ g_r,
                              float* __restrict__ part) {
  extern __shared__ float sm[];   // [kEsWarps][3 d + 1]
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const int row = 3 * d + 1;
  float* mine = sm + w * row;
  for (int t = lane; t < row; t += 32) mine[t] = 0.f;
  __syncwarp();
  float gb2 = 0.f;
  for (int64_t e = (int64_t)blockIdx.x * kEsWarps + w; e < E; e += (int64_t)gridDim.x * kEsWarps) {
    float gg = 0.f;
    for (int s = 0; s < nshare; ++s) gg += g_gate[e * nshare + s];
    const float gt = gate[e], rr = r[e];
    const float gz = gg * gt * (1.f - gt);            // through the Sigmoid
    gb2 += gz;
    float gr = 0.f;
    for (int h = lane; h < d; h += 32) {
      const float w1 = m.w1[h];
      const float pre = fmaf(w1, rr, m.b1[h]);
      const float gp = gz * m.w2[h] * act_bwd<ACT>(pre);
      mine[h] = fmaf(gp, rr, mine[h]);                // W1 [d,1]
      mine[d + h] += gp;                              // b1
      mine[2 * d + h] = fmaf(gz, act_fwd<ACT>(pre), mine[2 * d + h]);   // W2 [1,d]
      gr = fmaf(gp, w1, gr);
    }
    gr = warp_sum(gr);
    if (lane == 0) g_r[e] = gr;
  }
  if (lane == 0) mine[3 * d] = gb2;
  __syncthreads();
  for (int t = threadIdx.x; t < row; t += blockDim.x) {
    float s = 0.f;
#pragma unroll
    for (int q = 0; q < kEsWarps; ++q) s += sm[q * row + t];
    part[(int64_t)blockIdx.x * row + t] = s;
  }
}

__global__ void k_es_param_reduce(const float* __restrict__ part, int nblk, int d, EsMlp m, int accumulate) {
  const int row = 3 * d + 1;
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= row) return;
  float s = 0.f;
  for (int b = 0; b < nblk; ++b) s += part[(int64_t)b * row + t];
  float* base = t < d ? m.gw1 : (t < 2 * d ? m.gb1 : (t < 3 * d ? m.gw2 : m.gb2));
  if (!base) return;
  float* dst = base + (t < 3 * d ? t % d : 0);
  *dst = accumulate ? *dst + s : s;
}

// one warp per node, lanes across the k PE channels; in-edges (CSR) then out-edges (CSC), each in edge-id order
__global__ void k_es_pe_bwd(GpsGraph g, const float* __restrict__ pe, int k, const float* __restrict__ g_r,
                            float* __restrict__ grad_pe) {
  const int lane = threadIdx.x & 31;
  const int64_t w0 = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5, nw = ((int64_t)gridDim.x * blockDim.x) >> 5;
  for (int64_t n = w0; n < g.N; n += nw) {
    const int ib = g.dst_ptr[n], ie = g.dst_ptr[n + 1], ob = g.src_ptr[n], oe = g.src_ptr[n + 1];
    for (int c = lane; c < k; c += 32) {
      const float pn = pe[n * k + c];
      float acc = 0.f;
      for (int q = ib; q < ie; ++q) acc = fmaf(2.f * g_r[g.dst_eid[q]], pn - pe[(int64_t)g.dst_src[q] * k + c], acc);
      for (int q = ob; q < oe; ++q) acc = fmaf(2.f * g_r[g.src_eid[q]], pn - pe[(int64_t)g.src_dst[q] * k + c], acc);
      grad_pe[n * k + c] = acc;
    }
  }
}

static int64_t es_blocks(int64_t E) { return std::max<int64_t>(1, std::min<int64_t>(ceil_div(E, kEsWarps), 2 * kNumSMs)); }

}  // namespace

int es_gate_fwd(const GpsGraph& g, const float* pe, int64_t k, int64_t d, int act, const EsMlp& m, float* r, float* gate,
                cudaStream_t stream) {
  GPS_REQUIRE(pe && k > 0 && m.w1 && m.b1 && m.w2 && m.b2 && r && gate, GPS_ERR_ARG, "es_gate_fwd: null argument");
  if (g.N == 0 || g.E == 0) return GPS_OK;
  const unsigned blocks = (unsigned)std::min<int64_t>(ceil_div(g.N, 8), kNumSMs * 16);
  if (act == GPS_ACT_RELU)
    k_es_gate_fwd<GPS_ACT_RELU><<<blocks, 256, 0, stream>>>(g, pe, (int)k, (int)d, m, r, gate);
  else
    k_es_gate_fwd<GPS_ACT_GELU><<<blocks, 256, 0, stream>>>(g, pe, (int)k, (int)d, m, r, gate);
  GPS_LAUNCH_CHECK();
  return GPS_OK;
}

int64_t es_gate_bwd_bytes(int64_t E, int64_t d) { return round_up(es_blocks(E) * (3 * d + 1) * (int64_t)sizeof(float), 256); }

int es_gate_bwd(int64_t E, int64_t d, int act, const EsMlp& m, const float* r, const float* gate, const float* g_gate,
                int nshare, float* g_r, void* work, int64_t work_bytes, bool accumulate, cudaStream_t stream) {
  const size_t smem = (size_t)kEsWarps * (3 * d + 1) * sizeof(float);
  GPS_REQUIRE(smem <= 48 * 1024, GPS_ERR_UNSUPPORTED, "EquivStableLapPE gate backward supports dim_h <= 1023 (got %lld)",
              (long long)d);
  GPS_REQUIRE(m.w1 && m.b1 && m.w2 && work && (E == 0 || (r && gate && g_gate && g_r)), GPS_ERR_ARG,
              "es_gate_bwd: null argument");
  GPS_REQUIRE(work_bytes >= es_gate_bwd_bytes(E, d), GPS_ERR_ARG, "es_gate_bwd: workspace too small (%lld < %lld)",
              (long long)work_bytes, (long long)es_gate_bwd_bytes(E, d));
  const int nblk = (int)es_blocks(E);
  float* part = (float*)work;
  if (act == GPS_ACT_RELU)
    k_es_gate_bwd<GPS_ACT_RELU><<<nblk, kEsWarps * 32, smem, stream>>>(E, (int)d, m, r, gate, g_gate, nshare, g_r, part);
  else
    k_es_gate_bwd<GPS_ACT_GELU><<<nblk, kEsWarps * 32, smem, stream>>>(E, (int)d, m, r, gate, g_gate, nshare, g_r, part);
  GPS_LAUNCH_CHECK();
  k_es_param_reduce<<<(unsigned)ceil_div(3 * d + 1, 128), 128, 0, stream>>>(part, nblk, (int)d, m, accumulate ? 1 : 0);
  GPS_LAUNCH_CHECK();
  return GPS_OK;
}

int es_pe_bwd(const GpsGraph& g, const float* pe, int64_t k, const float* g_r, float* grad_pe, cudaStream_t stream) {
  GPS_REQUIRE(pe && grad_pe && k > 0 && (g.E == 0 || g_r), GPS_ERR_ARG, "es_pe_bwd: null argument");
  if (g.N == 0) return GPS_OK;
  const unsigned blocks = (unsigned)std::min<int64_t>(ceil_div(g.N, 8), kNumSMs * 16);
  k_es_pe_bwd<<<blocks, 256, 0, stream>>>(g, pe, (int)k, g_r, grad_pe);
  GPS_LAUNCH_CHECK();
  return GPS_OK;
}

}  // namespace gps
