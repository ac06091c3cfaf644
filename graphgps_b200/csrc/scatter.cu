// scatter.cu — the sparse (message-passing) half of GPSLayer as CSR/CSC segmented gather-reduce.
//
// GatedGCN message/aggregate/update: graphgps/layer/gatedgcn_layer.py:90-136
//   e_ij = Dx_i + Ex_j + Ce_ij ; sigma = sigmoid(e_ij)
//   x~_i = Ax_i + (sum_j sigma_ij * Bx_j) / (sum_j sigma_ij + 1e-6)
// GINE aggregate (PyG GINEConv; maths per graphgps/layer/gine_conv_layer.py:56-84):
//   out_i = (1+eps) x_i + sum_j relu(x_j + e_ij)
// GCN aggregate (PyG 2.2 GCNConv, gps_layer.py:49-51; gcn_norm with add_remaining_self_loops, unit edge weights):
//   deg_i = 1 + #{j -> i, j != i};  h_i = b + deg_i^-1/2 ( deg_i^-1/2 Y_i + sum_{j -> i, j != i} deg_j^-1/2 Y_j ),  Y = x W^T
// The reference materialises three [E,d] gathers and runs two atomic torch_scatter sums
// (gatedgcn_layer.py:118-123).  Here a thread owns (node, 4 channels): it walks the node's
// dst-sorted (or src-sorted) edge segment with 128-bit loads, reduces serially in registers — no
// atomics on feature data, deterministic order (edge-id order inside a segment) — and the
// BatchNorm column statistics of the two outputs are reduced thread -> CTA -> global doubles.
// Backward maths: SURVEY.md Appendix C.
#include <algorithm>

#include "kernels.cuh"

namespace gps {

namespace {

struct NodeGeom {
  dim3 block, grid;
  size_t smem;
};
static int node_geom(int64_t N, int64_t d, int nstat, NodeGeom* g) {
  GPS_REQUIRE(d > 0 && d % 4 == 0 && d / 4 <= 1024, GPS_ERR_UNSUPPORTED,
              "sparse stage needs d %% 4 == 0 and d <= 4096 (got %lld)", (long long)d);
  int C4 = (int)(d / 4);
  int RY = C4 >= 256 ? 1 : 256 / C4;
  int64_t cap = kNumSMs * 16;
  if (nstat > 0) {   // statistics epilogue: same-address double atomics serialise -> few, fat CTAs (see elementwise.cu)
    RY = C4 >= 1024 ? 1 : 1024 / C4;
    if (RY > 16) RY = 16;
    const int smem_cap = (int)(48 * 1024 / ((size_t)nstat * C4 * sizeof(float4)));   // static 48 KB limit
    if (RY > smem_cap) RY = smem_cap < 1 ? 1 : smem_cap;
    cap = kNumSMs;
  }
  int64_t blocks = ceil_div(N > 0 ? N : 1, (int64_t)RY * 2);
  if (blocks > cap) blocks = cap;
  g->block = dim3(C4, RY, 1);
  g->grid = dim3((unsigned)blocks, 1, 1);
  g->smem = RY > 1 ? (size_t)nstat * RY * C4 * sizeof(float4) : 0;
  return GPS_OK;
}

__device__ __forceinline__ float4 sigmoid4(float4 v) {
  return make_float4(sigmoidf_(v.x), sigmoidf_(v.y), sigmoidf_(v.z), sigmoidf_(v.w));
}

// CTA-level reduction of NS float4 accumulators over threadIdx.y, then double atomics by ry == 0.
template <int NS>
__device__ __forceinline__ void block_stats(float4* acc, double* const* ptrs, float4* sm) {
  const int c4 = threadIdx.x, ry = threadIdx.y, RY = blockDim.y, C4 = blockDim.x;
  if (RY > 1) {
#pragma unroll
    for (int s = 0; s < NS; ++s) sm[(s * RY + ry) * C4 + c4] = acc[s];
    __syncthreads();
    if (ry == 0) {
#pragma unroll
      for (int s = 0; s < NS; ++s)
        for (int y = 1; y < RY; ++y) acc[s] = f4add(acc[s], sm[(s * RY + y) * C4 + c4]);
    }
  }
  if (ry == 0) {
#pragma unroll
    for (int s = 0; s < NS; ++s) {
      double* p = ptrs[s];
      if (!p) continue;
      atomic_add_f64(p + c4 * 4 + 0, (double)acc[s].x);
      atomic_add_f64(p + c4 * 4 + 1, (double)acc[s].y);
      atomic_add_f64(p + c4 * 4 + 2, (double)acc[s].z);
      atomic_add_f64(p + c4 * 4 + 3, (double)acc[s].w);
    }
  }
}

// GATED: EquivStableLapPE edge gate (gatedgcn_layer.py:99-103), sigma_ij = sigmoid(e_ij) * gate[eid], one scalar per
// edge from eslappe.cu; the edge output e_ij stays ungated
template <bool STATS, bool GATED>
__global__ void __launch_bounds__(1024) k_gatedgcn_fwd(GpsGraph g, int d, const float* __restrict__ Ax, const float* __restrict__ Bx,
                               const float* __restrict__ Dx, const float* __restrict__ Ex, int64_t ldy,
                               float* __restrict__ Ce, float* __restrict__ xt, double* stats_x,
                               double* stats_e, const float* __restrict__ gate) {
  extern __shared__ float4 sm[];
  const int c = threadIdx.x * 4, ry = threadIdx.y, RY = blockDim.y;
  float4 acc[4] = {f4zero(), f4zero(), f4zero(), f4zero()};  // sum x~, sum x~^2, sum e, sum e^2
  for (int64_t i = (int64_t)blockIdx.x * RY + ry; i < g.N; i += (int64_t)gridDim.x * RY) {
    const float4 dx = ld4(Dx + i * ldy + c);
    float4 num = f4zero(), den = f4zero();
    const int kb = g.dst_ptr[i], ke = g.dst_ptr[i + 1];
    // two edges per iteration: 6 independent 128-bit gathers in flight per thread (the loop is latency bound).  The
    // gated variant takes one: with the gate scalars the statistics instantiation would exceed 64 registers and spill.
#pragma unroll 1
    for (int k = kb; k < ke; k += GATED ? 1 : 2) {
      const bool two = !GATED && k + 1 < ke;
      const int j0 = g.dst_src[k], j1 = two ? g.dst_src[k + 1] : j0;
      const int64_t e0 = g.dst_eid[k], e1 = two ? g.dst_eid[k + 1] : e0;
      const float4 ex0 = ld4(Ex + (int64_t)j0 * ldy + c), bx0 = ld4(Bx + (int64_t)j0 * ldy + c);
      float4 c0 = ld4(Ce + e0 * d + c);
      const float4 ex1 = ld4(Ex + (int64_t)j1 * ldy + c), bx1 = ld4(Bx + (int64_t)j1 * ldy + c);
      float4 c1 = ld4(Ce + e1 * d + c);
      c0 = f4add(c0, f4add(dx, ex0));
      st4(Ce + e0 * d + c, c0);
      float4 s0 = sigmoid4(c0);
      if (GATED) s0 = f4scale(s0, gate[e0]);
      num = f4fma(s0, bx0, num);
      den = f4add(den, s0);
      if (STATS) {
        acc[2] = f4add(acc[2], c0);
        acc[3] = f4fma(c0, c0, acc[3]);
      }
      if (two) {
        c1 = f4add(c1, f4add(dx, ex1));
        st4(Ce + e1 * d + c, c1);
        float4 s1 = sigmoid4(c1);
        if (GATED) s1 = f4scale(s1, gate[e1]);
        num = f4fma(s1, bx1, num);
        den = f4add(den, s1);
        if (STATS) {
          acc[2] = f4add(acc[2], c1);
          acc[3] = f4fma(c1, c1, acc[3]);
        }
      }
    }
    const float4 ax = ld4(Ax + i * ldy + c);
    float4 v = make_float4(ax.x + num.x / (den.x + 1e-6f), ax.y + num.y / (den.y + 1e-6f),
                           ax.z + num.z / (den.z + 1e-6f), ax.w + num.w / (den.w + 1e-6f));
    st4(xt + i * d + c, v);
    if (STATS) {
      acc[0] = f4add(acc[0], v);
      acc[1] = f4fma(v, v, acc[1]);
    }
  }
  if (STATS) {
    double* ptrs[4] = {stats_x, stats_x ? stats_x + d : nullptr, stats_e, stats_e ? stats_e + d : nullptr};
    block_stats<4>(acc, ptrs, sm);
  }
}

// GATED: sigma = sigmoid(ehat) * gate[eid].  The row of a node is padded to whole warps (blockDim.x = round_up(d/4, 32),
// lanes with c >= d only take part in the shuffles), and each warp writes its share of d loss / d gate[eid] =
// sum_c gs_c sigmoid(ehat)_c to g_gate[eid * nwarps + warp]; es_gate_bwd sums the shares in a fixed order.
template <bool GATED>
__global__ void k_gatedgcn_bwd_dst(GpsGraph g, int d, const float* __restrict__ g_xt, int64_t ldg,
                                   const float* __restrict__ ehat, const float* __restrict__ Bx, int64_t ldy,
                                   float* __restrict__ g_e, float* __restrict__ g_num,
                                   float* __restrict__ g_Dx, Planes g_e_p, Planes g_Dx_p,
                                   const float* __restrict__ gate, float* __restrict__ g_gate) {
  const int c = threadIdx.x * 4, ry = threadIdx.y, RY = blockDim.y;
  const bool on = !GATED || c < d;
  const int nw = GATED ? (int)(blockDim.x >> 5) : 1, wi = GATED ? (int)(threadIdx.x >> 5) : 0;
  for (int64_t i = (int64_t)blockIdx.x * RY + ry; i < g.N; i += (int64_t)gridDim.x * RY) {
    const int kb = g.dst_ptr[i], ke = g.dst_ptr[i + 1];
    float4 num = f4zero(), den = f4zero();
    if (on) {
      for (int k = kb; k < ke; ++k) {
        const int j = g.dst_src[k];
        const int64_t eid = g.dst_eid[k];
        float4 s = sigmoid4(ld4(ehat + eid * d + c));
        if (GATED) s = f4scale(s, gate[eid]);
        num = f4fma(s, ld4(Bx + (int64_t)j * ldy + c), num);
        den = f4add(den, s);
      }
    }
    const float4 inv = make_float4(1.f / (den.x + 1e-6f), 1.f / (den.y + 1e-6f), 1.f / (den.z + 1e-6f),
                                   1.f / (den.w + 1e-6f));
    const float4 agg = f4mul(num, inv);
    const float4 gx = on ? ld4(g_xt + i * ldg + c) : f4zero();
    const float4 gn = f4mul(gx, inv);                       // d/d num
    const float4 gd = make_float4(-gn.x * agg.x, -gn.y * agg.y, -gn.z * agg.z, -gn.w * agg.w);  // d/d den
    if (on) st4(g_num + i * d + c, gn);
    float4 gdx = f4zero();
    for (int k = kb; k < ke; ++k) {
      const int64_t eid = g.dst_eid[k];
      float gsum = 0.f;
      if (on) {
        const int j = g.dst_src[k];
        const float4 s = sigmoid4(ld4(ehat + eid * d + c));
        const float4 bx = ld4(Bx + (int64_t)j * ldy + c);
        float4 gs = f4fma(gn, bx, gd);                      // d/d sigma
        if (GATED) {
          gsum = gs.x * s.x + gs.y * s.y + gs.z * s.z + gs.w * s.w;
          gs = f4scale(gs, gate[eid]);                      // d/d sigmoid(ehat)
        }
        float4 ge = ld4(g_e + eid * d + c);
        ge.x += gs.x * s.x * (1.f - s.x);
        ge.y += gs.y * s.y * (1.f - s.y);
        ge.z += gs.z * s.z * (1.f - s.z);
        ge.w += gs.w * s.w * (1.f - s.w);
        st4(g_e + eid * d + c, ge);
        if (g_e_p.hi) planes_store4(g_e_p, eid, c, ge);
        gdx = f4add(gdx, ge);
      }
      if (GATED) {
        gsum = warp_sum(gsum);
        if ((threadIdx.x & 31) == 0) g_gate[eid * nw + wi] = gsum;
      }
    }
    if (on) {
      st4(g_Dx + i * ldg + c, gdx);
      if (g_Dx_p.hi) planes_store4(g_Dx_p, i, c, gdx);
    }
  }
}

template <bool GATED>
__global__ void k_gatedgcn_bwd_src(GpsGraph g, int d, const float* __restrict__ g_e,
                                   const float* __restrict__ ehat, const float* __restrict__ g_num,
                                   float* __restrict__ g_Ex, float* __restrict__ g_Bx, int64_t ldg, Planes g_Ex_p,
                                   Planes g_Bx_p, const float* __restrict__ gate) {
  const int c = threadIdx.x * 4, ry = threadIdx.y, RY = blockDim.y;
  for (int64_t j = (int64_t)blockIdx.x * RY + ry; j < g.N; j += (int64_t)gridDim.x * RY) {
    float4 gex = f4zero(), gbx = f4zero();
    const int kb = g.src_ptr[j], ke = g.src_ptr[j + 1];
    for (int k = kb; k < ke; ++k) {
      const int i = g.src_dst[k];
      const int64_t eid = g.src_eid[k];
      gex = f4add(gex, ld4(g_e + eid * d + c));
      float4 s = sigmoid4(ld4(ehat + eid * d + c));
      if (GATED) s = f4scale(s, gate[eid]);
      gbx = f4fma(ld4(g_num + (int64_t)i * d + c), s, gbx);
    }
    st4(g_Ex + j * ldg + c, gex);
    st4(g_Bx + j * ldg + c, gbx);
    if (g_Ex_p.hi) planes_store4(g_Ex_p, j, c, gex);
    if (g_Bx_p.hi) planes_store4(g_Bx_p, j, c, gbx);
  }
}

__global__ void k_gine_fwd(GpsGraph g, int d, const float* __restrict__ x, const float* __restrict__ e,
                           float eps, float* __restrict__ out, Planes outp) {
  const int c = threadIdx.x * 4, ry = threadIdx.y, RY = blockDim.y;
  for (int64_t i = (int64_t)blockIdx.x * RY + ry; i < g.N; i += (int64_t)gridDim.x * RY) {
    float4 acc = f4scale(ld4(x + i * d + c), 1.f + eps);
    const int kb = g.dst_ptr[i], ke = g.dst_ptr[i + 1];
    for (int k = kb; k < ke; ++k) {
      const int j = g.dst_src[k];
      const int64_t eid = g.dst_eid[k];
      const float4 m = f4add(ld4(x + (int64_t)j * d + c), ld4(e + eid * d + c));
      acc.x += fmaxf(m.x, 0.f);
      acc.y += fmaxf(m.y, 0.f);
      acc.z += fmaxf(m.z, 0.f);
      acc.w += fmaxf(m.w, 0.f);
    }
    st4(out + i * d + c, acc);
    if (outp.hi) planes_store4(outp, i, c, acc);
  }
}

__global__ void k_gine_bwd_dst(GpsGraph g, int d, const float* __restrict__ x, const float* __restrict__ e,
                               const float* __restrict__ g_o, float* __restrict__ g_e) {
  const int c = threadIdx.x * 4, ry = threadIdx.y, RY = blockDim.y;
  for (int64_t i = (int64_t)blockIdx.x * RY + ry; i < g.N; i += (int64_t)gridDim.x * RY) {
    const float4 go = ld4(g_o + i * d + c);
    const int kb = g.dst_ptr[i], ke = g.dst_ptr[i + 1];
    for (int k = kb; k < ke; ++k) {
      const int j = g.dst_src[k];
      const int64_t eid = g.dst_eid[k];
      const float4 m = f4add(ld4(x + (int64_t)j * d + c), ld4(e + eid * d + c));
      st4(g_e + eid * d + c, make_float4(m.x > 0.f ? go.x : 0.f, m.y > 0.f ? go.y : 0.f,
                                         m.z > 0.f ? go.z : 0.f, m.w > 0.f ? go.w : 0.f));
    }
  }
}

__global__ void k_gine_bwd_src(GpsGraph g, int d, const float* __restrict__ g_e, const float* __restrict__ g_o,
                               float eps, const float* __restrict__ add, float* __restrict__ g_x) {
  const int c = threadIdx.x * 4, ry = threadIdx.y, RY = blockDim.y;
  for (int64_t j = (int64_t)blockIdx.x * RY + ry; j < g.N; j += (int64_t)gridDim.x * RY) {
    float4 acc = f4scale(ld4(g_o + j * d + c), 1.f + eps);
    if (add) acc = f4add(acc, ld4(add + j * d + c));
    const int kb = g.src_ptr[j], ke = g.src_ptr[j + 1];
    for (int k = kb; k < ke; ++k) acc = f4add(acc, ld4(g_e + (int64_t)g.src_eid[k] * d + c));
    st4(g_x + j * d + c, acc);
  }
}

// ---- GCN (symmetric-normalised adjacency with one unit self loop per node)
__global__ void k_gcn_dinv(GpsGraph g, float* __restrict__ dinv) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= g.N) return;
  int deg = 1;   // the self loop; existing self-loop edges are replaced by it (add_remaining_self_loops)
  for (int k = g.dst_ptr[i]; k < g.dst_ptr[i + 1]; ++k) deg += g.dst_src[k] != (int)i;
  dinv[i] = rsqrtf((float)deg);
}

// x_loc_i = x_i + drop(b + dinv_i (dinv_i Y_i + sum_{j->i, j != i} dinv_j Y_j))  [+ column sums of x_loc]
template <bool STATS>
__global__ void __launch_bounds__(1024) k_gcn_fwd(GpsGraph g, int d, const float* __restrict__ Y, int64_t ldy,
                                                  const float* __restrict__ dinv, const float* __restrict__ bias,
                                                  const float* __restrict__ x, float* __restrict__ xloc, DropCfg drop,
                                                  double* stats) {
  extern __shared__ float4 sm[];
  const int c = threadIdx.x * 4, ry = threadIdx.y, RY = blockDim.y;
  const uint64_t offs = drop.offset + ((drop.p > 0.f && drop.offset_dev) ? *drop.offset_dev : 0ull);
  const float4 b4 = ld4(bias + c);
  float4 acc[2] = {f4zero(), f4zero()};
  for (int64_t i = (int64_t)blockIdx.x * RY + ry; i < g.N; i += (int64_t)gridDim.x * RY) {
    const float di = dinv[i];
    float4 a = f4scale(ld4(Y + i * ldy + c), di);
    for (int k = g.dst_ptr[i]; k < g.dst_ptr[i + 1]; ++k) {
      const int j = g.dst_src[k];
      if (j == (int)i) continue;
      a = f4fma(make_float4(dinv[j], dinv[j], dinv[j], dinv[j]), ld4(Y + (int64_t)j * ldy + c), a);
    }
    float4 h = f4add(f4scale(a, di), b4);
    if (drop.p > 0.f) h = f4mul(h, dropout_scale4(drop.p, drop.seed, offs, drop.site, ((uint64_t)i * (uint64_t)d + c) >> 2));
    const float4 v = f4add(ld4(x + i * d + c), h);
    st4(xloc + i * d + c, v);
    if (STATS) {
      acc[0] = f4add(acc[0], v);
      acc[1] = f4fma(v, v, acc[1]);
    }
  }
  if (STATS) {
    double* ptrs[2] = {stats, stats + d};
    block_stats<2>(acc, ptrs, sm);
  }
}

// gY_j = dinv_j (dinv_j g_h_j + sum_{j->i, i != j} dinv_i g_h_i)   (the adjoint of the aggregation above)
__global__ void k_gcn_bwd(GpsGraph g, int d, const float* __restrict__ g_h, const float* __restrict__ dinv,
                          float* __restrict__ gY, int64_t ldg, Planes gYp) {
  const int c = threadIdx.x * 4, ry = threadIdx.y, RY = blockDim.y;
  for (int64_t j = (int64_t)blockIdx.x * RY + ry; j < g.N; j += (int64_t)gridDim.x * RY) {
    const float dj = dinv[j];
    float4 a = f4scale(ld4(g_h + j * d + c), dj);
    for (int k = g.src_ptr[j]; k < g.src_ptr[j + 1]; ++k) {
      const int i = g.src_dst[k];
      if (i == (int)j) continue;
      a = f4fma(make_float4(dinv[i], dinv[i], dinv[i], dinv[i]), ld4(g_h + (int64_t)i * d + c), a);
    }
    st4(gY + j * ldg + c, f4scale(a, dj));
    if (gYp.hi) planes_store4(gYp, j, c, f4scale(a, dj));
  }
}

}  // namespace

int gcn_dinv(const GpsGraph& g, float* dinv, cudaStream_t stream) {
  if (g.N == 0) return GPS_OK;
  k_gcn_dinv<<<(unsigned)ceil_div(g.N, (int64_t)256), 256, 0, stream>>>(g, dinv);
  GPS_LAUNCH_CHECK();
  return GPS_OK;
}

int gcn_fwd(const GpsGraph& g, int64_t d, const float* Y, int64_t ldy, const float* dinv, const float* bias,
            const float* x, float* xloc, DropCfg drop, double* stats, cudaStream_t stream) {
  if (g.N == 0) return GPS_OK;
  NodeGeom ng;
  GPS_TRY(node_geom(g.N, d, stats ? 2 : 0, &ng));
  if (stats)
    k_gcn_fwd<true><<<ng.grid, ng.block, ng.smem, stream>>>(g, (int)d, Y, ldy, dinv, bias, x, xloc, drop, stats);
  else
    k_gcn_fwd<false><<<ng.grid, ng.block, 0, stream>>>(g, (int)d, Y, ldy, dinv, bias, x, xloc, drop, nullptr);
  GPS_LAUNCH_CHECK();
  return GPS_OK;
}

int gcn_bwd(const GpsGraph& g, int64_t d, const float* g_h, const float* dinv, float* gY, int64_t ldg,
            cudaStream_t stream, Planes gYp) {
  if (g.N == 0) return GPS_OK;
  NodeGeom ng;
  GPS_TRY(node_geom(g.N, d, 0, &ng));
  k_gcn_bwd<<<ng.grid, ng.block, 0, stream>>>(g, (int)d, g_h, dinv, gY, ldg, gYp);
  GPS_LAUNCH_CHECK();
  return GPS_OK;
}

int gatedgcn_fwd(const GpsGraph& g, int64_t d, const float* Ax, const float* Bx, const float* Dx, const float* Ex,
                 int64_t ldy, float* Ce, float* xt, double* stats_x, double* stats_e, cudaStream_t stream,
                 const float* gate) {
  if (g.N == 0) return GPS_OK;
  NodeGeom ng;
  const bool stats = stats_x || stats_e;
  GPS_TRY(node_geom(g.N, d, stats ? 4 : 0, &ng));
  if (stats && gate)
    k_gatedgcn_fwd<true, true><<<ng.grid, ng.block, ng.smem, stream>>>(g, (int)d, Ax, Bx, Dx, Ex, ldy, Ce, xt, stats_x,
                                                                         stats_e, gate);
  else if (stats)
    k_gatedgcn_fwd<true, false><<<ng.grid, ng.block, ng.smem, stream>>>(g, (int)d, Ax, Bx, Dx, Ex, ldy, Ce, xt, stats_x,
                                                                          stats_e, nullptr);
  else if (gate)
    k_gatedgcn_fwd<false, true><<<ng.grid, ng.block, 0, stream>>>(g, (int)d, Ax, Bx, Dx, Ex, ldy, Ce, xt, nullptr,
                                                                    nullptr, gate);
  else
    k_gatedgcn_fwd<false, false><<<ng.grid, ng.block, 0, stream>>>(g, (int)d, Ax, Bx, Dx, Ex, ldy, Ce, xt, nullptr,
                                                                     nullptr, nullptr);
  GPS_LAUNCH_CHECK();
  return GPS_OK;
}

int gatedgcn_es_nwarps(int64_t d) { return (int)(round_up(d / 4, 32) / 32); }

int gatedgcn_bwd_dst(const GpsGraph& g, int64_t d, const float* g_xt, int64_t ldg, const float* ehat, const float* Bx,
                     int64_t ldy, float* g_e, float* g_num, float* g_Dx, cudaStream_t stream, Planes g_e_p, Planes g_Dx_p,
                     const float* gate, float* g_gate) {
  if (g.N == 0) return GPS_OK;
  NodeGeom ng;
  GPS_TRY(node_geom(g.N, d, 0, &ng));
  if (gate) {
    GPS_REQUIRE(g_gate, GPS_ERR_ARG, "gatedgcn_bwd_dst: the gated pass needs the g_gate buffer");
    const int C4p = (int)round_up(d / 4, 32);   // whole warps per node row (node_geom allows d / 4 <= 1024)
    const int RY = C4p >= 256 ? 1 : 256 / C4p;
    const int64_t blocks = std::min<int64_t>(ceil_div(g.N, (int64_t)RY * 2), kNumSMs * 16);
    k_gatedgcn_bwd_dst<true><<<dim3((unsigned)blocks), dim3(C4p, RY), 0, stream>>>(g, (int)d, g_xt, ldg, ehat, Bx, ldy, g_e,
                                                                                   g_num, g_Dx, g_e_p, g_Dx_p, gate, g_gate);
  } else {
    k_gatedgcn_bwd_dst<false><<<ng.grid, ng.block, 0, stream>>>(g, (int)d, g_xt, ldg, ehat, Bx, ldy, g_e, g_num, g_Dx, g_e_p,
                                                                g_Dx_p, nullptr, nullptr);
  }
  GPS_LAUNCH_CHECK();
  return GPS_OK;
}

int gatedgcn_bwd_src(const GpsGraph& g, int64_t d, const float* g_e, const float* ehat, const float* g_num,
                     float* g_Ex, float* g_Bx, int64_t ldg, cudaStream_t stream, Planes g_Ex_p, Planes g_Bx_p,
                     const float* gate) {
  if (g.N == 0) return GPS_OK;
  NodeGeom ng;
  GPS_TRY(node_geom(g.N, d, 0, &ng));
  if (gate)
    k_gatedgcn_bwd_src<true><<<ng.grid, ng.block, 0, stream>>>(g, (int)d, g_e, ehat, g_num, g_Ex, g_Bx, ldg, g_Ex_p, g_Bx_p,
                                                               gate);
  else
    k_gatedgcn_bwd_src<false><<<ng.grid, ng.block, 0, stream>>>(g, (int)d, g_e, ehat, g_num, g_Ex, g_Bx, ldg, g_Ex_p,
                                                                g_Bx_p, nullptr);
  GPS_LAUNCH_CHECK();
  return GPS_OK;
}

int gine_fwd(const GpsGraph& g, int64_t d, const float* x, const float* e, float eps, float* out,
             cudaStream_t stream, Planes outp) {
  if (g.N == 0) return GPS_OK;
  NodeGeom ng;
  GPS_TRY(node_geom(g.N, d, 0, &ng));
  k_gine_fwd<<<ng.grid, ng.block, 0, stream>>>(g, (int)d, x, e, eps, out, outp);
  GPS_LAUNCH_CHECK();
  return GPS_OK;
}

int gine_bwd_dst(const GpsGraph& g, int64_t d, const float* x, const float* e, const float* g_o, float* g_e,
                 cudaStream_t stream) {
  if (g.N == 0) return GPS_OK;
  NodeGeom ng;
  GPS_TRY(node_geom(g.N, d, 0, &ng));
  k_gine_bwd_dst<<<ng.grid, ng.block, 0, stream>>>(g, (int)d, x, e, g_o, g_e);
  GPS_LAUNCH_CHECK();
  return GPS_OK;
}

int gine_bwd_src(const GpsGraph& g, int64_t d, const float* g_e, const float* g_o, float eps, const float* add,
                 float* g_x, cudaStream_t stream) {
  if (g.N == 0) return GPS_OK;
  NodeGeom ng;
  GPS_TRY(node_geom(g.N, d, 0, &ng));
  k_gine_bwd_src<<<ng.grid, ng.block, 0, stream>>>(g, (int)d, g_e, g_o, eps, add, g_x);
  GPS_LAUNCH_CHECK();
  return GPS_OK;
}

}  // namespace gps
