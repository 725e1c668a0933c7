// Edge weights for TAGConv / GCNConv: PyG 2.5.2's weighted gcn_norm (nn/conv/gcn_conv.py:gcn_norm with
// utils/loop.py:add_remaining_self_loops) on the device, its backward with respect to edge_weight, and the sampled
// dot-product kernel (SDDMM) that gives dL/dnorm_e from the saved hop inputs.
// Every per-node sum runs sequentially in CSR order (= original edge order), then the appended loop; no floating-point
// atomics.  The only atomic is the integer atomicMax that finds the last self-loop edge of each node, whose result does not
// depend on the order in which the edges arrive.
#include "common.cuh"

namespace {
using namespace dcb;

// loop_eid[n] = largest edge id e with src_e == dst_e == n (the loop whose weight PyG's `loop_attr[idx] = edge_attr[mask]`
// keeps on the CPU: the last write wins); stays -1 when n has no self-loop edge.
__global__ void last_loop_kernel(const int64_t* __restrict__ ei, int64_t E, int64_t N, int32_t* __restrict__ loop_eid) {
  const int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (e >= E) return;
  const int64_t s = ei[e], t = ei[E + e];
  if (s == t && s >= 0 && s < N) atomicMax(loop_eid + s, (int32_t)e);
}

// dis_i = deg_i^-1/2 (0 where deg_i == 0, NaN where deg_i < 0, as pow(-0.5) + masked_fill(inf, 0)),
// deg_i = sum of w over i's by-target CSR row in order, then + the loop weight (loop mode 1).
__device__ __forceinline__ float inv_sqrt_deg(float d) { return d == 0.f ? 0.f : __fdiv_rn(1.0f, __fsqrt_rn(d)); }

__global__ void norm_node_kernel(const int32_t* __restrict__ rowptr, const int32_t* __restrict__ eid, const float* __restrict__ w,
                                 float fill, int normalize, int loops, const int32_t* __restrict__ loop_eid, int64_t N,
                                 float* __restrict__ dis, float* __restrict__ loop_w, float* __restrict__ self_w) {
  const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i >= N) return;
  const float lw = loops ? (loop_eid[i] >= 0 ? w[loop_eid[i]] : fill) : 0.f;
  float di = 1.f;
  if (normalize) {
    float deg = 0.f;
    for (int p = rowptr[i]; p < rowptr[i + 1]; ++p) deg = __fadd_rn(deg, w[eid[p]]);
    if (loops) deg = __fadd_rn(deg, lw);
    di = inv_sqrt_deg(deg);
    dis[i] = di;
  }
  if (loops) {
    loop_w[i] = lw;
    self_w[i] = normalize ? __fmul_rn(__fmul_rn(di, lw), di) : lw;
  }
}

// norm_e = (dis[src] * w_e) * dis[dst] (PyG's order), or w_e without normalisation, written at every CSR position of one
// structure: blockIdx.y = 0 walks the by-target rows (nbr = source), 1 the by-source rows (nbr = target).
__global__ void norm_edges_kernel(const int32_t* __restrict__ rp0, const int32_t* __restrict__ nb0, const int32_t* __restrict__ id0,
                                  float* __restrict__ w0, int2* __restrict__ rec0, const int32_t* __restrict__ rp1,
                                  const int32_t* __restrict__ nb1, const int32_t* __restrict__ id1, float* __restrict__ w1,
                                  int2* __restrict__ rec1, const float* __restrict__ w, const float* __restrict__ dis, int64_t N) {
  const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i >= N) return;
  const bool by_src = blockIdx.y == 1;
  const int32_t* rp = by_src ? rp1 : rp0;
  const int32_t* nb = by_src ? nb1 : nb0;
  const int32_t* id = by_src ? id1 : id0;
  float* wo = by_src ? w1 : w0;
  int2* rec = by_src ? rec1 : rec0;
  const float di = dis ? dis[i] : 1.f;
  for (int p = rp[i]; p < rp[i + 1]; ++p) {
    const int j = nb[p];
    const float we = w[id[p]];
    float n = we;
    if (dis) n = by_src ? __fmul_rn(__fmul_rn(di, we), dis[j]) : __fmul_rn(__fmul_rn(dis[j], we), di);
    if (wo) wo[p] = n;
    if (rec) rec[p] = make_int2(j, __float_as_int(n));
  }
}

// SDDMM: one warp per receiver i; for each of i's CSR edges p (then the self term, when s_self is given)
//   s = sum_k <G_k[i], H_k[nbr[p]]>.
// A lane covers columns lane*VEC + 32*VEC*m.  Per (edge, pair) a lane sums its columns in fp32 (F/32 products), converts once
// to fp64, adds the pairs in fp64, and the warp reduces with a fixed xor-shuffle tree in fp64: the result is rounded to fp32
// once.  Edges go four at a time, so a lane has 4 row gathers in flight per pair and G_k[i] is read once per four edges
// (it stays in L1).
struct PairArgs {
  const float* g[DC_MAX_CHAIN];
  const float* h[DC_MAX_CHAIN];
  int64_t ldg[DC_MAX_CHAIN], ldh[DC_MAX_CHAIN];
};

template <int VEC>
__device__ __forceinline__ float dotv(const float* a, const float* b) {
  if constexpr (VEC == 4) {
    const float4 x = __ldg(reinterpret_cast<const float4*>(a)), y = __ldg(reinterpret_cast<const float4*>(b));
    return fmaf(x.w, y.w, fmaf(x.z, y.z, fmaf(x.y, y.y, x.x * y.x)));
  } else {
    return __ldg(a) * __ldg(b);
  }
}

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

template <int VEC>
__global__ void __launch_bounds__(256)
edge_sddmm_kernel(const int32_t* __restrict__ rowptr, const int32_t* __restrict__ nbr, const int32_t* __restrict__ eid,
                  const PairArgs pa, int np, int64_t N, int F, int accumulate, float* __restrict__ s_edge,
                  float* __restrict__ s_self) {
  const int lane = threadIdx.x & 31;
  const int64_t i = (int64_t)blockIdx.x * 8 + (threadIdx.x >> 5);
  if (i >= N) return;   // whole warp
  const int beg = rowptr[i], end = rowptr[i + 1] + (s_self ? 1 : 0);   // position rowptr[i+1] = the self term
  const int self_p = rowptr[i + 1];
  for (int p0 = beg; p0 < end; p0 += 4) {
    int64_t j[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) j[u] = (p0 + u < end && p0 + u != self_p) ? (int64_t)nbr[p0 + u] : i;
    double acc[4] = {0.0, 0.0, 0.0, 0.0};
#pragma unroll
    for (int k = 0; k < DC_MAX_CHAIN; ++k) {   // unrolled so that the pair arguments stay in the parameter bank
      if (k >= np) break;
      const float* g = pa.g[k] + i * pa.ldg[k];
      const float* h = pa.h[k];
      const int64_t ldh = pa.ldh[k];
      float part[4] = {0.f, 0.f, 0.f, 0.f};
      for (int c = lane * VEC; c < F; c += 32 * VEC) {
#pragma unroll
        for (int u = 0; u < 4; ++u) part[u] += dotv<VEC>(g + c, h + j[u] * ldh + c);
      }
#pragma unroll
      for (int u = 0; u < 4; ++u) acc[u] += (double)part[u];
    }
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const double v = warp_sum(acc[u]);
      const int p = p0 + u;
      if (lane == 0 && p < end) {
        float* dst = p == self_p ? s_self + i : s_edge + eid[p];
        *dst = accumulate ? (float)((double)*dst + v) : (float)v;
      }
    }
  }
}

// Backward of the normalisation, one thread per node n (fp64 throughout, rounded once per output):
//   dL/ddis_n = sum_{e: dst=n} s_e dis[src] w_e  (by-target row, CSR order)
//             + sum_{e: src=n} s_e w_e dis[dst]  (by-source row, CSR order)
//             + 2 s_loop_n lw_n dis_n             (appended loop)
//   dL/ddeg_n = -1/2 dis_n^3 dL/ddis_n, 0 where dis_n == 0 (deg_n == 0)
//   dL/dw_e   = s_e dis[src] dis[n] + dL/ddeg_n  for the by-target row of n,
//   dL/dw_loop_eid[n] = s_loop_n dis_n^2 + dL/ddeg_n  (the loop edge that supplied lw_n; other loop edges keep the 0 written
//   before the launch).
__global__ void norm_bwd_kernel(const int32_t* __restrict__ rowptr, const int32_t* __restrict__ nbr, const int32_t* __restrict__ eid,
                                const int32_t* __restrict__ rowptr_t, const int32_t* __restrict__ nbr_t,
                                const int32_t* __restrict__ eid_t, const float* __restrict__ w, const float* __restrict__ dis,
                                const float* __restrict__ loop_w, const int32_t* __restrict__ loop_eid,
                                const float* __restrict__ s_edge, const float* __restrict__ s_self, int64_t N,
                                float* __restrict__ dw) {
  const int64_t n = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (n >= N) return;
  const double dn = dis[n];
  double ddis = 0.0;
  for (int p = rowptr[n]; p < rowptr[n + 1]; ++p) {
    const int e = eid[p];
    ddis += (double)s_edge[e] * (double)dis[nbr[p]] * (double)w[e];
  }
  for (int p = rowptr_t[n]; p < rowptr_t[n + 1]; ++p) {
    const int e = eid_t[p];
    ddis += (double)s_edge[e] * (double)w[e] * (double)dis[nbr_t[p]];
  }
  if (s_self) ddis += 2.0 * (double)s_self[n] * (double)loop_w[n] * dn;
  const double ddeg = dn == 0.0 ? 0.0 : -0.5 * dn * dn * dn * ddis;
  for (int p = rowptr[n]; p < rowptr[n + 1]; ++p) {
    const int e = eid[p];
    dw[e] = (float)((double)s_edge[e] * (double)dis[nbr[p]] * dn + ddeg);
  }
  if (s_self && loop_eid[n] >= 0) dw[loop_eid[n]] = (float)((double)s_self[n] * dn * dn + ddeg);
}

bool al16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; }

}  // namespace

extern "C" int dc_gcn_norm_weighted(const int64_t* edge_index, int64_t E, int64_t N, const int32_t* rowptr, const int32_t* nbr,
                                    const int32_t* eid, const int32_t* rowptr_t, const int32_t* nbr_t, const int32_t* eid_t,
                                    const float* edge_weight, float fill_value, int normalize, int loop_mode, float* dis,
                                    float* loop_w, int32_t* loop_eid, float* self_w, float* w_fwd, void* edges_fwd, float* w_src,
                                    void* edges_src, dc_stream_t stream_) {
  cudaStream_t st = (cudaStream_t)stream_;
  DC_REQUIRE(N >= 0 && E >= 0 && N < (1ll << 31) - 1 && E < (1ll << 31) - 1, DC_EINVAL, "gcn_norm_weighted: N=%lld E=%lld",
             (long long)N, (long long)E);
  DC_REQUIRE(loop_mode == 0 || loop_mode == 1, DC_EINVAL, "gcn_norm_weighted: loop_mode must be 0 (none) or 1 (add remaining)");
  DC_REQUIRE(rowptr && (E == 0 || (nbr && eid && (w_fwd || edges_fwd))), DC_EINVAL,
             "gcn_norm_weighted: null pointer (by-target structure)");
  DC_REQUIRE(!(w_src || edges_src) || (rowptr_t && (E == 0 || (nbr_t && eid_t))), DC_EINVAL,
             "gcn_norm_weighted: null by-source structure");
  DC_REQUIRE(E == 0 || edge_weight, DC_EINVAL, "gcn_norm_weighted: null edge_weight");
  DC_REQUIRE(!normalize || dis, DC_EINVAL, "gcn_norm_weighted: normalize needs dis");
  DC_REQUIRE(loop_mode == 0 || (loop_w && loop_eid && self_w && (E == 0 || edge_index)), DC_EINVAL,
             "gcn_norm_weighted: loop mode needs edge_index, loop_w, loop_eid and self_w");
  DC_REQUIRE(!edges_fwd || (reinterpret_cast<uintptr_t>(edges_fwd) & 7) == 0, DC_EINVAL, "gcn_norm_weighted: records not 8-byte aligned");
  DC_REQUIRE(!edges_src || (reinterpret_cast<uintptr_t>(edges_src) & 7) == 0, DC_EINVAL, "gcn_norm_weighted: records not 8-byte aligned");
  if (N == 0) return DC_OK;
  const unsigned nb = (unsigned)cdiv(N, 256);
  if (loop_mode) {
    DC_CUDA(cudaMemsetAsync(loop_eid, 0xff, N * sizeof(int32_t), st));   // -1
    if (E > 0) {
      last_loop_kernel<<<(unsigned)cdiv(E, 256), 256, 0, st>>>(edge_index, E, N, loop_eid);
      DC_LAUNCH_CHECK();
    }
  }
  if (normalize || loop_mode) {
    norm_node_kernel<<<nb, 256, 0, st>>>(rowptr, eid, edge_weight, fill_value, normalize, loop_mode, loop_eid, N, dis, loop_w, self_w);
    DC_LAUNCH_CHECK();
  }
  if (E > 0) {
    const bool both = w_src || edges_src;
    norm_edges_kernel<<<dim3(nb, both ? 2 : 1), 256, 0, st>>>(rowptr, nbr, eid, w_fwd, static_cast<int2*>(edges_fwd), rowptr_t, nbr_t,
                                                             eid_t, w_src, static_cast<int2*>(edges_src), edge_weight,
                                                             normalize ? dis : nullptr, N);
    DC_LAUNCH_CHECK();
  }
  return DC_OK;
}

extern "C" int dc_edge_sddmm(const int32_t* rowptr, const int32_t* nbr, const int32_t* eid, const dc_sddmm_pair_t* pairs,
                             int32_t num_pairs, int64_t N, int32_t F, int accumulate, float* s_edge, float* s_self,
                             dc_stream_t stream_) {
  cudaStream_t st = (cudaStream_t)stream_;
  DC_REQUIRE(N >= 0 && F >= 1, DC_EINVAL, "edge_sddmm: N must be >= 0 and F >= 1");
  DC_REQUIRE(num_pairs >= 1 && num_pairs <= DC_MAX_CHAIN, DC_EINVAL, "edge_sddmm: 1 to %d pairs", DC_MAX_CHAIN);
  DC_REQUIRE(rowptr && nbr && eid && pairs && s_edge, DC_EINVAL, "edge_sddmm: null pointer");
  PairArgs a;
  bool vec = F % 4 == 0;
  for (int k = 0; k < DC_MAX_CHAIN; ++k) {
    const dc_sddmm_pair_t& q = pairs[k < num_pairs ? k : 0];
    if (k < num_pairs) {
      DC_REQUIRE(q.g && q.h, DC_EINVAL, "edge_sddmm: pair %d: null pointer", k);
      DC_REQUIRE(q.ldg >= F && q.ldh >= F, DC_EINVAL, "edge_sddmm: pair %d: leading dimension < F", k);
      vec = vec && q.ldg % 4 == 0 && q.ldh % 4 == 0 && al16(q.g) && al16(q.h);
    }
    a.g[k] = q.g; a.h[k] = q.h; a.ldg[k] = q.ldg; a.ldh[k] = q.ldh;
  }
  if (N == 0) return DC_OK;
  const unsigned grid = (unsigned)cdiv(N, 8);
  if (vec)
    edge_sddmm_kernel<4><<<grid, 256, 0, st>>>(rowptr, nbr, eid, a, num_pairs, N, F, accumulate ? 1 : 0, s_edge, s_self);
  else
    edge_sddmm_kernel<1><<<grid, 256, 0, st>>>(rowptr, nbr, eid, a, num_pairs, N, F, accumulate ? 1 : 0, s_edge, s_self);
  DC_LAUNCH_CHECK();
  return DC_OK;
}

extern "C" int dc_gcn_norm_weighted_backward(const int32_t* rowptr, const int32_t* nbr, const int32_t* eid, const int32_t* rowptr_t,
                                             const int32_t* nbr_t, const int32_t* eid_t, const float* edge_weight, const float* dis,
                                             const float* loop_w, const int32_t* loop_eid, const float* s_edge, const float* s_self,
                                             int64_t N, int64_t E, float* dw, dc_stream_t stream_) {
  cudaStream_t st = (cudaStream_t)stream_;
  DC_REQUIRE(N >= 0 && E >= 0, DC_EINVAL, "gcn_norm_weighted_backward: negative size");
  DC_REQUIRE(rowptr && rowptr_t && dis, DC_EINVAL, "gcn_norm_weighted_backward: null pointer");
  DC_REQUIRE(E == 0 || (nbr && eid && nbr_t && eid_t && edge_weight && s_edge && dw), DC_EINVAL,
             "gcn_norm_weighted_backward: null pointer");
  DC_REQUIRE(!s_self || (loop_w && loop_eid), DC_EINVAL, "gcn_norm_weighted_backward: the loop term needs loop_w and loop_eid");
  if (E > 0) DC_CUDA(cudaMemsetAsync(dw, 0, E * sizeof(float), st));
  if (N == 0) return DC_OK;
  norm_bwd_kernel<<<(unsigned)cdiv(N, 256), 256, 0, st>>>(rowptr, nbr, eid, rowptr_t, nbr_t, eid_t, edge_weight, dis, loop_w, loop_eid,
                                                         s_edge, s_self, N, dw);
  DC_LAUNCH_CHECK();
  return DC_OK;
}
