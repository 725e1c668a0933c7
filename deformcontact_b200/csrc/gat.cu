// K6 multi-head: PyG 2.5.x GATConv with any number of heads, concat or mean (nn/conv/gat_conv.py, utils/softmax.py).
// Forward softmax + aggregation in one kernel, the backward as one by-receiver and one by-source kernel, and the attention-vector
// gradients as a two-stage column reduction.  One group of G lanes (8 / 16 / 32, never wider than a warp) owns one node; lanes
// cover the node's row in VEC-float chunks (float4 when C % 4 == 0 and every row is 16-byte aligned, else scalar).
// Every sum per (node, head) is taken by one lane in CSR order (= original edge order), then the self loop: no atomics,
// bitwise reproducible.  Values a group writes in one phase and reads in the next (alpha, dalpha, da_src) go through global
// memory behind a __syncwarp(), which orders memory among the lanes of the warp; they are read with plain (coherent) loads.
#include "common.cuh"

namespace {
using namespace dcb;

constexpr int AG_ROWS = 2048;  // rows per stage-1 block of the attention-vector gradient (as dc_colsum)

__device__ __forceinline__ float leaky(float z, float slope) { return z > 0.f ? z : z * slope; }

template <int VEC>
struct Fv {
  float v[VEC];
};
template <int VEC>
__device__ __forceinline__ Fv<VEC> ldv(const float* __restrict__ p) {
  Fv<VEC> r;
  if constexpr (VEC == 4) {
    const float4 t = __ldg(reinterpret_cast<const float4*>(p));
    r.v[0] = t.x; r.v[1] = t.y; r.v[2] = t.z; r.v[3] = t.w;
  } else {
    r.v[0] = __ldg(p);
  }
  return r;
}
template <int VEC>
__device__ __forceinline__ void stv(float* __restrict__ p, const Fv<VEC>& r) {
  if constexpr (VEC == 4) *reinterpret_cast<float4*>(p) = make_float4(r.v[0], r.v[1], r.v[2], r.v[3]);
  else p[0] = r.v[0];
}
template <int VEC>
__device__ __forceinline__ void mul_add(Fv<VEC>& acc, float w, const Fv<VEC>& x) {
#pragma unroll
  for (int u = 0; u < VEC; ++u) acc.v[u] = __fadd_rn(acc.v[u], __fmul_rn(w, x.v[u]));
}

// Forward.  Phase 1 (lane = head, h += G): per-head max and exp-sum of z = leaky_relu(a_src[j] + a_dst[i]) over i's CSR edges,
// then the self loop, in the order of dc_gat_softmax but with the exponentials and their sum in fp64, so that alpha (written by
// original edge id, rounded once to fp32) is as exact as an fp32 value can be: the backward subtracts sum alpha*dalpha from
// dalpha, which amplifies any error of alpha.  Phase 2 (lane = output chunk, q += G):
// sum alpha * xs[j] in CSR order, then the self term; concat writes head h to columns [h*C, (h+1)*C), mean adds the heads in
// order and divides by H; then + bias and ReLU.
template <int VEC, int G>
__global__ void __launch_bounds__(256)
gat_aggregate_kernel(const int32_t* __restrict__ rowptr, const int32_t* __restrict__ nbr, const int32_t* __restrict__ eid,
                     const float* __restrict__ xs, int64_t ldx, const float* __restrict__ a_src, const float* __restrict__ a_dst,
                     float slope, int H, int C, int concat, const float* __restrict__ bias, int relu, int64_t N,
                     float* __restrict__ out, int64_t ldo, float* alpha_edge, float* alpha_self) {
  const int l = threadIdx.x % G;
  const int64_t i = (int64_t)blockIdx.x * (256 / G) + threadIdx.x / G;
  const bool live = i < N;
  const int beg = live ? rowptr[i] : 0, end = live ? rowptr[i + 1] : 0;
  if (live) {
    for (int h = l; h < H; h += G) {
      const float ad = a_dst[i * H + h];
      const float es = leaky(a_src[i * H + h] + ad, slope);
      float mx = es;
      for (int p = beg; p < end; ++p) mx = fmaxf(mx, leaky(a_src[(int64_t)nbr[p] * H + h] + ad, slope));
      const double m = mx;
      double sum = 0.0;
      for (int p = beg; p < end; ++p) sum += exp((double)leaky(a_src[(int64_t)nbr[p] * H + h] + ad, slope) - m);
      const double xself = exp((double)es - m);
      sum += xself;
      sum += 1e-16;
      for (int p = beg; p < end; ++p)
        alpha_edge[(int64_t)eid[p] * H + h] = (float)(exp((double)leaky(a_src[(int64_t)nbr[p] * H + h] + ad, slope) - m) / sum);
      alpha_self[i * H + h] = (float)(xself / sum);
    }
  }
  __syncwarp();
  if (!live) return;
  const int cq = C / VEC;
  const int nq = concat ? H * cq : cq;
  const int nh = concat ? 1 : H;
  for (int q = l; q < nq; q += G) {
    Fv<VEC> tot;
    for (int k = 0; k < nh; ++k) {
      const int h = concat ? q / cq : k;
      const int64_t col = (int64_t)h * C + (int64_t)(q % cq) * VEC;
      Fv<VEC> acc;
#pragma unroll
      for (int u = 0; u < VEC; ++u) acc.v[u] = 0.f;
#pragma unroll 4
      for (int p = beg; p < end; ++p)
        mul_add(acc, alpha_edge[(int64_t)eid[p] * H + h], ldv<VEC>(xs + (int64_t)nbr[p] * ldx + col));
      mul_add(acc, alpha_self[i * H + h], ldv<VEC>(xs + i * ldx + col));
      if (k == 0) tot = acc;
      else {
#pragma unroll
        for (int u = 0; u < VEC; ++u) tot.v[u] = __fadd_rn(tot.v[u], acc.v[u]);
      }
    }
    if (!concat) {
#pragma unroll
      for (int u = 0; u < VEC; ++u) tot.v[u] = __fdiv_rn(tot.v[u], (float)H);
    }
    if (bias) {
      const Fv<VEC> b = ldv<VEC>(bias + (int64_t)q * VEC);
#pragma unroll
      for (int u = 0; u < VEC; ++u) tot.v[u] = __fadd_rn(tot.v[u], b.v[u]);
    }
    if (relu) {
#pragma unroll
      for (int u = 0; u < VEC; ++u) tot.v[u] = fmaxf(tot.v[u], 0.f);
    }
    stv<VEC>(out + i * ldo + (int64_t)q * VEC, tot);
  }
}

// Backward by receiver.  Phase 1: i's (edge, head) pairs — CSR edges, then the self loop — are spread over the lanes; a lane takes
// dalpha = scale * <dout[i, h*hs : h*hs + C], xs[j, h*C : (h+1)*C]> sequentially (fp64 accumulator, for the same reason),
// with EXT adds the gradient that reaches alpha itself (dalpha_edge [E, H] by edge id, dalpha_self [N, H]; either may be null),
// and stashes it in dz_edge / dz_self.  Phase 2
// (lane = head): s = sum alpha * dalpha in CSR order then the self loop; dz = alpha * (dalpha - s) * leaky_relu'(z), written over
// the stash; da_dst[i, h] = sum of dz in the same order.
template <int VEC, int G, bool EXT>
__global__ void __launch_bounds__(256)
gat_bwd_edge_heads_kernel(const int32_t* __restrict__ rowptr, const int32_t* __restrict__ nbr, const int32_t* __restrict__ eid,
                          const float* __restrict__ a_src, const float* __restrict__ a_dst, float slope,
                          const float* __restrict__ alpha_edge, const float* __restrict__ alpha_self, const float* __restrict__ xs,
                          int64_t ldx, const float* __restrict__ dout, int64_t ldd, int64_t hs, float scale, int H, int C, int64_t N,
                          const float* __restrict__ dalpha_edge, const float* __restrict__ dalpha_self, float* dz_edge,
                          float* dz_self, float* __restrict__ da_dst) {
  const int l = threadIdx.x % G;
  const int64_t i = (int64_t)blockIdx.x * (256 / G) + threadIdx.x / G;
  const bool live = i < N;
  const int beg = live ? rowptr[i] : 0, end = live ? rowptr[i + 1] : 0;
  if (live) {
    const int64_t pairs = (int64_t)(end - beg + 1) * H;
    for (int64_t t = l; t < pairs; t += G) {
      const int p = beg + (int)(t / H);
      const int h = (int)(t % H);
      const bool self = p == end;
      const int64_t j = self ? i : nbr[p];
      const float* a = xs + j * ldx + (int64_t)h * C;
      const float* g = dout + i * ldd + h * hs;
      double acc = 0.0;   // fp64, rounded once: phase 2 subtracts sum alpha*dalpha from dalpha, which amplifies its rounding
#pragma unroll 2
      for (int c = 0; c < C; c += VEC) {
        const Fv<VEC> x = ldv<VEC>(a + c), y = ldv<VEC>(g + c);
#pragma unroll
        for (int u = 0; u < VEC; ++u) acc = fma((double)y.v[u], (double)x.v[u], acc);
      }
      float d = __fmul_rn((float)acc, scale);
      const int64_t k = self ? i * H + h : (int64_t)eid[p] * H + h;
      if constexpr (EXT) {
        const float* ext = self ? dalpha_self : dalpha_edge;
        if (ext) d = __fadd_rn(d, ext[k]);
      }
      if (self) dz_self[k] = d;
      else dz_edge[k] = d;
    }
  }
  __syncwarp();
  if (!live) return;
  for (int h = l; h < H; h += G) {
    float s = 0.f;
    for (int p = beg; p <= end; ++p) {
      const bool self = p == end;
      const int64_t k = self ? i * H + h : (int64_t)eid[p] * H + h;
      s = fmaf(self ? alpha_self[k] : alpha_edge[k], self ? dz_self[k] : dz_edge[k], s);
    }
    const float ad = a_dst[i * H + h];
    float tot = 0.f;
    for (int p = beg; p <= end; ++p) {
      const bool self = p == end;
      const int64_t k = self ? i * H + h : (int64_t)eid[p] * H + h;
      const float al = self ? alpha_self[k] : alpha_edge[k];
      const float dal = self ? dz_self[k] : dz_edge[k];
      const float z = a_src[(self ? i : (int64_t)nbr[p]) * H + h] + ad;
      const float dz = al * (dal - s) * (z > 0.f ? 1.f : slope);
      if (self) dz_self[k] = dz;
      else dz_edge[k] = dz;
      tot += dz;
    }
    da_dst[i * H + h] = tot;
  }
}

// Backward by source j (rows of the by-source CSR: nbr = receivers).  Phase 1 (lane = head): da_src[j, h] = sum dz over j's
// out-edges in CSR order, then dz_self.  Phase 2 (lane = chunk of the H*C row):
//   dxs[j, h, c] = scale * (sum_e alpha[e, h] dout[dst_e, h*hs + c] + alpha_self[j, h] dout[j, h*hs + c])
//                  + da_src[j, h] att_src[h, c] + da_dst[j, h] att_dst[h, c].
template <int VEC, int G>
__global__ void __launch_bounds__(256)
gat_scatter_heads_kernel(const int32_t* __restrict__ rowptr, const int32_t* __restrict__ nbr, const int32_t* __restrict__ eid,
                         const float* __restrict__ alpha_edge, const float* __restrict__ alpha_self,
                         const float* __restrict__ dz_edge, const float* __restrict__ dz_self, const float* __restrict__ da_dst,
                         const float* __restrict__ att_src, const float* __restrict__ att_dst, const float* __restrict__ dout,
                         int64_t ldd, int64_t hs, float scale, int H, int C, int64_t N, float* __restrict__ dxs, int64_t lddx,
                         float* da_src) {
  const int l = threadIdx.x % G;
  const int64_t j = (int64_t)blockIdx.x * (256 / G) + threadIdx.x / G;
  const bool live = j < N;
  const int beg = live ? rowptr[j] : 0, end = live ? rowptr[j + 1] : 0;
  if (live) {
    for (int h = l; h < H; h += G) {
      float s = 0.f;
      for (int p = beg; p < end; ++p) s += dz_edge[(int64_t)eid[p] * H + h];
      da_src[j * H + h] = s + dz_self[j * H + h];
    }
  }
  __syncwarp();
  if (!live) return;
  const int cq = C / VEC;
  for (int q = l; q < H * cq; q += G) {
    const int h = q / cq;
    const int64_t c = (int64_t)(q % cq) * VEC;
    const int64_t gc = h * hs + c;
    Fv<VEC> acc;
#pragma unroll
    for (int u = 0; u < VEC; ++u) acc.v[u] = 0.f;
#pragma unroll 4
    for (int p = beg; p < end; ++p) mul_add(acc, alpha_edge[(int64_t)eid[p] * H + h], ldv<VEC>(dout + (int64_t)nbr[p] * ldd + gc));
    mul_add(acc, alpha_self[j * H + h], ldv<VEC>(dout + j * ldd + gc));
    const float ds = da_src[j * H + h], dd = da_dst[j * H + h];
    const Fv<VEC> as = ldv<VEC>(att_src + (int64_t)h * C + c), at = ldv<VEC>(att_dst + (int64_t)h * C + c);
#pragma unroll
    for (int u = 0; u < VEC; ++u) {
      float v = scale == 1.f ? acc.v[u] : __fmul_rn(acc.v[u], scale);
      v = __fadd_rn(v, __fmul_rn(ds, as.v[u]));
      acc.v[u] = __fadd_rn(v, __fmul_rn(dd, at.v[u]));
    }
    stv<VEC>(dxs + j * lddx + (int64_t)q * VEC, acc);
  }
}

// datt_src[h, c] = sum_n da_src[n, h] xs[n, h*C + c] and datt_dst likewise.  Stage 1: partial[chunk, {src, dst}, n] over AG_ROWS
// rows (8 interleaved row lanes, then a fixed tree in shared memory); stage 2 adds the chunks in order.  As dc_colsum.
__global__ void __launch_bounds__(256)
gat_att_grad_stage1(const float* __restrict__ xs, int64_t ldx, const float* __restrict__ da_src, const float* __restrict__ da_dst,
                    int64_t M, int H, int C, float* __restrict__ partial) {
  __shared__ float sm[2][8][33];
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  const int64_t HC = (int64_t)H * C;
  const int64_t n = (int64_t)blockIdx.x * 32 + tx;
  const int64_t r0 = (int64_t)blockIdx.y * AG_ROWS;
  const int64_t r1 = min(M, r0 + AG_ROWS);
  float s = 0.f, d = 0.f;
  if (n < HC) {
    const int h = (int)(n / C);
    for (int64_t r = r0 + ty; r < r1; r += 8) {
      const float x = xs[r * ldx + n];
      s = fmaf(da_src[r * H + h], x, s);
      d = fmaf(da_dst[r * H + h], x, d);
    }
  }
  sm[0][ty][tx] = s;
  sm[1][ty][tx] = d;
  __syncthreads();
  if (ty == 0 && n < HC) {
    float ts = sm[0][0][tx], td = sm[1][0][tx];
#pragma unroll
    for (int k = 1; k < 8; ++k) { ts += sm[0][k][tx]; td += sm[1][k][tx]; }
    partial[((int64_t)blockIdx.y * 2) * HC + n] = ts;
    partial[((int64_t)blockIdx.y * 2 + 1) * HC + n] = td;
  }
}
__global__ void gat_att_grad_stage2(const float* __restrict__ partial, int64_t chunks, int64_t HC, float* __restrict__ datt_src,
                                    float* __restrict__ datt_dst) {
  const int64_t n = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (n >= 2 * HC) return;
  float s = 0.f;
  for (int64_t c = 0; c < chunks; ++c) s += partial[c * 2 * HC + n];
  if (n < HC) datt_src[n] = s;
  else datt_dst[n - HC] = s;
}

bool al16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; }

// lanes per node: enough for the chunks of one row, at most a warp
int group_width(int64_t chunks) { return chunks <= 8 ? 8 : chunks <= 16 ? 16 : 32; }

}  // namespace

#define DC_GAT_DISPATCH(VEC_, G_, LAUNCH)                               \
  do {                                                                  \
    if ((VEC_) == 4) {                                                  \
      if ((G_) == 8) LAUNCH(4, 8); else if ((G_) == 16) LAUNCH(4, 16); else LAUNCH(4, 32); \
    } else {                                                            \
      if ((G_) == 8) LAUNCH(1, 8); else if ((G_) == 16) LAUNCH(1, 16); else LAUNCH(1, 32); \
    }                                                                   \
  } while (0)

extern "C" int dc_gat_aggregate(const int32_t* rowptr, const int32_t* nbr, const int32_t* eid, const float* xs, int64_t ldx,
                                const float* a_src, const float* a_dst, float slope, int32_t H, int32_t C, int32_t concat,
                                const float* bias, int32_t relu, int64_t N, float* out, int64_t ldo, float* alpha_edge,
                                float* alpha_self, dc_stream_t stream_) {
  cudaStream_t st = (cudaStream_t)stream_;
  DC_REQUIRE(H >= 1 && C >= 1 && N >= 0, DC_EINVAL, "gat_aggregate: heads and C must be >= 1");
  const int64_t width = concat ? (int64_t)H * C : C;
  DC_REQUIRE(ldx >= (int64_t)H * C && ldo >= width, DC_EINVAL, "gat_aggregate: ld smaller than the row");
  if (N == 0) return DC_OK;
  DC_REQUIRE(rowptr && xs && a_src && a_dst && out && alpha_edge && alpha_self, DC_EINVAL, "gat_aggregate: null pointer");
  const int vec = (C % 4 == 0 && ldx % 4 == 0 && ldo % 4 == 0 && al16(xs) && al16(out) && (!bias || al16(bias))) ? 4 : 1;
  const int G = group_width(width / vec);
#define DC_GAT_AGG(V, GG)                                                                                                   \
  gat_aggregate_kernel<V, GG><<<(unsigned)cdiv(N, 256 / GG), 256, 0, st>>>(rowptr, nbr, eid, xs, ldx, a_src, a_dst, slope, H, C, \
                                                                         concat ? 1 : 0, bias, relu ? 1 : 0, N, out, ldo,     \
                                                                         alpha_edge, alpha_self)
  DC_GAT_DISPATCH(vec, G, DC_GAT_AGG);
#undef DC_GAT_AGG
  DC_LAUNCH_CHECK();
  return DC_OK;
}

namespace {
// Both by-receiver entry points: the same checks, then the kernel without (EXT false) or with the external alpha gradient.
template <bool EXT>
int gat_bwd_edge_heads_launch(const int32_t* rowptr, const int32_t* nbr, const int32_t* eid, const float* a_src, const float* a_dst,
                              float slope, const float* alpha_edge, const float* alpha_self, const float* xs, int64_t ldx,
                              const float* dout, int64_t ldd, int64_t dout_head_stride, float dout_scale, int32_t H, int32_t C,
                              int64_t N, const float* dalpha_edge, const float* dalpha_self, float* dz_edge, float* dz_self,
                              float* da_dst, cudaStream_t st) {
  DC_REQUIRE(H >= 1 && C >= 1 && N >= 0 && dout_head_stride >= 0, DC_EINVAL, "gat_bwd_edge_heads: heads and C must be >= 1");
  DC_REQUIRE(ldx >= (int64_t)H * C && ldd >= (int64_t)(H - 1) * dout_head_stride + C, DC_EINVAL,
             "gat_bwd_edge_heads: ld smaller than the row");
  if (N == 0) return DC_OK;
  DC_REQUIRE(rowptr && a_src && a_dst && alpha_edge && alpha_self && xs && dout && dz_edge && dz_self && da_dst,
             DC_EINVAL, "gat_bwd_edge_heads: null pointer");
  const int vec = (C % 4 == 0 && ldx % 4 == 0 && ldd % 4 == 0 && dout_head_stride % 4 == 0 && al16(xs) && al16(dout)) ? 4 : 1;
  const int G = group_width(9 * (int64_t)H);     // pairs of a receiver of degree 8
#define DC_GAT_BWD(V, GG)                                                                                                        \
  gat_bwd_edge_heads_kernel<V, GG, EXT><<<(unsigned)cdiv(N, 256 / GG), 256, 0, st>>>(                                            \
      rowptr, nbr, eid, a_src, a_dst, slope, alpha_edge, alpha_self, xs, ldx, dout, ldd, dout_head_stride, dout_scale, H, C, N,  \
      dalpha_edge, dalpha_self, dz_edge, dz_self, da_dst)
  DC_GAT_DISPATCH(vec, G, DC_GAT_BWD);
#undef DC_GAT_BWD
  DC_LAUNCH_CHECK();
  return DC_OK;
}
}  // namespace

extern "C" int dc_gat_bwd_edge_heads(const int32_t* rowptr, const int32_t* nbr, const int32_t* eid, const float* a_src,
                                     const float* a_dst, float slope, const float* alpha_edge, const float* alpha_self, const float* xs,
                                     int64_t ldx, const float* dout, int64_t ldd, int64_t dout_head_stride, float dout_scale, int32_t H,
                                     int32_t C, int64_t N, float* dz_edge, float* dz_self, float* da_dst, dc_stream_t stream_) {
  return gat_bwd_edge_heads_launch<false>(rowptr, nbr, eid, a_src, a_dst, slope, alpha_edge, alpha_self, xs, ldx, dout, ldd,
                                          dout_head_stride, dout_scale, H, C, N, nullptr, nullptr, dz_edge, dz_self, da_dst,
                                          (cudaStream_t)stream_);
}

extern "C" int dc_gat_bwd_edge_heads_ext(const int32_t* rowptr, const int32_t* nbr, const int32_t* eid, const float* a_src,
                                         const float* a_dst, float slope, const float* alpha_edge, const float* alpha_self,
                                         const float* xs, int64_t ldx, const float* dout, int64_t ldd, int64_t dout_head_stride,
                                         float dout_scale, int32_t H, int32_t C, int64_t N, const float* dalpha_edge,
                                         const float* dalpha_self, float* dz_edge, float* dz_self, float* da_dst,
                                         dc_stream_t stream_) {
  if (!dalpha_edge && !dalpha_self)     // nothing to add: the kernel of dc_gat_bwd_edge_heads, bit for bit
    return gat_bwd_edge_heads_launch<false>(rowptr, nbr, eid, a_src, a_dst, slope, alpha_edge, alpha_self, xs, ldx, dout, ldd,
                                            dout_head_stride, dout_scale, H, C, N, nullptr, nullptr, dz_edge, dz_self, da_dst,
                                            (cudaStream_t)stream_);
  return gat_bwd_edge_heads_launch<true>(rowptr, nbr, eid, a_src, a_dst, slope, alpha_edge, alpha_self, xs, ldx, dout, ldd,
                                         dout_head_stride, dout_scale, H, C, N, dalpha_edge, dalpha_self, dz_edge, dz_self, da_dst,
                                         (cudaStream_t)stream_);
}

extern "C" int dc_gat_scatter_heads(const int32_t* rowptr_t, const int32_t* nbr_t, const int32_t* eid_t, const float* alpha_edge,
                                    const float* alpha_self, const float* dz_edge, const float* dz_self, const float* da_dst,
                                    const float* att_src, const float* att_dst, const float* dout, int64_t ldd, int64_t dout_head_stride,
                                    float dout_scale, int32_t H, int32_t C, int64_t N, float* dxs, int64_t lddx, float* da_src,
                                    dc_stream_t stream_) {
  cudaStream_t st = (cudaStream_t)stream_;
  DC_REQUIRE(H >= 1 && C >= 1 && N >= 0 && dout_head_stride >= 0, DC_EINVAL, "gat_scatter_heads: heads and C must be >= 1");
  DC_REQUIRE(lddx >= (int64_t)H * C && ldd >= (int64_t)(H - 1) * dout_head_stride + C, DC_EINVAL,
             "gat_scatter_heads: ld smaller than the row");
  if (N == 0) return DC_OK;
  DC_REQUIRE(rowptr_t && alpha_edge && alpha_self && dz_edge && dz_self && da_dst && att_src && att_dst && dout &&
             dxs && da_src, DC_EINVAL, "gat_scatter_heads: null pointer");
  const int vec = (C % 4 == 0 && ldd % 4 == 0 && lddx % 4 == 0 && dout_head_stride % 4 == 0 && al16(dout) && al16(dxs) &&
                   al16(att_src) && al16(att_dst)) ? 4 : 1;
  const int G = group_width((int64_t)H * C / vec);
#define DC_GAT_SCT(V, GG)                                                                                                       \
  gat_scatter_heads_kernel<V, GG><<<(unsigned)cdiv(N, 256 / GG), 256, 0, st>>>(rowptr_t, nbr_t, eid_t, alpha_edge, alpha_self,     \
                                                                             dz_edge, dz_self, da_dst, att_src, att_dst, dout,   \
                                                                             ldd, dout_head_stride, dout_scale, H, C, N, dxs,    \
                                                                             lddx, da_src)
  DC_GAT_DISPATCH(vec, G, DC_GAT_SCT);
#undef DC_GAT_SCT
  DC_LAUNCH_CHECK();
  return DC_OK;
}

extern "C" size_t dc_gat_att_grad_workspace_bytes(int64_t N, int32_t H, int32_t C) {
  const int64_t hc = (int64_t)(H > 0 ? H : 1) * (C > 0 ? C : 1);
  return dcb::align_up((size_t)dcb::cdiv(N > 0 ? N : 1, AG_ROWS) * 2 * hc * sizeof(float), 256);
}

extern "C" int dc_gat_att_grad(const float* xs, int64_t ldx, const float* da_src, const float* da_dst, int64_t N, int32_t H, int32_t C,
                               float* datt_src, float* datt_dst, void* workspace, size_t workspace_bytes, dc_stream_t stream_) {
  cudaStream_t st = (cudaStream_t)stream_;
  DC_REQUIRE(H >= 1 && C >= 1 && N >= 0, DC_EINVAL, "gat_att_grad: heads and C must be >= 1");
  DC_REQUIRE(ldx >= (int64_t)H * C, DC_EINVAL, "gat_att_grad: ld smaller than the row");
  DC_REQUIRE(datt_src && datt_dst, DC_EINVAL, "gat_att_grad: null pointer");
  const int64_t HC = (int64_t)H * C;
  if (N == 0) {
    DC_CUDA(cudaMemsetAsync(datt_src, 0, HC * sizeof(float), st));
    DC_CUDA(cudaMemsetAsync(datt_dst, 0, HC * sizeof(float), st));
    return DC_OK;
  }
  DC_REQUIRE(xs && da_src && da_dst, DC_EINVAL, "gat_att_grad: null pointer");
  DC_REQUIRE(workspace && workspace_bytes >= dc_gat_att_grad_workspace_bytes(N, H, C), DC_EWORKSPACE, "gat_att_grad: workspace");
  const int64_t chunks = cdiv(N, AG_ROWS);
  DC_REQUIRE(chunks <= 65535, DC_ENOSUP, "gat_att_grad: too many nodes");
  dim3 grid((unsigned)cdiv(HC, 32), (unsigned)chunks);
  gat_att_grad_stage1<<<grid, 256, 0, st>>>(xs, ldx, da_src, da_dst, N, H, C, static_cast<float*>(workspace));
  gat_att_grad_stage2<<<(unsigned)cdiv(2 * HC, 256), 256, 0, st>>>(static_cast<float*>(workspace), chunks, HC, datt_src, datt_dst);
  DC_LAUNCHED(2);
  return DC_OK;
}
