// Screening pass of DUNE on the warp-level tensor pipe (mma.sync m16n8k16, fp16 in / fp32 accumulate): same contract, same
// candidate lists and the same operand image as dune_screen_kernel (dune_screen_kernel.cuh), different execution shape.
//
// Why a second shape for this one pass.  The screening network is SINGLE-pass fp16 (no hi/lo split): per 32-wide layer and 128
// points it needs 3 tcgen05.mma of 128x32x16 -- the tensor pipe is 1 % busy -- but pays the full tcgen05 round trip five times
// per tile: tcgen05.st of the A operand, block barrier, elected issue, mbarrier wait, tcgen05.ld of 32 fp32 columns per point
// (544 B per point through the 64 B/clk TMEM read port).  ncu of dune_screen_kernel: 16 warps/SM, issue slots 53 % busy, no
// pipe above 40 %, and two thirds of a warp's time spent in those variable waits.  With mma.sync m16n8k16 the accumulator
// fragment of layer l IS the A fragment of layer l+1 (same lane <-> (row, column pair) map), so 32 points travel through all
// six layers inside one warp's registers: no TMEM, no mbarrier, no block barrier inside the network, warps drift freely and the
// MUFU (tanh), FMA, ALU and tensor phases of the four warps of a scheduler overlap.  The single fp16 pass costs 68 HMMA per 32
// points (585 clk of the legacy tensor pipe per scheduler) against 792 clk of MUFU.TANH -- the exact path (3 passes, 204 HMMA)
// is the one that needs tcgen05, and keeps it (dune_refine_kernel / dune_tcp_kernel).
//
// Two shapes share the per-tile code below (sm::screen_point): dune_screen_warp_kernel (the default, one warp per (environment, step)
// item, at the end of this file) and dune_screen_mma_kernel (one CTA of 4 warps per item, kept for A/B timing: NB_SCREEN_MMA=2).
// Mapping of dune_screen_mma_kernel (clouds of up to 1024 points; see the kP template parameter): CTA = 4 warps = one item at a time; pass p, warp w: points [128 p + 32 w, +32) as two m16 tiles.
// Lane (g = lane >> 2, tq = lane & 3) holds rows g, g+8 (tile 0), g, g+8 (tile 1) -- "row slots" 0..3 = local points g + 8 r --
// and columns 8 j + 2 tq, +1 (j = 0..3) of every 32-wide activation; it OWNS local point 8 tq + g (coordinates in, key out), so
// the four row slots of a quad are exactly the points its four lanes own (one shuffle each way, no shared memory).
// LayerNorm: per-row sum of squares by a transposing quad reduction (3 shuffles: lane tq ends with the total of row slot tq),
// one MUFU.RSQ per lane, 4 shuffles to hand the four factors round.  The inputs arrive centred (host image), see ln_tanh_screen.
#pragma once
#include "dune_screen_kernel.cuh"

namespace nb {

namespace sm {

using tc::f2;

#ifndef NB_WHATIF
#define NB_WHATIF 0  // timing experiments only (wrong results): 1 = no MUFU.TANH, 2 = no HMMA, 4 = no selection, 8 = no LayerNorm scale math
#endif

constexpr int kFragBytes = 5 * 2 * 2 * 32 * 16;  // B fragments, [layer][k-step][n-tile pair][lane] uint4 = {b0,b1 (tile 2jp), b0,b1 (2jp+1)}
enum { V_W0X, V_W0Y, V_B0, V_G1, V_BE1, V_G6, V_BE6, V_G11, V_BE11, kVecs };
constexpr int kVecBytes = kVecs * 32 * 4;  // the fp32 vectors, permuted so that a lane's 8 columns are contiguous: [tq][j][h]
// the dense layers' biases as ready-made C fragments: [layer][tq][j] = {b[8j+2tq], b[8j+2tq+1], same, same} (rows g and g+8 share them),
// so that one LDS.128 delivers the aligned register quad HMMA wants (building it from a pair costs 4 moves per HMMA)
constexpr int kBiasQBytes = 5 * 4 * 4 * 16;

// D = A.B + C: the first k-step of a layer (C = the bias fragment of the lane's column pair, the same for both rows)
__device__ __forceinline__ void mma_init(f2& d01, f2& d23, const uint32_t (&a)[4], uint32_t b0, uint32_t b1, const float4& c) {
  if (NB_WHATIF & 2) {
    d01 = tc::pku(a[0] ^ b0, a[1] ^ __float_as_uint(c.x));
    d23 = tc::pku(a[2] ^ b1, a[3] ^ __float_as_uint(c.y));
    return;
  }
  asm("{\n\t.reg .f32 e0, e1, e2, e3;\n\t"
      "mma.sync.aligned.m16n8k16.row.col.f32.f16.f16.f32 {e0, e1, e2, e3}, {%2, %3, %4, %5}, {%6, %7}, {%8, %9, %10, %11};\n\t"
      "mov.b64 %0, {e0, e1};\n\tmov.b64 %1, {e2, e3};\n\t}"
      : "=l"(d01), "=l"(d23)
      : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1), "f"(c.x), "f"(c.y), "f"(c.z), "f"(c.w));
}
__device__ __forceinline__ void mma_acc(f2& d01, f2& d23, const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
  if (NB_WHATIF & 2) {
    d01 ^= tc::pku(a[0] ^ b0, a[1]);
    d23 ^= tc::pku(a[2] ^ b1, a[3]);
    return;
  }
  asm("{\n\t.reg .f32 e0, e1, e2, e3;\n\t"
      "mov.b64 {e0, e1}, %0;\n\tmov.b64 {e2, e3}, %1;\n\t"
      "mma.sync.aligned.m16n8k16.row.col.f32.f16.f16.f32 {e0, e1, e2, e3}, {%2, %3, %4, %5}, {%6, %7}, {e0, e1, e2, e3};\n\t"
      "mov.b64 %0, {e0, e1};\n\tmov.b64 %1, {e2, e3};\n\t}"
      : "+l"(d01), "+l"(d23)
      : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}

// v[r] = this lane's partial of row slot r; returns the quad total of row slot tq (lane tq of the quad)
__device__ __forceinline__ float quad_transpose_sum(const float (&v)[4], int tq) {
  const bool b0 = tq & 1, b1 = tq & 2;
  float k0 = b0 ? v[1] : v[0], s0 = b0 ? v[0] : v[1];
  float k1 = b0 ? v[3] : v[2], s1 = b0 ? v[2] : v[3];
  k0 += __shfl_xor_sync(0xffffffffu, s0, 1);
  k1 += __shfl_xor_sync(0xffffffffu, s1, 1);
  const float k = b1 ? k1 : k0, s = b1 ? k0 : k1;
  return k + __shfl_xor_sync(0xffffffffu, s, 2);
}

// LayerNorm (centred inputs, eps 1e-5, biased variance) + tanh (MUFU.TANH) on the lane's 4 row slots x 8 columns; the result is
// written as the A fragments of the next layer: a[m-tile][k-step][a0..a3]
__device__ __forceinline__ void ln_tanh_frag(const f2 (&acc)[4][4], const float* __restrict__ vg, const float* __restrict__ vb, int lane,
                                             uint32_t (&a)[2][2][4]) {
  float q[4];
#pragma unroll
  for (int r = 0; r < 4; ++r) {
    f2 s = tc::mul2(acc[r][0], acc[r][0]);
    s = tc::fma2(acc[r][1], acc[r][1], s);
    s = tc::fma2(acc[r][2], acc[r][2], s);
    s = tc::fma2(acc[r][3], acc[r][3], s);
    float lo, hi;
    tc::upk(s, lo, hi);
    q[r] = lo + hi;
  }
  const float qq = quad_transpose_sum(q, lane & 3);
  float rs;
  asm("rsqrt.approx.ftz.f32 %0, %1;" : "=f"(rs) : "f"(fmaf(qq, 1.0f / 32, 1e-5f)));
  const ulonglong2 g01 = *reinterpret_cast<const ulonglong2*>(vg), g23 = *reinterpret_cast<const ulonglong2*>(vg + 4);
  const ulonglong2 b01 = *reinterpret_cast<const ulonglong2*>(vb), b23 = *reinterpret_cast<const ulonglong2*>(vb + 4);
  const f2 gg[4] = {g01.x, g01.y, g23.x, g23.y}, bb[4] = {b01.x, b01.y, b23.x, b23.y};
#pragma unroll
  for (int r = 0; r < 4; ++r) {
    const float rr = __shfl_sync(0xffffffffu, rs, (lane & ~3) | r);
    const f2 r2 = tc::pk(rr, rr);
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      float a0, a1, t0, t1;
      if (NB_WHATIF & 8) tc::upk(tc::add2(acc[r][j], r2), a0, a1);
      else tc::upk(tc::fma2(tc::mul2(acc[r][j], r2), gg[j], bb[j]), a0, a1);
      if (NB_WHATIF & 1) { t0 = a0; t1 = a1; }
      else {
        asm("tanh.approx.f32 %0, %1;" : "=f"(t0) : "f"(a0));
        asm("tanh.approx.f32 %0, %1;" : "=f"(t1) : "f"(a1));
      }
      asm("cvt.rn.f16x2.f32 %0, %1, %2;" : "=r"(a[r >> 1][j >> 1][(j & 1) * 2 + (r & 1)]) : "f"(t1), "f"(t0));
    }
  }
}

__device__ __forceinline__ void relu_frag(const f2 (&acc)[4][4], uint32_t (&a)[2][2][4]) {
#pragma unroll
  for (int r = 0; r < 4; ++r)
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      float a0, a1;
      tc::upk(acc[r][j], a0, a1);
      asm("cvt.rn.relu.f16x2.f32 %0, %1, %2;" : "=r"(a[r >> 1][j >> 1][(j & 1) * 2 + (r & 1)]) : "f"(a1), "f"(a0));
    }
}

// one dense layer (K = 32) for both m-tiles: NT n-tiles of 8 columns; wl = the layer's fragments + lane, bq = its bias fragments + 4 tq
template <int NT>
__device__ __forceinline__ void dense_frag(const uint4* __restrict__ wl, const float4* __restrict__ bq, const uint32_t (&a)[2][2][4],
                                           f2 (&acc)[4][NT]) {
  float4 bj[NT];
#pragma unroll
  for (int j = 0; j < NT; ++j) bj[j] = bq[j];
#pragma unroll
  for (int s = 0; s < 2; ++s)
#pragma unroll
    for (int jp = 0; jp < (NT + 1) / 2; ++jp) {
      const uint4 w = wl[(s * 2 + jp) * 32];
#pragma unroll
      for (int jj = 0; jj < 2; ++jj) {
        const int j = 2 * jp + jj;
        if (j < NT) {
          const uint32_t b0 = jj ? w.z : w.x, b1 = jj ? w.w : w.y;
#pragma unroll
          for (int mt = 0; mt < 2; ++mt) {
            if (s == 0) mma_init(acc[2 * mt][j], acc[2 * mt + 1][j], a[mt][0], b0, b1, bj[j]);
            else mma_acc(acc[2 * mt][j], acc[2 * mt + 1][j], a[mt][1], b0, b1);
          }
        }
      }
    }
}

// the screen image of dune_screen_kernel (K-major UMMA layout, hi halves) re-ordered into mma.sync B fragments, the permuted fp32
// vectors and the bias fragments, by the 128 threads of a CTA
__device__ __forceinline__ void stage_operands(const unsigned char* __restrict__ image, unsigned char* smem_dyn, int tid) {
  using I = TcImage;
  uint4* wfrag = reinterpret_cast<uint4*>(smem_dyn);
  float* vec = reinterpret_cast<float*>(smem_dyn + kFragBytes);
  float4* biasq = reinterpret_cast<float4*>(smem_dyn + kFragBytes + kVecBytes);
  uint32_t* wf = reinterpret_cast<uint32_t*>(wfrag);
  for (int x = tid; x < kFragBytes / 4; x += 128) {
    const int c = x & 3, ln = (x >> 2) & 31, jp = (x >> 7) & 1, s = (x >> 8) & 1, l = x >> 9;
    const int n = 8 * (2 * jp + (c >> 1)) + (ln >> 2), k = 16 * s + 2 * (ln & 3) + 8 * (c & 1);
    const size_t off = (size_t)l * I::kLayerStride + (size_t)(k / 16) * 1024 + ((k % 16) / 8) * 512 + (n / 8) * 128 + (n % 8) * 16 + (k % 8) * 2;
    wf[x] = *reinterpret_cast<const uint32_t*>(image + off);
  }
  const float* fl = reinterpret_cast<const float*>(image + I::kFloatOff);
  for (int x = tid; x < kVecs * 32; x += 128) {
    const int v = x >> 5, e = x & 31, q = e >> 3, j = (e >> 1) & 3, h = e & 1;
    const int src = v == V_W0X ? I::W0X : v == V_W0Y ? I::W0Y : v == V_B0 ? I::B0 : I::G1 + 32 * (v - V_G1);
    vec[x] = fl[src + 8 * j + 2 * q + h];
  }
  for (int x = tid; x < 5 * 4 * 4; x += 128) {  // [layer][tq][j]
    const int l = x >> 4, q = (x >> 2) & 3, j = x & 3;
    const float bx = fl[I::BH + 32 * l + 8 * j + 2 * q], by = fl[I::BH + 32 * l + 8 * j + 2 * q + 1];
    biasq[x] = make_float4(bx, by, bx, by);
  }
}

// smallest value above k whose low kIdxBits bits carry the point's index: keys become unique (a REDUX round removes exactly one entry);
// rounding an upper bound UP only widens the candidate set
template <int kIdxBits>
__device__ __forceinline__ uint32_t unique_key(uint32_t k, int idx) {
  constexpr uint32_t kIdxMask = (1u << kIdxBits) - 1u;
  return ((min(k, 0xFFFFF000u) + (kIdxMask + 1u)) & ~kIdxMask) | (uint32_t)idx;
}

// geometry rows of the lane's two head channels 2 tq, 2 tq + 1 (zero beyond E: their partial distance is 0)
struct HeadGeo {
  float gx0, gy0, h0, gx1, gy1, h1;
};
__device__ __forceinline__ HeadGeo head_geo(const DuneParams& prm, int tq) {
  const int e0 = 2 * tq, e1 = 2 * tq + 1, E = prm.geo.E;
  HeadGeo hg;
  hg.gx0 = e0 < E ? prm.geo.G[e0][0] : 0.f; hg.gy0 = e0 < E ? prm.geo.G[e0][1] : 0.f; hg.h0 = e0 < E ? prm.geo.h[e0] : 0.f;
  hg.gx1 = e1 < E ? prm.geo.G[e1][0] : 0.f; hg.gy1 = e1 < E ? prm.geo.G[e1][1] : 0.f; hg.h1 = e1 < E ? prm.geo.h[e1] : 0.f;
  return hg;
}

// one warp's 32 points through the screening network: (x0, y0) = the lane's own point in the robot frame (zeros for rows beyond n);
// returns its screened distance d~ and error radius eps.  vq / wl / bqq: the lane's views of the staged operands.
__device__ __forceinline__ void screen_point(const DuneParams& prm, const HeadGeo& hg, const float* __restrict__ vq, const uint4* __restrict__ wl,
                                             const float4* __restrict__ bqq, int lane, float x0, float y0, float& d, float& eps) {
  const int tq = lane & 3;
  float xr[4], yr[4];
#pragma unroll
  for (int r = 0; r < 4; ++r) {
    xr[r] = __shfl_sync(0xffffffffu, x0, (lane & ~3) | r);
    yr[r] = __shfl_sync(0xffffffffu, y0, (lane & ~3) | r);
  }
  f2 acc[4][4];
  uint32_t a[2][2][4];
  {  // layer 0 (2 -> 32) on the FMA pipe, directly in accumulator layout
    const ulonglong2 wx01 = *reinterpret_cast<const ulonglong2*>(vq + 32 * V_W0X), wx23 = *reinterpret_cast<const ulonglong2*>(vq + 32 * V_W0X + 4);
    const ulonglong2 wy01 = *reinterpret_cast<const ulonglong2*>(vq + 32 * V_W0Y), wy23 = *reinterpret_cast<const ulonglong2*>(vq + 32 * V_W0Y + 4);
    const ulonglong2 b01 = *reinterpret_cast<const ulonglong2*>(vq + 32 * V_B0), b23 = *reinterpret_cast<const ulonglong2*>(vq + 32 * V_B0 + 4);
    const f2 wx[4] = {wx01.x, wx01.y, wx23.x, wx23.y}, wy[4] = {wy01.x, wy01.y, wy23.x, wy23.y}, bb[4] = {b01.x, b01.y, b23.x, b23.y};
#pragma unroll
    for (int r = 0; r < 4; ++r) {
      const f2 x2 = tc::pk(xr[r], xr[r]), y2 = tc::pk(yr[r], yr[r]);
#pragma unroll
      for (int j = 0; j < 4; ++j) acc[r][j] = tc::fma2(wy[j], y2, tc::fma2(wx[j], x2, bb[j]));
    }
  }
  ln_tanh_frag(acc, vq + 32 * V_G1, vq + 32 * V_BE1, lane, a);
  dense_frag<4>(wl + 0 * 128, bqq + 16 * 0, a, acc);
  relu_frag(acc, a);
  dense_frag<4>(wl + 1 * 128, bqq + 16 * 1, a, acc);
  ln_tanh_frag(acc, vq + 32 * V_G6, vq + 32 * V_BE6, lane, a);
  dense_frag<4>(wl + 2 * 128, bqq + 16 * 2, a, acc);
  relu_frag(acc, a);
  dense_frag<4>(wl + 3 * 128, bqq + 16 * 3, a, acc);
  ln_tanh_frag(acc, vq + 32 * V_G11, vq + 32 * V_BE11, lane, a);
  f2 mu[4][1];
  dense_frag<1>(wl + 4 * 128, bqq + 16 * 4, a, mu);

  // head: d~ = relu(mu)^T (G p0 - h): partial over the lane's two channels for each row slot, transposing quad reduction
  float dp[4];
#pragma unroll
  for (int r = 0; r < 4; ++r) {
    float m0, m1;
    tc::upk(mu[r][0], m0, m1);
    const float ge0 = fmaf(hg.gy0, yr[r], hg.gx0 * xr[r]) - hg.h0, ge1 = fmaf(hg.gy1, yr[r], hg.gx1 * xr[r]) - hg.h1;
    dp[r] = fmaf(fmaxf(m1, 0.f), ge1, fmaxf(m0, 0.f) * ge0);
  }
  d = quad_transpose_sum(dp, tq);  // the lane's own point
  float sa = 0.f;
#pragma unroll
  for (int e = 0; e < kMaxEdges; ++e)
    if (e < prm.geo.E) sa += fabsf(fmaf(prm.geo.G[e][1], y0, prm.geo.G[e][0] * x0) - prm.geo.h[e]);
  eps = fmaf(prm.c_mu, sa, 1e-4f);
}

}  // namespace sm

// shared memory: B fragments | permuted vectors | bias fragments | raw points of the item in flight (x | y | vx | vy, N floats each) |
// per-warp upper-bound candidates (4 M x 4)
__host__ __device__ inline size_t dune_screen_mma_smem_bytes(int N, int M) {
  return (size_t)sm::kFragBytes + sm::kVecBytes + sm::kBiasQBytes + (size_t)N * 16 + (size_t)4 * M * 4 + 64;
}

#ifndef NB_SMMA_BLOCKS
#define NB_SMMA_BLOCKS 5  // CTAs per SM the register allocation is made for: 96 registers, 12 B of spills (4: 21.57, 5: 21.37, 6: 21.81 ms per C4 step)
#endif
// kP = the most 128-point passes an item can need: every thread keeps the bounds of its <= kP points in registers, with the point's
// index in the low kIdxBits bits of the key.  kP = 4: N <= 512 (96 registers, 5 CTAs per SM); kP = 8: N <= 1024 (4 CTAs per SM).  The
// launcher sends larger clouds to dune_screen_kernel, whose shared-memory key arrays have no such limit.
template <int kP>
__global__ void __launch_bounds__(128, kP <= 4 ? NB_SMMA_BLOCKS : 4) dune_screen_mma_kernel(const DuneParams prm, const unsigned char* __restrict__ image) {
  extern __shared__ __align__(1024) unsigned char smem_dyn[];
  uint4* wfrag = reinterpret_cast<uint4*>(smem_dyn);
  float* vec = reinterpret_cast<float*>(smem_dyn + sm::kFragBytes);
  float4* biasq = reinterpret_cast<float4*>(smem_dyn + sm::kFragBytes + sm::kVecBytes);
  float* raw = reinterpret_cast<float*>(smem_dyn + sm::kFragBytes + sm::kVecBytes + sm::kBiasQBytes);
  uint32_t* c32 = reinterpret_cast<uint32_t*>(raw + (size_t)4 * prm.N);
  __shared__ int cnt_s[2];
  __shared__ int list_s[kCandMax];
  __shared__ float ldt_s[kCandMax];

  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, g = lane >> 2, tq = lane & 3;
  sm::stage_operands(image, smem_dyn, tid);
  if (tid < 2) cnt_s[tid] = 0;
  __syncthreads();
  const uint4* wl = wfrag + lane;
  const float* vq = vec + 8 * tq;
  const float4* bqq = biasq + 4 * tq;

  const int T1 = prm.T + 1, N = prm.N, M = prm.M;
  const int items = prm.B * T1;
  const sm::HeadGeo hg = sm::head_geo(prm, tq);
  const int own0 = 32 * warp + 8 * tq + g;  // the lane's point in pass 0 (pass p: + 128 p)
  constexpr int kIdxBits = kP <= 4 ? 9 : 10;
  constexpr uint32_t kIdxMask = (1u << kIdxBits) - 1u;

  // The raw point data of an item are copied asynchronously (cp.async, each thread exactly the <= 4 entries it reads itself: no
  // barrier) -- for the NEXT item as soon as this thread has read its last point of the current one.
  int staged = -1;
  auto stage_points = [&](int it) -> bool {
    const int bb = it / T1;
    if (prm.skip_t0 && it == bb * T1) return false;
    int nn = prm.num_points ? prm.num_points[bb] : N;
    nn = nn > N ? N : nn;
    if ((nn <= kCandMax && !prm.calibrate) || nn <= 0) return false;
    const float* px = prm.points + (size_t)bb * 2 * N;
    const float* vx = prm.velocities ? prm.velocities + (size_t)bb * 2 * N : nullptr;
#pragma unroll
    for (int j = 0; j < kP; ++j) {
      const int i = own0 + 128 * j;
      if (i < nn) {
        tc::cp_async4(raw + i, px + i);
        tc::cp_async4(raw + N + i, px + N + i);
        if (vx) {
          tc::cp_async4(raw + 2 * N + i, vx + i);
          tc::cp_async4(raw + 3 * N + i, vx + N + i);
        }
      }
    }
    return true;
  };

  int par = 0;  // which of the two candidate counters this item uses (the other one is reset meanwhile)
  for (int item = blockIdx.x; item < items; item += gridDim.x) {
    const int b = item / T1, t = item - b * T1;
    if (prm.skip_t0 && t == 0) {  // same inputs as in the previous PAN iteration: its outputs stand
      if (tid == 0) prm.cand_cnt[item] = 0;
      continue;
    }
    int32_t* out_idx = prm.cand_idx + (size_t)item * kCandMax;
    float* out_dt = prm.cand_dt + (size_t)item * kCandMax;
    const int act = prm.active ? prm.active[b] : 1;
    int n = prm.num_points ? prm.num_points[b] : N;
    const tc::ItemFrame fr = tc::item_frame(prm, b, t);
    if (act == 0) {
      if (tid == 0) prm.cand_cnt[item] = 0;
      continue;
    }
    n = n < 0 ? 0 : (n > N ? N : n);
    const int cnt = n < M ? n : M;
    if (t == 0 && tid == 0) {
      prm.sel_count[b] = cnt;
      if (n == 0 && prm.min_dist) prm.min_dist[b] = __int_as_float(0x7f800000);
    }
    if (n <= kCandMax && !prm.calibrate) {  // nothing to screen: every point is a candidate
      if (tid < n) { out_idx[tid] = tid; out_dt[tid] = __int_as_float(0x7fc00000); }
      if (tid == 0) { prm.cand_cnt[item] = n; tc::refine_append(prm, item, n); }
      continue;
    }
    if (staged != item) {
      tc::cp_async_wait_all();  // an abandoned copy (its item was skipped) must not land after this one
      stage_points(item);
      staged = item;
    }
    tc::cp_async_wait_all();
    // the bounds of the thread's points: a shift register (newest first); the point's index rides in the low 9 bits of the key
    uint32_t kk[kP];
    float ll[kP], dd[kP];
#pragma unroll
    for (int j = 0; j < kP; ++j) { kk[j] = 0xFFFFFFFFu; ll[j] = 0.f; dd[j] = 0.f; }

#pragma unroll 1
    for (int base = 32 * warp; base < n; base += 128) {  // this warp's 32-point tiles
      const int i = base + 8 * tq + g;
      float x0 = 0.f, y0 = 0.f;
      if (i < n) {  // rows beyond n run on zeros (their results are never looked at)
        float gx = raw[i], gy = raw[N + i];
        if (fr.vx) {
          gx = flow(gx, raw[2 * N + i], fr.dt, fr.t);
          gy = flow(gy, raw[3 * N + i], fr.dt, fr.t);
        }
        const float dx = gx - fr.sx, dy = gy - fr.sy;
        x0 = fmaf(fr.cs, dx, fr.sn * dy);
        y0 = fmaf(fr.cs, dy, -(fr.sn * dx));
      }
      float d, eps;
      sm::screen_point(prm, hg, vq, wl, bqq, lane, x0, y0, d, eps);
#pragma unroll
      for (int j = kP - 1; j > 0; --j) { kk[j] = kk[j - 1]; ll[j] = ll[j - 1]; dd[j] = dd[j - 1]; }
      kk[0] = i < n ? sm::unique_key<kIdxBits>(orderable(d + eps), i) : 0xFFFFFFFFu;
      ll[0] = d - eps; dd[0] = d;
    }
    if (item + (int)gridDim.x < items) {  // this thread is done with `raw`: its part of the next item
      if (stage_points(item + (int)gridDim.x)) staged = item + (int)gridDim.x;
    }
    if (NB_WHATIF & 4) {
      if (tid == 0) prm.cand_cnt[item] = (kk[0] ^ kk[kP - 1]) == 12345u ? (int)(ll[0] + ll[kP - 1] + dd[0] + dd[kP - 1]) : 0;
      continue;
    }
    if (n <= kCandMax) {  // calibration mode: all points (they belong to warp 0's only tile), with their screened distance
      if (kk[0] != 0xFFFFFFFFu) { out_idx[kk[0] & kIdxMask] = (int)(kk[0] & kIdxMask); out_dt[kk[0] & kIdxMask] = dd[0]; }
      if (tid == 0) { prm.cand_cnt[item] = n; tc::refine_append(prm, item, n); }
      continue;
    }
    // ---- tau = the M-th smallest upper bound: unique 32-bit keys, M REDUX rounds per warp (each removes the one entry that equals
    // the minimum), then every warp merges the 4 M survivors the same way.  Two block barriers per item: the per-warp lists, and
    // the candidate list; the candidate counter alternates between two words so that resetting it needs no third one.
    {
      uint32_t q[kP];
#pragma unroll
      for (int j = 0; j < kP; ++j) q[j] = kk[j];
      for (int m = 0; m < M; ++m) {
        uint32_t mine = q[0];
#pragma unroll
        for (int j = 1; j < kP; ++j) mine = min(mine, q[j]);
        const uint32_t md = __reduce_min_sync(0xffffffffu, mine);
#pragma unroll
        for (int j = 0; j < kP; ++j) q[j] = q[j] == md ? 0xFFFFFFFFu : q[j];
        if (lane == 0) c32[warp * M + m] = md;
      }
    }
    __syncthreads();
    uint32_t tau = 0xFFFFFFFFu;
    {
      const int nc4 = 4 * M;  // <= 128 (M <= 32)
      uint32_t q0 = lane < nc4 ? c32[lane] : 0xFFFFFFFFu;
      uint32_t q1 = lane + 32 < nc4 ? c32[lane + 32] : 0xFFFFFFFFu;
      uint32_t q2 = lane + 64 < nc4 ? c32[lane + 64] : 0xFFFFFFFFu;
      uint32_t q3 = lane + 96 < nc4 ? c32[lane + 96] : 0xFFFFFFFFu;
      for (int m = 0; m < M; ++m) {  // n > kCandMax >= M: M finite keys exist
        tau = __reduce_min_sync(0xffffffffu, min(min(q0, q1), min(q2, q3)));
        q0 = q0 == tau ? 0xFFFFFFFFu : q0; q1 = q1 == tau ? 0xFFFFFFFFu : q1;
        q2 = q2 == tau ? 0xFFFFFFFFu : q2; q3 = q3 == tau ? 0xFFFFFFFFu : q3;
      }
    }
    auto take = [&](uint32_t k, float lb, float dt) {
      if (k != 0xFFFFFFFFu && orderable(lb) <= tau) {
        const int pos = atomicAdd(&cnt_s[par], 1);
        if (pos < kCandMax) { list_s[pos] = (int)(k & kIdxMask); ldt_s[pos] = dt; }
      }
    };
#pragma unroll
    for (int j = 0; j < kP; ++j) take(kk[j], ll[j], dd[j]);
    __syncthreads();
    const int nc = cnt_s[par];
    if (nc <= kCandMax) {
      if (tid < nc) { out_idx[tid] = list_s[tid]; out_dt[tid] = ldt_s[tid]; }
      if (tid == 0) {
        prm.cand_cnt[item] = nc;
        tc::refine_append(prm, item, nc);
        atomicAdd(&prm.screen_stats[2], (unsigned)nc);
        atomicAdd(&prm.screen_stats[3], 1u);
      }
    } else if (tid == 0) {
      prm.cand_cnt[item] = -1;  // too many candidates: the exact kernel evaluates this item in full
      atomicAdd(&prm.screen_stats[1], 1u);
      prm.flag_list[atomicAdd(prm.flag_count, 1)] = item;
    }
    // every thread has passed this item's first barrier, hence finished reading the OTHER counter (the previous item's) long ago
    if (tid == 0) cnt_s[par ^ 1] = 0;
    par ^= 1;
  }
  tc::cp_async_wait_all();
}


// ---- The default shape: one warp per (environment, step) item.
//
// dune_screen_mma_kernel above spreads an item over the 4 warps of a CTA, and every warp pays an item skeleton of its own: the
// accurate cos / sin of the item frame, cp.async staging, M REDUX rounds over its keys and M more to merge the 4 M survivors, a
// shared-memory candidate counter and two block barriers -- 856 of the 3,852 instructions a warp spends on an item at N = 500.  Here
// one warp takes an item from its frame to its candidate list and shares nothing with the other warps but the staged operands:
//  * per 32-point tile: the same network, keys and bounds (sm::screen_point, sm::unique_key), hence the same tau and the same
//    candidate set; only the order of the list differs (the refine kernel ranks candidates by (distance, index));
//  * points: the lane's point of the NEXT tile is loaded into registers while the current tile runs (plain loads: the T + 1 items of
//    an environment read the same points, mostly from L2);
//  * d~ and eps of the lane's point of every tile go to the warp's slab in shared memory, written and read by that lane only (no
//    barrier); after the last tile the network's registers are free, the <= 4 kP keys of the lane are rebuilt there and M REDUX rounds
//    over them give tau -- no merge;
//  * the candidate list is compacted with __ballot_sync and a __popc prefix and written straight to global memory;
//  * items are handed out by a counter (flag_count[3], zeroed by the launcher with the other three words), the next ticket requested
//    while the current item runs: at ~7 items per warp and launch a static stride leaves a tail of up to one item.
// The only block barrier is the one after the operand staging.

// shared memory: B fragments | permuted vectors | bias fragments | per warp: d~ and eps of its item (N rounded up to 32, 4 B each)
__host__ __device__ inline size_t dune_screen_warp_smem_bytes(int N) {
  return (size_t)sm::kFragBytes + sm::kVecBytes + sm::kBiasQBytes + (size_t)4 * 2 * ((N + 31) / 32 * 32) * 4;
}

// kP: as above (N <= 128 kP): the lane rebuilds its <= 4 kP keys in registers for the selection
template <int kP>
__global__ void __launch_bounds__(128, kP <= 4 ? NB_SMMA_BLOCKS : 4) dune_screen_warp_kernel(const DuneParams prm, const unsigned char* __restrict__ image) {
  extern __shared__ __align__(1024) unsigned char smem_dyn[];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, tq = lane & 3;
  const int T1 = prm.T + 1, N = prm.N, M = prm.M;
  sm::stage_operands(image, smem_dyn, tid);
  if (prm.skip_t0)  // step-0 items are not handed out below: same inputs as in the previous PAN iteration, its outputs stand
    for (int b = blockIdx.x * 128 + tid; b < prm.B; b += gridDim.x * 128) prm.cand_cnt[(size_t)b * T1] = 0;
  __syncthreads();
  const uint4* wl = reinterpret_cast<const uint4*>(smem_dyn) + lane;
  const float* vq = reinterpret_cast<const float*>(smem_dyn + sm::kFragBytes) + 8 * tq;
  const float4* bqq = reinterpret_cast<const float4*>(smem_dyn + sm::kFragBytes + sm::kVecBytes) + 4 * tq;
  const int np = (N + 31) & ~31;
  float* sd = reinterpret_cast<float*>(smem_dyn + sm::kFragBytes + sm::kVecBytes + sm::kBiasQBytes) + (size_t)warp * 2 * np;  // [tile][lane]
  float* se = sd + np;
  const sm::HeadGeo hg = sm::head_geo(prm, tq);
  const int own = 8 * tq + (lane >> 2);  // the lane's point in a tile
  constexpr int kIdxBits = kP <= 4 ? 9 : 10;
  constexpr int kTiles = 4 * kP;
  const unsigned lanes_below = (1u << lane) - 1u;

  auto run_item = [&](int b, int t) {
    const int item = b * T1 + t;
    int32_t* out_idx = prm.cand_idx + (size_t)item * kCandMax;
    float* out_dt = prm.cand_dt + (size_t)item * kCandMax;
    const int act = prm.active ? prm.active[b] : 1;
    if (act == 0) {
      if (lane == 0) prm.cand_cnt[item] = 0;
      return;
    }
    int n = prm.num_points ? prm.num_points[b] : N;
    n = n < 0 ? 0 : (n > N ? N : n);
    if (t == 0 && lane == 0) {
      prm.sel_count[b] = n < M ? n : M;
      if (n == 0 && prm.min_dist) prm.min_dist[b] = __int_as_float(0x7f800000);
    }
    if (n <= kCandMax && !prm.calibrate) {  // nothing to screen: every point is a candidate
      if (lane < n) { out_idx[lane] = lane; out_dt[lane] = __int_as_float(0x7fc00000); }
      if (lane == 0) { prm.cand_cnt[item] = n; tc::refine_append(prm, item, n); }
      return;
    }
    const tc::ItemFrame fr = tc::item_frame(prm, b, t);
    const int tiles = (n + 31) >> 5;
    float px = 0.f, py = 0.f, pvx = 0.f, pvy = 0.f;  // the lane's point of the next tile
    auto fetch = [&](int i) {
      if (i < n) {
        px = fr.px[i]; py = fr.py[i];
        if (fr.vx) { pvx = fr.vx[i]; pvy = fr.vy[i]; }
      }
    };
    fetch(own);
#pragma unroll 1
    for (int tile = 0; tile < tiles; ++tile) {
      const int i = 32 * tile + own;
      float gx = px, gy = py;
      const float vx = pvx, vy = pvy;
      fetch(i + 32);
      float x0 = 0.f, y0 = 0.f;
      if (i < n) {  // rows beyond n run on zeros (their results are never looked at)
        if (fr.vx) {
          gx = flow(gx, vx, fr.dt, fr.t);
          gy = flow(gy, vy, fr.dt, fr.t);
        }
        const float dx = gx - fr.sx, dy = gy - fr.sy;
        x0 = fmaf(fr.cs, dx, fr.sn * dy);
        y0 = fmaf(fr.cs, dy, -(fr.sn * dx));
      }
      float d, eps;
      sm::screen_point(prm, hg, vq, wl, bqq, lane, x0, y0, d, eps);
      sd[32 * tile + lane] = d;
      se[32 * tile + lane] = eps;
    }
    if (n <= kCandMax) {  // calibration mode: all points (one tile), with their screened distance
      if (own < n) { out_idx[own] = own; out_dt[own] = sd[lane]; }
      if (lane == 0) { prm.cand_cnt[item] = n; tc::refine_append(prm, item, n); }
      return;
    }
    // tau = the M-th smallest upper bound: the keys are unique, so each REDUX round removes exactly one of them (n > kCandMax >= M:
    // M finite keys exist)
    uint32_t q[kTiles];
#pragma unroll
    for (int j = 0; j < kTiles; ++j) {
      const int i = 32 * j + own;
      q[j] = i < n ? sm::unique_key<kIdxBits>(orderable(sd[32 * j + lane] + se[32 * j + lane]), i) : 0xFFFFFFFFu;
    }
    uint32_t tau;
    for (int m = 0;; ++m) {
      uint32_t mine = q[0];
#pragma unroll
      for (int j = 1; j < kTiles; ++j) mine = min(mine, q[j]);
      tau = __reduce_min_sync(0xffffffffu, mine);
      if (m == M - 1) break;
#pragma unroll
      for (int j = 0; j < kTiles; ++j) q[j] = q[j] == tau ? 0xFFFFFFFFu : q[j];
    }
    // candidates: lower bound <= tau, in (tile, lane) order
    int nc = 0;
#pragma unroll
    for (int j = 0; j < kTiles; ++j) {
      if (32 * j < n) {  // warp-uniform
        const int i = 32 * j + own;
        const float d = sd[32 * j + lane];
        const bool take = i < n && orderable(d - se[32 * j + lane]) <= tau;
        const unsigned bal = __ballot_sync(0xffffffffu, take);
        const int pos = nc + __popc(bal & lanes_below);
        if (take && pos < kCandMax) { out_idx[pos] = i; out_dt[pos] = d; }
        nc += __popc(bal);
      }
    }
    if (lane == 0) {
      if (nc <= kCandMax) {
        prm.cand_cnt[item] = nc;
        tc::refine_append(prm, item, nc);
        atomicAdd(&prm.screen_stats[2], (unsigned)nc);
        atomicAdd(&prm.screen_stats[3], 1u);
      } else {
        prm.cand_cnt[item] = -1;  // too many candidates: the exact kernel evaluates this item in full
        atomicAdd(&prm.screen_stats[1], 1u);
        prm.flag_list[atomicAdd(prm.flag_count, 1)] = item;
      }
    }
  };

  const int steps = prm.skip_t0 ? prm.T : T1;  // items handed out per environment (t = 1..T with skip_t0)
  const int work = prm.B * steps;
  int* const counter = prm.flag_count + 3;
  int w = 0;
  if (lane == 0) w = atomicAdd(counter, 1);
  w = __shfl_sync(0xffffffffu, w, 0);
  while (w < work) {
    int next = 0;
    if (lane == 0) next = atomicAdd(counter, 1);
    const int b = w / steps;
    run_item(b, w - b * steps + (prm.skip_t0 ? 1 : 0));
    w = __shfl_sync(0xffffffffu, next, 0);
  }
}

}  // namespace nb
