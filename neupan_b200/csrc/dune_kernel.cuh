// DUNE kernel: point flow -> robot frame -> ObsPointNet -> distance -> M closest points.
//
// Replaces, for a whole batch of environments and all T+1 horizon steps in ONE launch:
//   PAN.generate_point_flow / point_state_transform   neupan/blocks/pan.py:150-212
//   ObsPointNet.forward                                neupan/blocks/obs_point_net.py:31-49
//   DUNE.forward / cal_objective_distance              neupan/blocks/dune.py:58-127
// Only the first M = nrmp_max_num sorted columns are ever consumed downstream
// (nrmp.py:136-138,254-256; pan.py:234-237), so the full argsort of dune.py:100 is replaced by a
// deterministic top-M selection (ascending distance, ties -> lower point index).
//
// Work item = one (environment b, horizon step t): N points.  Persistent CTAs stride over the
// B*(T+1) items; the 18.6 KB of MLP weights are staged into shared memory once per CTA and read
// with warp-broadcast LDS.128; each thread carries P points through the six layers in registers
// (FP32 FFMA, LayerNorm and tanh in registers, no intermediate ever touches HBM).  Per item the
// kernel writes only M*(E+5) floats.
#pragma once
#include "common.cuh"

namespace nb {

struct DuneParams {
  const float* weights;       // packed checkpoint (device)
  const float* nom_s;         // (B,3,T+1)
  const float* points;        // (B,2,N)
  const float* velocities;    // (B,2,N) or nullptr
  const int32_t* num_points;  // (B) or nullptr
  const int32_t* active;      // (B) or nullptr: env skipped when 0
  float* sel_mu;              // (B,T+1,M,E)
  float* sel_lam;             // (B,T+1,M,2)
  float* sel_pts;             // (B,T+1,M,2)
  float* sel_dist;            // (B,T+1,M)
  int32_t* sel_count;         // (B)
  float* min_dist;            // (B) or nullptr
  int B, N, T, M;
  float dt;
  Geometry geo;
  // screening (NB_OPT_DUNE_KERNEL = 4, dune_screen_kernel.cuh): candidate lists written by dune_screen_kernel, consumed by
  // dune_refine_kernel; all nullptr / 0 in the other variants
  int32_t* cand_idx;        // (B (T+1), 32) point indices
  int32_t* cand_cnt;        // (B (T+1)): candidates of the item; -1 = evaluate the item exactly; 0 = nothing to do
  float* cand_dt;           // (B (T+1), 32) screened distance of each candidate (NaN: not screened) -- statistics only
  unsigned* screen_stats;   // [0] max |d~ - d| / sum|t| over candidates (float bits), [1] items sent to the exact kernel, [2] candidates, [3] items screened
  float c_mu;               // bound on |mu~_e - mu_e| of the screening network
  int32_t* flag_list;       // (B (T+1)) the items with cand_cnt == -1, in the order the screen kernel met them
  int32_t* flag_count;      // (4) [0] their number, [1] / [2] the lengths of the two refine lists, [3] the item counter of dune_screen_warp_kernel;
                            // zeroed by the launcher before the screen kernel
  int32_t* refine_list;     // (2 B (T+1)) work lists of dune_refine_kernel, appended by the screen kernels: [0, B (T+1)) the items with 1..16
                            // candidates (two of them share a warp), [B (T+1), 2 B (T+1)) those with 17..32 (one warp each)
  int only_flagged;         // exact kernel: process only the items of flag_list
  int skip_t0;              // screen kernels: step-0 items are skipped (cand_cnt = 0) and keep the outputs of the previous launch -- set by
                            // nb_pan_forward for PAN iterations k > 0: nom_s[:, 0] is the fixed initial state (robot.py:234; the NRMP kernel
                            // copies the column bit for bit), so item (b, 0) has the same inputs and the same result in every iteration
  int screen_mma;           // launcher hint (NB_OPT_DUNE_SCREEN_MMA): screening pass on mma.sync (dune_screen_mma_kernel.cuh) where N <= 1024,
                            // 1 = one warp per item (dune_screen_warp_kernel) if the launch has an item per resident warp, else one CTA per
                            // item (dune_screen_mma_kernel); 2 / 3 = always the CTA / warp shape; 0 = tcgen05
  int calibrate;            // screen kernel: items with N <= 32 are NOT short-cut: all their points become candidates with their screened
                            // distance, so that the refine kernel's statistics compare the two networks on every point (nb_pan calibration)
};

__device__ __forceinline__ uint32_t orderable(float d) {
  if (d != d) return 0xFFFFFFFFu;  // NaN sorts last
  uint32_t u = __float_as_uint(d);
  return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}

template <int P>
__device__ __forceinline__ void layernorm_tanh(float (&v)[P][kHidden], const float* __restrict__ g, const float* __restrict__ be) {
#pragma unroll
  for (int p = 0; p < P; ++p) {
    float s = 0.f;
#pragma unroll
    for (int j = 0; j < kHidden; ++j) s += v[p][j];
    const float mean = s * (1.0f / kHidden);
    float q = 0.f;
#pragma unroll
    for (int j = 0; j < kHidden; ++j) {
      const float d = v[p][j] - mean;
      q = fmaf(d, d, q);
    }
    const float rstd = 1.0f / sqrtf(q * (1.0f / kHidden) + 1e-5f);  // nn.LayerNorm eps, biased variance
#pragma unroll
    for (int j = 0; j < kHidden; ++j) v[p][j] = tanhf(fmaf((v[p][j] - mean) * rstd, g[j], be[j]));
  }
}

// out[p][j] = act(b[j] + sum_k W[j][k] * in[p][k]); W row-major (out, in) in shared memory.
template <int P, bool RELU>
__device__ __forceinline__ void dense32(const float* __restrict__ W, const float* __restrict__ b,
                                        const float (&in)[P][kHidden], float (&out)[P][kHidden]) {
#pragma unroll
  for (int j = 0; j < kHidden; ++j) {
    float acc[P];
#pragma unroll
    for (int p = 0; p < P; ++p) acc[p] = b[j];
#pragma unroll
    for (int k4 = 0; k4 < kHidden / 4; ++k4) {
      const float4 w = reinterpret_cast<const float4*>(W + j * kHidden)[k4];
#pragma unroll
      for (int p = 0; p < P; ++p) {
        acc[p] = fmaf(w.x, in[p][4 * k4 + 0], acc[p]);
        acc[p] = fmaf(w.y, in[p][4 * k4 + 1], acc[p]);
        acc[p] = fmaf(w.z, in[p][4 * k4 + 2], acc[p]);
        acc[p] = fmaf(w.w, in[p][4 * k4 + 3], acc[p]);
      }
    }
#pragma unroll
    for (int p = 0; p < P; ++p) out[p][j] = RELU ? fmaxf(acc[p], 0.f) : acc[p];
  }
}

template <int E, int P>
__device__ __forceinline__ void obs_point_net(const float* __restrict__ sw, const float (&x)[P], const float (&y)[P], float (&mu)[P][E]) {
  using L = WeightLayout;
  float a[P][kHidden], c[P][kHidden];
#pragma unroll
  for (int j = 0; j < kHidden; ++j) {
    const float w0 = sw[L::W0 + 2 * j], w1 = sw[L::W0 + 2 * j + 1], bj = sw[L::B0 + j];
#pragma unroll
    for (int p = 0; p < P; ++p) a[p][j] = fmaf(w1, y[p], fmaf(w0, x[p], bj));
  }
  layernorm_tanh<P>(a, sw + L::G1, sw + L::BE1);
  dense32<P, true>(sw + L::W3, sw + L::B3, a, c);
  dense32<P, false>(sw + L::W5, sw + L::B5, c, a);
  layernorm_tanh<P>(a, sw + L::G6, sw + L::BE6);
  dense32<P, true>(sw + L::W8, sw + L::B8, a, c);
  dense32<P, false>(sw + L::W10, sw + L::B10, c, a);
  layernorm_tanh<P>(a, sw + L::G11, sw + L::BE11);
#pragma unroll
  for (int e = 0; e < E; ++e) {
    float acc[P];
#pragma unroll
    for (int p = 0; p < P; ++p) acc[p] = sw[L::b13(E) + e];
#pragma unroll
    for (int k4 = 0; k4 < kHidden / 4; ++k4) {
      const float4 w = reinterpret_cast<const float4*>(sw + L::W13 + e * kHidden)[k4];
#pragma unroll
      for (int p = 0; p < P; ++p) {
        acc[p] = fmaf(w.x, a[p][4 * k4 + 0], acc[p]);
        acc[p] = fmaf(w.y, a[p][4 * k4 + 1], acc[p]);
        acc[p] = fmaf(w.z, a[p][4 * k4 + 2], acc[p]);
        acc[p] = fmaf(w.w, a[p][4 * k4 + 3], acc[p]);
      }
    }
#pragma unroll
    for (int p = 0; p < P; ++p) mu[p][e] = fmaxf(acc[p], 0.f);
  }
}

// p_t = p + t*(v*dt) with the reference's rounding sequence (pan.py:182), no FMA contraction
__device__ __forceinline__ float flow(float p, float v, float dt, int t) {
  return __fadd_rn(p, __fmul_rn((float)t, __fmul_rn(v, dt)));
}

constexpr int kDuneMaxWarps = 8;

// dynamic shared memory: [weights | keys (N x u64) | mu (N x E)]
template <int E>
__host__ __device__ inline size_t dune_smem_bytes(int N) {
  size_t w = ((size_t)WeightLayout::count(E) * 4 + 15) / 16 * 16;
  return w + (size_t)N * 8 + (size_t)N * E * 4;
}

template <int E, int P, int THREADS>
__global__ void __launch_bounds__(THREADS, 1) dune_kernel(const DuneParams prm) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  constexpr int NW = THREADS / 32;
  float* sw = reinterpret_cast<float*>(smem_raw);
  const size_t w_bytes = ((size_t)WeightLayout::count(E) * 4 + 15) / 16 * 16;
  unsigned long long* keys = reinterpret_cast<unsigned long long*>(smem_raw + w_bytes);
  float* smu = reinterpret_cast<float*>(smem_raw + w_bytes + (size_t)prm.N * 8);
  __shared__ unsigned long long warp_min[2][kDuneMaxWarps];

  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  for (int i = tid; i < WeightLayout::count(E); i += THREADS) sw[i] = prm.weights[i];
  __syncthreads();

  const int T1 = prm.T + 1, N = prm.N, M = prm.M;
  const int items = prm.B * T1;
  for (int item = blockIdx.x; item < items; item += gridDim.x) {
    const int b = item / T1, t = item - b * T1;
    if (prm.active && prm.active[b] == 0) continue;  // uniform per CTA
    int n = prm.num_points ? prm.num_points[b] : N;
    n = n < 0 ? 0 : (n > N ? N : n);
    const int cnt = n < M ? n : M;
    if (t == 0 && tid == 0) {
      prm.sel_count[b] = cnt;
      if (n == 0 && prm.min_dist) prm.min_dist[b] = __int_as_float(0x7f800000);
    }
    if (n == 0) continue;

    const float* ns = prm.nom_s + (size_t)b * 3 * T1;
    const float sx = ns[t], sy = ns[T1 + t], th = ns[2 * T1 + t];
    const float cs = cosf(th), sn = sinf(th);  // torch.cos / torch.sin on float32 (pan.py:208)
    const float* px = prm.points + (size_t)b * 2 * N;
    const float* py = px + N;
    const float* vx = prm.velocities ? prm.velocities + (size_t)b * 2 * N : nullptr;
    const float* vy = vx ? vx + N : nullptr;

    // ---- phase 1: every point through the network ------------------------------------
    for (int base = 0; base < n; base += THREADS * P) {
      float x0[P], y0[P];
#pragma unroll
      for (int p = 0; p < P; ++p) {
        int i = base + p * THREADS + tid;
        i = i < n ? i : n - 1;
        float gx = px[i], gy = py[i];
        if (vx) {
          gx = flow(gx, vx[i], prm.dt, t);
          gy = flow(gy, vy[i], prm.dt, t);
        }
        const float dx = gx - sx, dy = gy - sy;  // p0 = R^T (p_t - trans)   (pan.py:210)
        x0[p] = fmaf(cs, dx, sn * dy);
        y0[p] = fmaf(cs, dy, -(sn * dx));
      }
      float mu[P][E];
      obs_point_net<E, P>(sw, x0, y0, mu);
#pragma unroll
      for (int p = 0; p < P; ++p) {
        const int i = base + p * THREADS + tid;
        if (i < n) {
          float d = 0.f;  // dist = mu^T (G p0 - h)   (dune.py:119-122)
#pragma unroll
          for (int e = 0; e < E; ++e) {
            const float ge = fmaf(prm.geo.G[e][1], y0[p], prm.geo.G[e][0] * x0[p]) - prm.geo.h[e];
            d = fmaf(mu[p][e], ge, d);
            smu[i * E + e] = mu[p][e];
          }
          keys[i] = ((unsigned long long)orderable(d) << 32) | (unsigned)i;
        }
      }
    }
    __syncthreads();

    // ---- phase 2: M rounds of block-wide arg-min (each thread owns keys tid, tid+THREADS, ..) ----
    unsigned long long mine = ~0ull;
    for (int m = 0; m < cnt; ++m) {
      unsigned long long best = ~0ull;
      for (int i = tid; i < n; i += THREADS) {
        const unsigned long long k = keys[i];
        best = k < best ? k : best;
      }
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
        const unsigned long long other = __shfl_xor_sync(0xffffffffu, best, o);
        best = other < best ? other : best;
      }
      if (lane == 0) warp_min[m & 1][warp] = best;
      __syncthreads();
      best = warp_min[m & 1][0];
#pragma unroll
      for (int w = 1; w < NW; ++w) {
        const unsigned long long other = warp_min[m & 1][w];
        best = other < best ? other : best;
      }
      const unsigned idx = (unsigned)(best & 0xffffffffull);
      if ((int)(idx % THREADS) == tid) keys[idx] = ~0ull;  // only the owner ever re-reads it
      if (tid == m) mine = best;
    }

    // ---- phase 3: thread m writes the m-th closest point --------------------------------
    if (tid < cnt) {
      const unsigned idx = (unsigned)(mine & 0xffffffffull);
      uint32_t u = (uint32_t)(mine >> 32);
      u = (u & 0x80000000u) ? (u & 0x7fffffffu) : ~u;
      const float d = __uint_as_float(u);
      float gx = px[idx], gy = py[idx];
      if (vx) {
        gx = flow(gx, vx[idx], prm.dt, t);
        gy = flow(gy, vy[idx], prm.dt, t);
      }
      const size_t o = ((size_t)b * T1 + t) * M + tid;
      // lam = ((-R) G^T) mu   (dune.py:89: unary minus binds first, then left-to-right matmuls)
      float lx = 0.f, ly = 0.f;
#pragma unroll
      for (int e = 0; e < E; ++e) {
        const float m_e = smu[idx * E + e];
        const float rgx = fmaf(sn, prm.geo.G[e][1], -cs * prm.geo.G[e][0]);   // (-R G^T)[0][e]
        const float rgy = fmaf(-cs, prm.geo.G[e][1], -sn * prm.geo.G[e][0]);  // (-R G^T)[1][e]
        lx = fmaf(rgx, m_e, lx);
        ly = fmaf(rgy, m_e, ly);
        prm.sel_mu[o * E + e] = m_e;
      }
      prm.sel_lam[o * 2 + 0] = lx;
      prm.sel_lam[o * 2 + 1] = ly;
      prm.sel_pts[o * 2 + 0] = gx;
      prm.sel_pts[o * 2 + 1] = gy;
      prm.sel_dist[o] = d;
      if (t == 0 && tid == 0 && prm.min_dist) prm.min_dist[b] = d;  // dune.py:97-98
    }
    __syncthreads();  // keys / smu are reused by the next item
  }
}

}  // namespace nb
