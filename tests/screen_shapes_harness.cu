// Test harness for tests/test_gpu_screen_warp.py: runs ONE of the two mma.sync screening kernels (csrc/dune_screen_mma_kernel.cuh) on
// host inputs and returns everything the screening pass writes -- candidate lists, counts, refine / flag lists, statistics -- so that
// the two shapes can be compared item by item.  The screen operand image is built by the library (nb::build_tc_image), which this
// shared object links against.
#include <cstdint>
#include <cstring>
#include <vector>

#include "dune_screen_mma_kernel.cuh"

namespace nb {
int build_tc_image(const float* w, int E, std::vector<unsigned char>& out, bool screen);
}

template <typename T>
static cudaError_t upload(T** d, const T* h, size_t n) {
  *d = nullptr;
  if (!h) return cudaSuccess;
  cudaError_t e = cudaMalloc(d, n * sizeof(T));
  return e != cudaSuccess ? e : cudaMemcpy(*d, h, n * sizeof(T), cudaMemcpyHostToDevice);
}

template <typename T>
static cudaError_t alloc_fill(T** d, size_t n, int byte) {
  cudaError_t e = cudaMalloc(d, n * sizeof(T));
  return e != cudaSuccess ? e : cudaMemset(*d, byte, n * sizeof(T));
}

// shape 1 = dune_screen_warp_kernel, 2 = dune_screen_mma_kernel.  Outputs (host): cand_idx / cand_dt (B (T+1) 32), cand_cnt (B (T+1)),
// flag_list (B (T+1)), refine_list (2 B (T+1)), flag_count (4), stats (4), sel_count (B), min_dist (B).  Integer outputs start as
// 0x7f7f7f7f and float outputs as the same bytes, so entries a kernel does not write compare equal only if neither kernel writes them.
extern "C" int nb_test_screen(int shape, int B, int N, int T, int M, int E, const float* G, const float* h, float c_mu, float dt, int skip_t0,
                              int calibrate, const float* nom_s, const float* points, const float* velocities, const int32_t* num_points,
                              const int32_t* active, const float* weights, int32_t* cand_idx, float* cand_dt, int32_t* cand_cnt, int32_t* flag_list,
                              int32_t* refine_list, int32_t* flag_count, uint32_t* stats, int32_t* sel_count, float* min_dist) {
  using namespace nb;
  if (N > 1024 || E > kMaxEdges) return -1;
  const size_t T1 = (size_t)T + 1, items = (size_t)B * T1;
  std::vector<unsigned char> img;
  build_tc_image(weights, E, img, true);
  DuneParams prm{};
  unsigned char* d_img = nullptr;
  float *d_ns, *d_pts, *d_vel, *d_cdt, *d_md;
  int32_t *d_np, *d_act, *d_cidx, *d_ccnt, *d_fl, *d_rl, *d_fc, *d_sc;
  unsigned* d_st;
  cudaError_t e = upload(&d_img, img.data(), img.size());
  if (e == cudaSuccess) e = upload(&d_ns, nom_s, (size_t)B * 3 * T1);
  if (e == cudaSuccess) e = upload(&d_pts, points, (size_t)B * 2 * N);
  if (e == cudaSuccess) e = upload(&d_vel, velocities, (size_t)B * 2 * N);
  if (e == cudaSuccess) e = upload(&d_np, num_points, (size_t)B);
  if (e == cudaSuccess) e = upload(&d_act, active, (size_t)B);
  if (e == cudaSuccess) e = alloc_fill(&d_cidx, items * kCandMax, 0x7f);
  if (e == cudaSuccess) e = alloc_fill(&d_cdt, items * kCandMax, 0x7f);
  if (e == cudaSuccess) e = alloc_fill(&d_ccnt, items, 0x7f);
  if (e == cudaSuccess) e = alloc_fill(&d_fl, items, 0x7f);
  if (e == cudaSuccess) e = alloc_fill(&d_rl, 2 * items, 0x7f);
  if (e == cudaSuccess) e = alloc_fill(&d_fc, (size_t)4, 0);
  if (e == cudaSuccess) e = alloc_fill(&d_st, (size_t)4, 0);
  if (e == cudaSuccess) e = alloc_fill(&d_sc, (size_t)B, 0x7f);
  if (e == cudaSuccess) e = alloc_fill(&d_md, (size_t)B, 0x7f);
  if (e != cudaSuccess) return -2;
  prm.nom_s = d_ns; prm.points = d_pts; prm.velocities = d_vel; prm.num_points = d_np; prm.active = d_act;
  prm.sel_count = d_sc; prm.min_dist = d_md;
  prm.B = B; prm.N = N; prm.T = T; prm.M = M; prm.dt = dt;
  prm.geo.E = E;
  for (int i = 0; i < E; ++i) { prm.geo.G[i][0] = G[2 * i]; prm.geo.G[i][1] = G[2 * i + 1]; prm.geo.h[i] = h[i]; }
  prm.cand_idx = d_cidx; prm.cand_cnt = d_ccnt; prm.cand_dt = d_cdt; prm.screen_stats = d_st; prm.c_mu = c_mu;
  prm.flag_list = d_fl; prm.flag_count = d_fc; prm.refine_list = d_rl; prm.skip_t0 = skip_t0; prm.calibrate = calibrate;
  prm.screen_mma = shape;
  int sms = 0;
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, 0);
  auto go = [&](auto kern, size_t smem, int grid) {
    if (e == cudaSuccess) e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e == cudaSuccess) {
      kern<<<grid, 128, smem>>>(prm, d_img);
      e = cudaGetLastError();
    }
  };
  const int grid = sms * 4;  // fewer CTAs than items: every kernel loops over several
  if (shape == 1) {
    if (N <= 512) go(dune_screen_warp_kernel<4>, dune_screen_warp_smem_bytes(N), grid);
    else go(dune_screen_warp_kernel<8>, dune_screen_warp_smem_bytes(N), grid);
  } else {
    if (N <= 512) go(dune_screen_mma_kernel<4>, dune_screen_mma_smem_bytes(N, M), grid);
    else go(dune_screen_mma_kernel<8>, dune_screen_mma_smem_bytes(N, M), grid);
  }
  if (e == cudaSuccess) e = cudaDeviceSynchronize();
  if (e == cudaSuccess) e = cudaMemcpy(cand_idx, d_cidx, items * kCandMax * 4, cudaMemcpyDeviceToHost);
  if (e == cudaSuccess) e = cudaMemcpy(cand_dt, d_cdt, items * kCandMax * 4, cudaMemcpyDeviceToHost);
  if (e == cudaSuccess) e = cudaMemcpy(cand_cnt, d_ccnt, items * 4, cudaMemcpyDeviceToHost);
  if (e == cudaSuccess) e = cudaMemcpy(flag_list, d_fl, items * 4, cudaMemcpyDeviceToHost);
  if (e == cudaSuccess) e = cudaMemcpy(refine_list, d_rl, 2 * items * 4, cudaMemcpyDeviceToHost);
  if (e == cudaSuccess) e = cudaMemcpy(flag_count, d_fc, 4 * 4, cudaMemcpyDeviceToHost);
  if (e == cudaSuccess) e = cudaMemcpy(stats, d_st, 4 * 4, cudaMemcpyDeviceToHost);
  if (e == cudaSuccess) e = cudaMemcpy(sel_count, d_sc, (size_t)B * 4, cudaMemcpyDeviceToHost);
  if (e == cudaSuccess) e = cudaMemcpy(min_dist, d_md, (size_t)B * 4, cudaMemcpyDeviceToHost);
  for (void* p : {(void*)d_img, (void*)d_ns, (void*)d_pts, (void*)d_vel, (void*)d_np, (void*)d_act, (void*)d_cidx, (void*)d_cdt, (void*)d_ccnt,
                  (void*)d_fl, (void*)d_rl, (void*)d_fc, (void*)d_st, (void*)d_sc, (void*)d_md})
    if (p) cudaFree(p);
  return e == cudaSuccess ? 0 : -3;
}
