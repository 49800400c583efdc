// C-ABI of the PAN hot path (include/neupan_b200.h): handle, workspaces, launch logic.
// No torch, no C++ types across the boundary.  One handle = one (process, GPU); not thread-safe.
#include "../../include/neupan_b200.h"

#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <new>

#include "common.cuh"
#include "dune_launch.cuh"
#include "nrmp_kernel.cuh"
#include "scan_kernel.cuh"
#include "ipath_kernel.cuh"
#include "dune_train_kernel.cuh"

#include <vector>

namespace nb {
// dune_mma.cu
void build_mma_image(const float* w, int E, std::vector<unsigned char>& out);
int launch_dune_mma(const DuneParams& prm, const unsigned char* d_image, int sm_count, int max_smem_optin, int cta_per_sm_limit, cudaStream_t st,
                    char* err, size_t errlen);
// dune_tc.cu
int build_tc_image(const float* w, int E, std::vector<unsigned char>& out, bool screen);
int launch_dune_tc(const DuneParams& prm, const unsigned char* d_image, const unsigned char* d_screen_image, int image_flags, int variant, int sm_count,
                   int max_smem_optin, cudaStream_t st, char* err, size_t errlen);
}  // namespace nb

namespace {

thread_local char g_err[512] = "";
long long g_launches = 0;

int fail(int code, const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
  return code;
}

#define NB_CUDA(call)                                                                             \
  do {                                                                                            \
    cudaError_t e__ = (call);                                                                     \
    if (e__ != cudaSuccess) return fail(NB_ERR_CUDA, "%s failed: %s", #call, cudaGetErrorString(e__)); \
  } while (0)

template <typename T>
cudaError_t dalloc(T** p, size_t n) {
  return cudaMalloc((void**)p, (n ? n : 1) * sizeof(T));
}

}  // namespace

struct nb_ipath {
  nb_ipath_config cfg;
  int B = 0;
  int64_t P = 0;
  double* d_pts = nullptr;
  int32_t* d_curve_begin = nullptr;
  int32_t* d_env_curve_begin = nullptr;
  double* d_interval = nullptr;
  int32_t* d_curve_index = nullptr;
  int32_t* d_point_index = nullptr;
  int32_t* d_arrive_flag = nullptr;
};

struct nb_dune_train {
  int E = 0, device = 0, n_weights = 0;
  float G[nb::kMaxEdges][2];
  float h[nb::kMaxEdges];
  float *d_weights = nullptr, *d_m = nullptr, *d_v = nullptr, *d_thetas = nullptr;
  double* d_losses = nullptr;
  size_t thetas_cap = 0;
  long long steps = 0;  // optimiser steps taken so far (Adam bias correction)
};

struct nb_pan {
  nb_pan_config cfg;
  nb::Geometry geo;
  int sm_count = 0;
  int max_smem_optin = 0;
  // device buffers
  float* d_weights = nullptr;
  unsigned char* d_image = nullptr;  // fragment-ordered fp16 hi/lo weight image of the mma.sync DUNE kernel
  unsigned char* d_tc_image = nullptr;  // UMMA operand image of the tcgen05 DUNE kernel
  int tc_flags = 0;                     // build_tc_image(): bit 0 = bounded tanh arguments
  unsigned char* d_tc_screen = nullptr; // operand image of the screening network (NB_OPT_DUNE_KERNEL = 4)
  int32_t *cand_idx = nullptr, *cand_cnt = nullptr, *flag_list = nullptr, *flag_count = nullptr, *refine_list = nullptr;
  float* cand_dt = nullptr;
  unsigned* screen_stats = nullptr;
  float c_mu = 0.012f;                  // bound on the screening network's |mu~ - mu|: set by calibrate_screen() to 4 x the largest error
                                        // measured for THIS checkpoint and polygon (NB_SCREEN_CMU overrides; DESIGN.md 3.1)
  bool screen_calibrated = false;
  float screen_cal_ratio = 0.f;
  int dune_variant = 2;              // NB_OPT_DUNE_KERNEL: 0 = FP32 FFMA, 1 = mma.sync tensor-core, 2 = tcgen05 tensor-core kernel
  int overlap = 1;                   // NB_OPT_OVERLAP: number of env sub-batches pipelined on internal streams
  cudaStream_t streams[4] = {nullptr, nullptr, nullptr, nullptr};
  cudaEvent_t ev_fork = nullptr, ev_join[4] = {nullptr, nullptr, nullptr, nullptr};
  // host-input entry points: uploads run on copy_stream in env chunks; ev_chunk[c] = chunk c (and everything before it) has landed
  static constexpr int kMaxChunks = 8;
  cudaStream_t copy_stream = nullptr;
  cudaEvent_t ev_chunk[kMaxChunks] = {}, ev_inputs_free = nullptr;
  int h2d_chunks = 4;               // NB_H2D_CHUNKS (developer switch, read at create); 1 = no overlap
  float *sel_mu = nullptr, *sel_lam = nullptr, *sel_pts = nullptr, *sel_dist = nullptr;
  int32_t* sel_count = nullptr;
  float *prev_s = nullptr, *prev_u = nullptr, *prev_mu = nullptr, *prev_lam = nullptr;
  int32_t *prev_count = nullptr, *prev_valid = nullptr, *active = nullptr, *iters = nullptr, *status = nullptr, *ipm_it = nullptr;
  float* min_dist = nullptr;
  // differentiable mode (NB_OPT_DIFFERENTIABLE): adjoint records of every (iteration, env) solve + gradient workspaces
  int differentiable = 0, adj_iters = 0;
  double *adj_rec = nullptr, *adj_gs = nullptr, *adj_gu = nullptr, *adj_gd = nullptr, *adj_gtheta = nullptr;
  int32_t* adj_valid = nullptr;
  int* work_counters = nullptr;     // dynamic env -> warp assignment of the NRMP kernel, one counter per internal stream
  int dune_skip_t0 = 1;             // NB_OPT_DUNE_SKIP_T0: PAN iterations k > 0 keep the step-0 items of iteration 0 (screening variant)
  int screen_mma = 1;               // NB_OPT_DUNE_SCREEN_MMA: screening pass on mma.sync (N <= 512) instead of tcgen05
  int screen_shape = 1;             // the mma.sync screening pass: 1 = by batch size, 2 = one CTA of 4 warps per item, 3 = one warp per item (NB_SCREEN_MMA)
  int nrmp_defer_stop_min = 256;    // NB_NRMP_DEFER_STOP_MIN (developer switch, read at create): smallest batch whose stop criterion runs as its own kernel
  int nrmp_dynamic = 1;             // NB_NRMP_STATIC=1 (developer switch, read at create) turns the persistent-warp schedule off
  float* warm = nullptr;            // NRMP warm-start records, nrmp_warm_floats(T, M) per environment
  int32_t* warm_valid = nullptr;
  int nrmp_warm = 0;                // NB_OPT_NRMP_WARM (off by default: see DESIGN.md 3.2)
  double nrmp_gap_tol = 1e-12;      // NB_NRMP_GAP_TOL (developer switch, read once at create)
  int warm_check_it = 12;           // NB_NRMP_RESTART_IT / NB_NRMP_RESTART_GAP (developer switches): early cold restart of a warm start
  double warm_check_gap = 1e-5;
  // staging for the host-pointer entry point
  float *h_in = nullptr, *h_out = nullptr;  // device staging
  size_t h_in_floats = 0, h_out_floats = 0;
  int32_t* h_np = nullptr;
  int32_t* h_io = nullptr;
  bool dune_attr_set = false, nrmp_attr_set = false;
};

namespace {

int check_forward_args(const nb_pan* p, int B, int N) {
  if (!p) return fail(NB_ERR_INVALID, "null handle");
  if (B <= 0) return fail(NB_ERR_INVALID, "B must be positive (got %d)", B);
  if (B > p->cfg.max_envs) return fail(NB_ERR_CAPACITY, "B=%d exceeds max_envs=%d", B, p->cfg.max_envs);
  if (N < 0) return fail(NB_ERR_INVALID, "N must be >= 0");
  if (N > p->cfg.max_points) return fail(NB_ERR_CAPACITY, "N=%d exceeds max_points=%d", N, p->cfg.max_points);
  return NB_OK;
}

// NB_EDGE_MASK: bit E set <=> dune_inst.cu was compiled for that edge count (build script)
#ifndef NB_EDGE_MASK
#define NB_EDGE_MASK 0x10
#endif

int launch_dune(nb_pan* p, const nb::DuneParams& prm, cudaStream_t st, int cta_limit = 0) {
  int rc = NB_ERR_INVALID;
  char msg[256] = "";
  if (p->dune_variant >= 2) {
    rc = nb::launch_dune_tc(prm, p->d_tc_image, p->d_tc_screen, p->tc_flags, p->dune_variant, p->sm_count, p->max_smem_optin, st, msg, sizeof(msg));
    if (rc) return fail(rc, "%s", msg);
    g_launches += p->dune_variant == 4 ? 3 : 1;
    return NB_OK;
  }
  if (p->dune_variant == 1) {
    rc = nb::launch_dune_mma(prm, p->d_image, p->sm_count, p->max_smem_optin, cta_limit, st, msg, sizeof(msg));
    if (rc) return fail(rc, "%s", msg);
    ++g_launches;
    return NB_OK;
  }
  switch (p->cfg.edge_dim) {
#define NB_CASE(E_)                                                                                        \
  case E_:                                                                                                 \
    rc = nb::launch_dune_e<E_>(prm, p->sm_count, p->max_smem_optin, st, msg, sizeof(msg));                 \
    break;
#if NB_EDGE_MASK & (1 << 3)
    NB_CASE(3)
#endif
#if NB_EDGE_MASK & (1 << 4)
    NB_CASE(4)
#endif
#if NB_EDGE_MASK & (1 << 5)
    NB_CASE(5)
#endif
#if NB_EDGE_MASK & (1 << 6)
    NB_CASE(6)
#endif
#if NB_EDGE_MASK & (1 << 7)
    NB_CASE(7)
#endif
#if NB_EDGE_MASK & (1 << 8)
    NB_CASE(8)
#endif
#undef NB_CASE
    default:
      return fail(NB_ERR_INVALID, "edge_dim %d not built into this library (mask 0x%x)", p->cfg.edge_dim, NB_EDGE_MASK);
  }
  if (rc) return fail(rc, "%s", msg);
  ++g_launches;
  return NB_OK;
}

int launch_nrmp(nb_pan* p, nb::NrmpParams prm, cudaStream_t st, int counter_slot = 0) {
  const nb_pan_config& c = p->cfg;
  prm.T = c.receding; prm.M = c.nrmp_max_num; prm.E = c.edge_dim; prm.kin = c.kinematics;
  prm.max_ipm_iter = 60;
  prm.gap_tol = p->nrmp_gap_tol;
  prm.warm_check_it = p->warm_check_it; prm.warm_check_gap = p->warm_check_gap;
  prm.iter_threshold = c.iter_threshold;
  prm.dt = c.step_time; prm.L = c.wheelbase;
  for (int i = 0; i < 3; ++i) prm.q[i] = c.q_s[i];
  prm.p_u = c.p_u; prm.eta = c.eta; prm.d_max = c.d_max; prm.d_min = c.d_min;
  prm.ro = c.ro_obs; prm.bk = c.bk;
  for (int i = 0; i < 2; ++i) {
    prm.speed[i] = c.max_speed[i];
    prm.acce[i] = c.max_acce[i] * c.step_time;
  }
  for (int e = 0; e < nb::kMaxEdges; ++e) prm.h[e] = p->geo.h[e];
  // large batches: the stop criterion's ~1300 dependent global reads per environment leave the solve kernel (where each warp waits for
  // them alone) for a kernel of its own; small batches keep it inside (one launch less per PAN iteration matters more there)
  prm.defer_stop = (prm.prev_valid != nullptr && prm.B >= p->nrmp_defer_stop_min) ? 1 : 0;
  const size_t wd = nb::nrmp_warp_doubles(prm.T, prm.M);
  const size_t extra = nb::nrmp_cta_extra_bytes(prm.T);
  const int TM = prm.T * prm.M;
  if (TM > 256) return fail(NB_ERR_CAPACITY, "receding*nrmp_max_num = %d exceeds 256", TM);
  int warps = (int)(((size_t)p->max_smem_optin - extra) / (wd * sizeof(double)));
  if (warps < 1) return fail(NB_ERR_CAPACITY, "T=%d, M=%d need %zu B of shared memory per environment", prm.T, prm.M, wd * 8);
  // small CTAs (<= 2 warps): many of them fit per SM and each warp retires independently
  if (warps > 2) warps = 2;
  if (prm.T == 10 && prm.M == 10) warps = NB_NRMP_WPC;
  const size_t smem = (size_t)warps * wd * sizeof(double) + extra;
  int grid = (prm.B + warps - 1) / warps;
  auto go = [&](auto kern) -> int {
    NB_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, p->max_smem_optin));
    if (p->nrmp_dynamic && p->work_counters) {
      // persistent warps: as many CTAs as are resident at once; they pull environments from a counter until the batch is done
      int per_sm = 0;
      NB_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, warps * 32, smem));
      static int cap = -1;  // NB_NRMP_CTA_CAP (developer switch): fewer resident CTAs per SM, to share the SMs with a kernel of another stream
      if (cap < 0) {
        const char* v = getenv("NB_NRMP_CTA_CAP");
        cap = v ? atoi(v) : 0;
      }
      if (cap > 0 && cap < per_sm) per_sm = cap;
      const int resident = (per_sm > 0 ? per_sm : 1) * p->sm_count;
      if (grid > resident) {
        grid = resident;
        prm.work_counter = p->work_counters + counter_slot;
        NB_CUDA(cudaMemsetAsync(prm.work_counter, 0, sizeof(int), st));
      }
    }
    kern<<<grid, warps * 32, smem, st>>>(prm, warps, (int)wd);
    ++g_launches;
    if (prm.defer_stop) {  // section 8 (stop criterion, PAN.current_nom_values) as a bandwidth kernel over the batch
      nb::nrmp_stop_kernel<<<(prm.B + 3) / 4, 128, 0, st>>>(prm);
      ++g_launches;
    }
    NB_CUDA(cudaGetLastError());
    return NB_OK;
  };
  const int hpl = (TM + 31) / 32;
  // specialisations with compile-time (T, M) for the reference's shipped configurations
  if (prm.T == 10 && prm.M == 10) return go(nb::nrmp_kernel<4, true, 10, 10>);
  if (prm.T == 15 && prm.M == 10) return go(nb::nrmp_kernel<5, true, 15, 10>);
  if (prm.T <= 16) {  // 2T <= 32: one row of the reduced system per lane
    if (hpl <= 1) return go(nb::nrmp_kernel<1, true, 0, 0>);
    if (hpl <= 2) return go(nb::nrmp_kernel<2, true, 0, 0>);
    if (hpl <= 4) return go(nb::nrmp_kernel<4, true, 0, 0>);
    if (hpl <= 5) return go(nb::nrmp_kernel<5, true, 0, 0>);
    return go(nb::nrmp_kernel<8, true, 0, 0>);
  }
  if (hpl <= 4) return go(nb::nrmp_kernel<4, false, 0, 0>);
  return go(nb::nrmp_kernel<8, false, 0, 0>);
}

// Screening bound of this handle: the screen and the exact network evaluate the same 32-point items (points uniform in the square the
// reference trains DUNE on, [-25, 25]^2, and in [-6, 6]^2 around the robot, identity frame) and the refine kernel's statistics give
// max |d~ - d| / sum_e |G_e p - h_e| over every point; c_mu = 4 x that, clamped to [0.004, 0.05].
int calibrate_screen(nb_pan* p, cudaStream_t st) {
  const nb_pan_config& c = p->cfg;
  const int T1 = c.receding + 1, N = 32;
  int Bc = c.max_envs < 512 ? c.max_envs : 512;
  const int rounds = (4096 + Bc * T1 - 1) / (Bc * T1) < 1 ? 1 : (4096 + Bc * T1 - 1) / (Bc * T1);
  std::vector<float> pts((size_t)Bc * 2 * N), ns((size_t)Bc * 3 * T1, 0.f);
  float *d_pts = nullptr, *d_ns = nullptr, *d_md = nullptr;
  NB_CUDA(dalloc(&d_pts, pts.size()));
  NB_CUDA(dalloc(&d_ns, ns.size()));
  NB_CUDA(dalloc(&d_md, (size_t)Bc));
  NB_CUDA(cudaMemcpyAsync(d_ns, ns.data(), ns.size() * sizeof(float), cudaMemcpyHostToDevice, st));
  unsigned saved[4];
  NB_CUDA(cudaStreamSynchronize(st));
  NB_CUDA(cudaMemcpy(saved, p->screen_stats, sizeof(saved), cudaMemcpyDeviceToHost));
  NB_CUDA(cudaMemset(p->screen_stats, 0, sizeof(saved)));
  unsigned long long rng = 0x9E3779B97F4A7C15ull;
  auto uni = [&]() { rng = rng * 6364136223846793005ull + 1442695040888963407ull; return (float)((rng >> 40) * (1.0 / 16777216.0)); };
  const int variant = p->dune_variant;
  p->dune_variant = 4;
  int rc = NB_OK;
  for (int r = 0; r < (rounds > 16 ? 16 : rounds) && rc == NB_OK; ++r) {
    for (int b = 0; b < Bc; ++b) {
      const float R = ((b + r) & 1) ? 25.f : 6.f;
      for (int i = 0; i < N; ++i) { pts[((size_t)b * 2) * N + i] = R * (2.f * uni() - 1.f); pts[((size_t)b * 2 + 1) * N + i] = R * (2.f * uni() - 1.f); }
    }
    cudaError_t e = cudaMemcpyAsync(d_pts, pts.data(), pts.size() * sizeof(float), cudaMemcpyHostToDevice, st);
    if (e != cudaSuccess) { rc = fail(NB_ERR_CUDA, "calibrate_screen: %s", cudaGetErrorString(e)); break; }
    nb::DuneParams prm{};
    prm.weights = p->d_weights; prm.nom_s = d_ns; prm.points = d_pts;
    prm.sel_mu = p->sel_mu; prm.sel_lam = p->sel_lam; prm.sel_pts = p->sel_pts; prm.sel_dist = p->sel_dist; prm.sel_count = p->sel_count; prm.min_dist = d_md;
    prm.B = Bc; prm.N = N; prm.T = c.receding; prm.M = c.nrmp_max_num; prm.dt = (float)c.step_time; prm.geo = p->geo;
    prm.cand_idx = p->cand_idx; prm.cand_cnt = p->cand_cnt; prm.cand_dt = p->cand_dt; prm.screen_stats = p->screen_stats; prm.c_mu = p->c_mu;
    prm.flag_list = p->flag_list; prm.flag_count = p->flag_count; prm.refine_list = p->refine_list; prm.calibrate = 1;
    for (int shape = 0; shape < 2 && rc == NB_OK; ++shape) {  // both screening kernels (tcgen05 / mma.sync): the bound holds whichever option is set later
      prm.screen_mma = shape ? p->screen_shape : 0;
      rc = launch_dune(p, prm, st);
      if (rc == NB_OK && cudaStreamSynchronize(st) != cudaSuccess) rc = fail(NB_ERR_CUDA, "calibrate_screen: kernel failed");
    }
  }
  p->dune_variant = variant;
  if (rc == NB_OK) {
    unsigned h[4];
    NB_CUDA(cudaMemcpy(h, p->screen_stats, sizeof(h), cudaMemcpyDeviceToHost));
    float ratio;
    memcpy(&ratio, &h[0], 4);
    p->screen_cal_ratio = ratio;
    float cm = 4.f * ratio;
    p->c_mu = cm < 0.008f ? 0.008f : (cm > 0.05f ? 0.05f : cm);
    if (const char* e = getenv("NB_SCREEN_CMU")) p->c_mu = (float)atof(e);
    p->screen_calibrated = true;
  }
  cudaMemcpy(p->screen_stats, saved, sizeof(saved), cudaMemcpyHostToDevice);
  cudaFree(d_pts); cudaFree(d_ns); cudaFree(d_md);
  return rc;
}

__global__ void init_run_kernel(int B, int32_t* active, int32_t* iters, int32_t* status, float* min_dist, int32_t* sel_count, int32_t* warm_valid) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < B) {
    active[i] = 1; iters[i] = 0; status[i] = 0;
    warm_valid[i] = 0;  // the first NRMP solve of a forward() is cold: results do not depend on earlier calls
    min_dist[i] = __int_as_float(0x7f800000);
    sel_count[i] = 0;
  }
}

__global__ void finish_run_kernel(int B, const int32_t* iters, const int32_t* status, const float* min_dist,
                                  int32_t* out_iters, int32_t* out_status, float* out_min_dist) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < B) {
    if (out_iters) out_iters[i] = iters[i];
    if (out_status) out_status[i] = status[i];
    if (out_min_dist) out_min_dist[i] = min_dist[i];
  }
}

}  // namespace

extern "C" {

int64_t nb_weight_count(int32_t edge_dim) { return nb::WeightLayout::count(edge_dim); }
int nb_version(void) { return NB_VERSION; }
const char* nb_last_error(void) { return g_err; }
int64_t nb_launch_count(void) { return g_launches; }

int nb_pan_create(const nb_pan_config* cfg, const float* weights, int64_t n_weights, const float* G, const float* h, nb_pan_t** out) {
  if (!cfg || !out) return fail(NB_ERR_INVALID, "null argument");
  *out = nullptr;
  if (cfg->receding < 1 || cfg->receding > 32) return fail(NB_ERR_INVALID, "receding must be in 1..32 (got %d)", cfg->receding);
  if (cfg->kinematics < 0 || cfg->kinematics > 2) return fail(NB_ERR_INVALID, "kinematics must be NB_KIN_DIFF/ACKER/OMNI");
  if (cfg->nrmp_max_num < 0 || cfg->nrmp_max_num > 32) return fail(NB_ERR_INVALID, "nrmp_max_num must be in 0..32");
  if (cfg->iter_num < 0) return fail(NB_ERR_INVALID, "iter_num must be >= 0");
  if (cfg->max_envs < 1 || cfg->max_points < 0) return fail(NB_ERR_INVALID, "max_envs >= 1 and max_points >= 0 required");
  if (!(cfg->step_time > 0)) return fail(NB_ERR_INVALID, "step_time must be positive");
  if (cfg->kinematics == NB_KIN_ACKER && !(cfg->wheelbase > 0)) return fail(NB_ERR_INVALID, "acker needs a positive wheelbase");
  if (cfg->receding * cfg->nrmp_max_num > 256)
    return fail(NB_ERR_CAPACITY, "receding * nrmp_max_num = %d exceeds 256 (the NRMP kernel keeps at most 8 hinge rows per lane)", cfg->receding * cfg->nrmp_max_num);
  const bool with_dune = cfg->nrmp_max_num > 0;
  if (with_dune) {
    if (cfg->edge_dim < 3 || cfg->edge_dim > nb::kMaxEdges) return fail(NB_ERR_INVALID, "edge_dim must be in 3..%d", nb::kMaxEdges);
    if (!weights || !G || !h) return fail(NB_ERR_INVALID, "weights, G and h are required when nrmp_max_num > 0");
    if (n_weights != nb::WeightLayout::count(cfg->edge_dim))
      return fail(NB_ERR_INVALID, "expected %d weights for edge_dim %d, got %lld", nb::WeightLayout::count(cfg->edge_dim), cfg->edge_dim, (long long)n_weights);
  }
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0)
    return fail(NB_ERR_NO_DEVICE, "no CUDA device available: neupan_b200 has no CPU fallback");
  if (cfg->device < 0 || cfg->device >= ndev) return fail(NB_ERR_INVALID, "device %d out of range (%d devices)", cfg->device, ndev);
  NB_CUDA(cudaSetDevice(cfg->device));
  nb_pan* p = new (std::nothrow) nb_pan();
  if (!p) return fail(NB_ERR_INVALID, "out of host memory");
  p->cfg = *cfg;
  NB_CUDA(cudaDeviceGetAttribute(&p->sm_count, cudaDevAttrMultiProcessorCount, cfg->device));
  NB_CUDA(cudaDeviceGetAttribute(&p->max_smem_optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, cfg->device));
  memset(&p->geo, 0, sizeof(p->geo));
  p->geo.E = cfg->edge_dim;
  const size_t B = cfg->max_envs, T1 = cfg->receding + 1, T = cfg->receding, M = cfg->nrmp_max_num, E = with_dune ? cfg->edge_dim : 1;
  if (with_dune) {
    for (int e = 0; e < cfg->edge_dim; ++e) {
      p->geo.G[e][0] = G[2 * e]; p->geo.G[e][1] = G[2 * e + 1]; p->geo.h[e] = h[e];
    }
    NB_CUDA(dalloc(&p->d_weights, (size_t)n_weights));
    NB_CUDA(cudaMemcpy(p->d_weights, weights, (size_t)n_weights * sizeof(float), cudaMemcpyHostToDevice));
    std::vector<unsigned char> image;
    nb::build_mma_image(weights, cfg->edge_dim, image);
    NB_CUDA(dalloc(&p->d_image, image.size()));
    NB_CUDA(cudaMemcpy(p->d_image, image.data(), image.size(), cudaMemcpyHostToDevice));
    p->tc_flags = nb::build_tc_image(weights, cfg->edge_dim, image, false);
    NB_CUDA(dalloc(&p->d_tc_image, image.size()));
    NB_CUDA(cudaMemcpy(p->d_tc_image, image.data(), image.size(), cudaMemcpyHostToDevice));
    nb::build_tc_image(weights, cfg->edge_dim, image, true);
    NB_CUDA(dalloc(&p->d_tc_screen, image.size()));
    NB_CUDA(cudaMemcpy(p->d_tc_screen, image.data(), image.size(), cudaMemcpyHostToDevice));
    NB_CUDA(dalloc(&p->cand_idx, (size_t)cfg->max_envs * (cfg->receding + 1) * nb::kCandMax));
    NB_CUDA(dalloc(&p->cand_dt, (size_t)cfg->max_envs * (cfg->receding + 1) * nb::kCandMax));
    NB_CUDA(dalloc(&p->cand_cnt, (size_t)cfg->max_envs * (cfg->receding + 1)));
    NB_CUDA(dalloc(&p->flag_list, (size_t)cfg->max_envs * (cfg->receding + 1)));
    NB_CUDA(dalloc(&p->flag_count, (size_t)32));  // 4 words per internal stream: flagged items, the two refine list lengths, the screen item counter
    NB_CUDA(dalloc(&p->refine_list, (size_t)2 * cfg->max_envs * (cfg->receding + 1)));
    NB_CUDA(dalloc(&p->screen_stats, (size_t)4));
    NB_CUDA(cudaMemset(p->screen_stats, 0, 4 * sizeof(unsigned)));
    if (const char* e = getenv("NB_SCREEN_CMU")) p->c_mu = (float)atof(e);
  }
  NB_CUDA(dalloc(&p->sel_mu, B * T1 * M * E));
  NB_CUDA(dalloc(&p->sel_lam, B * T1 * M * 2));
  NB_CUDA(dalloc(&p->sel_pts, B * T1 * M * 2));
  NB_CUDA(dalloc(&p->sel_dist, B * T1 * M));
  NB_CUDA(dalloc(&p->sel_count, B));
  NB_CUDA(dalloc(&p->prev_s, B * 3 * T1));
  NB_CUDA(dalloc(&p->prev_u, B * 2 * T));
  NB_CUDA(dalloc(&p->prev_mu, B * T1 * M * E));
  NB_CUDA(dalloc(&p->prev_lam, B * T1 * M * 2));
  NB_CUDA(dalloc(&p->prev_count, B));
  NB_CUDA(dalloc(&p->prev_valid, B));
  NB_CUDA(dalloc(&p->active, B));
  NB_CUDA(dalloc(&p->iters, B));
  NB_CUDA(dalloc(&p->status, B));
  NB_CUDA(dalloc(&p->ipm_it, B));
  NB_CUDA(cudaMemset(p->ipm_it, 0, B * sizeof(int32_t)));
  NB_CUDA(dalloc(&p->min_dist, B));
  NB_CUDA(dalloc(&p->warm, B * nb::nrmp_warm_floats(cfg->receding, cfg->nrmp_max_num)));
  NB_CUDA(dalloc(&p->warm_valid, B));
  NB_CUDA(dalloc(&p->work_counters, (size_t)8));
  if (getenv("NB_NRMP_STATIC")) p->nrmp_dynamic = 0;
  if (const char* e = getenv("NB_NRMP_DEFER_STOP_MIN")) p->nrmp_defer_stop_min = atoi(e);
  if (const char* e = getenv("NB_H2D_CHUNKS")) { p->h2d_chunks = atoi(e); if (p->h2d_chunks < 1) p->h2d_chunks = 1; if (p->h2d_chunks > nb_pan::kMaxChunks) p->h2d_chunks = nb_pan::kMaxChunks; }
  if (const char* e = getenv("NB_DUNE_SKIP_T0")) p->dune_skip_t0 = atoi(e) != 0;  // developer overrides of the option defaults
  if (const char* e = getenv("NB_SCREEN_MMA")) {  // 0 / 1: the option's initial value; 2 / 3: on, with the CTA-per-item / warp-per-item kernel
    p->screen_mma = atoi(e) != 0;
    p->screen_shape = atoi(e) == 2 || atoi(e) == 3 ? atoi(e) : 1;
  }
  if (const char* e = getenv("NB_NRMP_RESTART_IT")) p->warm_check_it = atoi(e);
  if (const char* e = getenv("NB_NRMP_RESTART_GAP")) p->warm_check_gap = atof(e);
  NB_CUDA(cudaMemset(p->warm_valid, 0, B * sizeof(int32_t)));
  if (const char* e = getenv("NB_NRMP_GAP_TOL")) p->nrmp_gap_tol = atof(e);
  NB_CUDA(cudaMemset(p->prev_valid, 0, B * sizeof(int32_t)));
  NB_CUDA(cudaMemset(p->prev_count, 0, B * sizeof(int32_t)));
  NB_CUDA(cudaMemset(p->sel_count, 0, B * sizeof(int32_t)));
  if (int rc = nb_pan_set_option(p, NB_OPT_OVERLAP, 2)) {  // the default: two sub-batches on internal streams (streams / events are made here)
    nb_pan_destroy(p);
    return rc;
  }
  *out = p;
  return NB_OK;
}

int nb_pan_destroy(nb_pan_t* p) {
  if (!p) return NB_OK;
  cudaSetDevice(p->cfg.device);
  for (int i = 0; i < 4; ++i) {
    if (p->streams[i]) cudaStreamDestroy(p->streams[i]);
    if (p->ev_join[i]) cudaEventDestroy(p->ev_join[i]);
  }
  if (p->ev_fork) cudaEventDestroy(p->ev_fork);
  if (p->copy_stream) cudaStreamDestroy(p->copy_stream);
  if (p->ev_inputs_free) cudaEventDestroy(p->ev_inputs_free);
  for (cudaEvent_t e : p->ev_chunk)
    if (e) cudaEventDestroy(e);
  void* bufs[] = {p->d_tc_image, p->d_image, p->d_weights, p->sel_mu, p->sel_lam, p->sel_pts, p->sel_dist, p->sel_count, p->prev_s, p->prev_u, p->prev_mu,
                  p->prev_lam, p->prev_count, p->prev_valid, p->active, p->iters, p->status, p->ipm_it, p->min_dist, p->h_in, p->h_out, p->h_np, p->h_io,
                  p->d_tc_screen, p->cand_idx, p->cand_cnt, p->cand_dt, p->screen_stats, p->flag_list, p->flag_count, p->refine_list, p->warm, p->warm_valid, p->work_counters, p->adj_rec, p->adj_gs, p->adj_gu, p->adj_gd, p->adj_gtheta, p->adj_valid};
  for (void* b : bufs)
    if (b) cudaFree(b);
  delete p;
  return NB_OK;
}

int nb_pan_set_adjust(nb_pan_t* p, const float q_s[3], float p_u, float eta, float d_max, float d_min) {
  if (!p || !q_s) return fail(NB_ERR_INVALID, "null argument");
  for (int i = 0; i < 3; ++i) p->cfg.q_s[i] = q_s[i];
  p->cfg.p_u = p_u; p->cfg.eta = eta; p->cfg.d_max = d_max; p->cfg.d_min = d_min;
  return NB_OK;
}

int nb_pan_set_iteration(nb_pan_t* p, int32_t iter_num, float iter_threshold) {
  if (!p || iter_num < 0) return fail(NB_ERR_INVALID, "bad argument");
  p->cfg.iter_num = iter_num; p->cfg.iter_threshold = iter_threshold;
  return NB_OK;
}

int nb_pan_set_option(nb_pan_t* p, int32_t option, int32_t value) {
  if (!p) return fail(NB_ERR_INVALID, "null handle");
  if (option == NB_OPT_DUNE_KERNEL) {
    if (value < 0 || value > 4)
      return fail(NB_ERR_INVALID, "NB_OPT_DUNE_KERNEL takes 0 (fp32 ffma), 1 (mma.sync), 2 (tcgen05), 3 (tcgen05, two threads per point) or 4 (tcgen05 with screening)");
    p->dune_variant = value;
    if (value == 4 && !p->screen_calibrated && p->d_tc_screen) {
      NB_CUDA(cudaSetDevice(p->cfg.device));
      return calibrate_screen(p, nullptr);
    }
    return NB_OK;
  }
  if (option == NB_OPT_OVERLAP) {
    if (value < 1 || value > 4) return fail(NB_ERR_INVALID, "NB_OPT_OVERLAP takes 1..4");
    NB_CUDA(cudaSetDevice(p->cfg.device));
    for (int i = 0; i < value && value > 1; ++i) {
      if (!p->streams[i]) NB_CUDA(cudaStreamCreateWithFlags(&p->streams[i], cudaStreamNonBlocking));
      if (!p->ev_join[i]) NB_CUDA(cudaEventCreateWithFlags(&p->ev_join[i], cudaEventDisableTiming));
    }
    if (value > 1 && !p->ev_fork) NB_CUDA(cudaEventCreateWithFlags(&p->ev_fork, cudaEventDisableTiming));
    p->overlap = value;
    return NB_OK;
  }
  if (option == NB_OPT_DIFFERENTIABLE) {
    if (value < 0 || value > 1) return fail(NB_ERR_INVALID, "NB_OPT_DIFFERENTIABLE takes 0 or 1");
    p->differentiable = value;
    return NB_OK;
  }
  if (option == NB_OPT_DUNE_SCREEN_MMA || option == NB_OPT_DUNE_SKIP_T0) {
    if (value < 0 || value > 1) return fail(NB_ERR_INVALID, "NB_OPT_DUNE_SCREEN_MMA / NB_OPT_DUNE_SKIP_T0 take 0 or 1");
    (option == NB_OPT_DUNE_SCREEN_MMA ? p->screen_mma : p->dune_skip_t0) = value;
    return NB_OK;
  }
  if (option == NB_OPT_NRMP_WARM) {
    if (value < 0 || value > 1) return fail(NB_ERR_INVALID, "NB_OPT_NRMP_WARM takes 0 or 1");
    p->nrmp_warm = value;
    return NB_OK;
  }
  return fail(NB_ERR_INVALID, "unknown option %d", option);
}

int nb_pan_reset_state_async(nb_pan_t* p, void* stream) {
  if (!p) return fail(NB_ERR_INVALID, "null handle");
  NB_CUDA(cudaSetDevice(p->cfg.device));
  NB_CUDA(cudaMemsetAsync(p->prev_valid, 0, (size_t)p->cfg.max_envs * sizeof(int32_t), (cudaStream_t)stream));
  NB_CUDA(cudaMemsetAsync(p->prev_count, 0, (size_t)p->cfg.max_envs * sizeof(int32_t), (cudaStream_t)stream));
  return NB_OK;
}

int nb_pan_reset_state(nb_pan_t* p) {
  if (int rc = nb_pan_reset_state_async(p, nullptr)) return rc;
  NB_CUDA(cudaStreamSynchronize(nullptr));
  return NB_OK;
}

int nb_dune_forward(nb_pan_t* p, int32_t B, int32_t N, const float* nom_s, const float* points, const float* velocities,
                    const int32_t* num_points, float* out_min_distance, void* stream) {
  if (int rc = check_forward_args(p, B, N)) return rc;
  if (p->cfg.nrmp_max_num == 0) return fail(NB_ERR_INVALID, "handle was created in no_obs mode");
  if (!nom_s || !points) return fail(NB_ERR_INVALID, "nom_s and points are required");
  if (N == 0) return fail(NB_ERR_INVALID, "N must be positive");
  NB_CUDA(cudaSetDevice(p->cfg.device));
  nb::DuneParams prm{};
  prm.weights = p->d_weights; prm.nom_s = nom_s; prm.points = points; prm.velocities = velocities; prm.num_points = num_points;
  prm.active = nullptr;
  prm.sel_mu = p->sel_mu; prm.sel_lam = p->sel_lam; prm.sel_pts = p->sel_pts; prm.sel_dist = p->sel_dist; prm.sel_count = p->sel_count;
  prm.min_dist = out_min_distance;
  prm.B = B; prm.N = N; prm.T = p->cfg.receding; prm.M = p->cfg.nrmp_max_num; prm.dt = (float)p->cfg.step_time; prm.geo = p->geo;
  prm.cand_idx = p->cand_idx; prm.cand_cnt = p->cand_cnt; prm.cand_dt = p->cand_dt; prm.screen_stats = p->screen_stats; prm.c_mu = p->c_mu;
  prm.flag_list = p->flag_list; prm.flag_count = p->flag_count; prm.refine_list = p->refine_list; prm.screen_mma = p->screen_mma ? p->screen_shape : 0;
  return launch_dune(p, prm, (cudaStream_t)stream);
}

int nb_nrmp_forward(nb_pan_t* p, int32_t B, const float* nom_s, const float* nom_u, const float* ref_s, const float* ref_us,
                    const float* fa, const float* fb, float* out_s, float* out_u, float* out_d, int32_t* out_status, void* stream) {
  if (int rc = check_forward_args(p, B, 0)) return rc;
  if (!nom_s || !nom_u || !ref_s || !ref_us || !out_s || !out_u || !out_d) return fail(NB_ERR_INVALID, "null tensor argument");
  if ((fa == nullptr) != (fb == nullptr)) return fail(NB_ERR_INVALID, "fa and fb must be given together");
  NB_CUDA(cudaSetDevice(p->cfg.device));
  nb::NrmpParams prm{};
  prm.nom_s = nom_s; prm.nom_u = nom_u; prm.ref_s = ref_s; prm.ref_us = ref_us; prm.fa = fa; prm.fb = fb;
  prm.out_s = out_s; prm.out_u = out_u; prm.out_d = out_d; prm.status = out_status;
  prm.B = B;
  return launch_nrmp(p, prm, (cudaStream_t)stream);
}

namespace {
// env chunks whose inputs arrive on another stream: chunk c = environments [bound[c], bound[c+1]), usable once ev[c] has fired
struct ChunkPlan {
  int n = 0;
  int bound[nb_pan::kMaxChunks + 1] = {};
  cudaEvent_t ev[nb_pan::kMaxChunks] = {};
};
int pan_forward_impl(nb_pan_t* p, int32_t B, int32_t N, const float* nom_s, const float* nom_u, const float* ref_s, const float* ref_us,
                     const float* points, const float* velocities, const int32_t* num_points, float* out_s, float* out_u, float* out_d,
                     float* out_min_distance, int32_t* out_iters, int32_t* out_status, void* stream, const ChunkPlan* plan);
}  // namespace

int nb_pan_forward(nb_pan_t* p, int32_t B, int32_t N, const float* nom_s, const float* nom_u, const float* ref_s, const float* ref_us,
                   const float* points, const float* velocities, const int32_t* num_points, float* out_s, float* out_u, float* out_d,
                   float* out_min_distance, int32_t* out_iters, int32_t* out_status, void* stream) {
  return pan_forward_impl(p, B, N, nom_s, nom_u, ref_s, ref_us, points, velocities, num_points, out_s, out_u, out_d, out_min_distance, out_iters,
                          out_status, stream, nullptr);
}

namespace {
int pan_forward_impl(nb_pan_t* p, int32_t B, int32_t N, const float* nom_s, const float* nom_u, const float* ref_s, const float* ref_us,
                     const float* points, const float* velocities, const int32_t* num_points, float* out_s, float* out_u, float* out_d,
                     float* out_min_distance, int32_t* out_iters, int32_t* out_status, void* stream, const ChunkPlan* plan) {
  if (int rc = check_forward_args(p, B, N)) return rc;
  if (!nom_s || !nom_u || !ref_s || !ref_us || !out_s || !out_u || !out_d) return fail(NB_ERR_INVALID, "null tensor argument");
  if (velocities && !points) return fail(NB_ERR_INVALID, "velocities given without points");
  NB_CUDA(cudaSetDevice(p->cfg.device));
  cudaStream_t st = (cudaStream_t)stream;
  const nb_pan_config& c = p->cfg;
  const int T = c.receding, T1 = T + 1;
  const bool with_dune = c.nrmp_max_num > 0 && points != nullptr && N > 0;  // pan.py:130
  if (p->differentiable && (p->adj_rec == nullptr || p->adj_iters < c.iter_num)) {  // (re)allocate the adjoint records for K iterations
    void* old[] = {p->adj_rec, p->adj_valid, p->adj_gs, p->adj_gu, p->adj_gd, p->adj_gtheta};
    for (void* o : old)
      if (o) cudaFree(o);
    p->adj_rec = nullptr; p->adj_valid = nullptr; p->adj_gs = p->adj_gu = p->adj_gd = p->adj_gtheta = nullptr;
    const size_t Bm = c.max_envs, Ks = c.iter_num > 0 ? c.iter_num : 1;
    NB_CUDA(dalloc(&p->adj_rec, Ks * Bm * nb::nrmp_adj_doubles(T, c.nrmp_max_num)));
    NB_CUDA(dalloc(&p->adj_valid, Ks * Bm));
    NB_CUDA(dalloc(&p->adj_gs, Bm * 3 * T1));
    NB_CUDA(dalloc(&p->adj_gu, Bm * 2 * T));
    NB_CUDA(dalloc(&p->adj_gd, Bm * T));
    NB_CUDA(dalloc(&p->adj_gtheta, Bm * 7));
    p->adj_iters = (int)Ks;
  }
  if (p->differentiable) NB_CUDA(cudaMemsetAsync(p->adj_valid, 0, (size_t)p->adj_iters * c.max_envs * sizeof(int32_t), st));
  if (plan && plan->n > 0) NB_CUDA(cudaStreamWaitEvent(st, plan->ev[0], 0));  // the small tensors travel ahead of chunk 0
  const int tb = 128, gb = (B + tb - 1) / tb;
  init_run_kernel<<<gb, tb, 0, st>>>(B, p->active, p->iters, p->status, p->min_dist, p->sel_count, p->warm_valid);
  ++g_launches;
  // the nominal trajectory lives in the output buffers and is updated in place every iteration
  NB_CUDA(cudaMemcpyAsync(out_s, nom_s, (size_t)B * 3 * T1 * sizeof(float), cudaMemcpyDeviceToDevice, st));
  NB_CUDA(cudaMemcpyAsync(out_u, nom_u, (size_t)B * 2 * T * sizeof(float), cudaMemcpyDeviceToDevice, st));
  NB_CUDA(cudaMemsetAsync(out_d, 0, (size_t)B * T * sizeof(float), st));
  // K iterations of {DUNE, NRMP} for the environments [lo, hi) on stream s
  auto run_range = [&](int lo, int hi, cudaStream_t s, int dune_cta_limit, int counter_slot, int k0, int k1) -> int {
    const int nb_ = hi - lo;
    const size_t T1s = (size_t)T1, Ms = (size_t)c.nrmp_max_num, Es = (size_t)(c.edge_dim > 0 ? c.edge_dim : 1);
    for (int k = k0; k < k1; ++k) {
      if (with_dune) {
        nb::DuneParams d{};
        d.weights = p->d_weights; d.nom_s = out_s + (size_t)lo * 3 * T1s; d.points = points + (size_t)lo * 2 * N;
        d.velocities = velocities ? velocities + (size_t)lo * 2 * N : nullptr;
        d.num_points = num_points ? num_points + lo : nullptr;
        d.active = p->active + lo;
        d.sel_mu = p->sel_mu + (size_t)lo * T1s * Ms * Es; d.sel_lam = p->sel_lam + (size_t)lo * T1s * Ms * 2;
        d.sel_pts = p->sel_pts + (size_t)lo * T1s * Ms * 2; d.sel_dist = p->sel_dist + (size_t)lo * T1s * Ms; d.sel_count = p->sel_count + lo;
        d.min_dist = p->min_dist + lo;
        d.B = nb_; d.N = N; d.T = T; d.M = c.nrmp_max_num; d.dt = (float)c.step_time; d.geo = p->geo;
        d.cand_idx = p->cand_idx + (size_t)lo * T1s * nb::kCandMax; d.cand_dt = p->cand_dt + (size_t)lo * T1s * nb::kCandMax;
        d.cand_cnt = p->cand_cnt + (size_t)lo * T1s; d.screen_stats = p->screen_stats; d.c_mu = p->c_mu;
        d.flag_list = p->flag_list + (size_t)lo * T1s; d.flag_count = p->flag_count + 4 * counter_slot; d.refine_list = p->refine_list + (size_t)2 * lo * T1s;
        d.screen_mma = p->screen_mma ? p->screen_shape : 0;
        d.skip_t0 = (k > 0 && p->dune_skip_t0) ? 1 : 0;  // the step-0 items of iteration 0 stand (DuneParams::skip_t0)
        if (k == 0 && plan && plan->n > 1) {
          // the first DUNE pass of this range chunk by chunk, each as soon as its points have landed: the upload of chunk c+1 overlaps the
          // work on chunk c (d describes the environments [lo, hi); a chunk's part of them is [clo, chi))
          for (int ch = 0; ch < plan->n; ++ch) {
            const int clo = plan->bound[ch] > lo ? plan->bound[ch] : lo, chi = plan->bound[ch + 1] < hi ? plan->bound[ch + 1] : hi;
            if (chi <= clo) continue;
            const size_t off = (size_t)(clo - lo);
            NB_CUDA(cudaStreamWaitEvent(s, plan->ev[ch], 0));
            nb::DuneParams dc = d;
            dc.nom_s = d.nom_s + off * 3 * T1s; dc.points = d.points + off * 2 * N;
            dc.velocities = d.velocities ? d.velocities + off * 2 * N : nullptr;
            dc.num_points = d.num_points ? d.num_points + off : nullptr;
            dc.active = d.active + off;
            dc.sel_mu = d.sel_mu + off * T1s * Ms * Es; dc.sel_lam = d.sel_lam + off * T1s * Ms * 2;
            dc.sel_pts = d.sel_pts + off * T1s * Ms * 2; dc.sel_dist = d.sel_dist + off * T1s * Ms; dc.sel_count = d.sel_count + off;
            dc.min_dist = d.min_dist + off;
            dc.B = chi - clo;
            dc.cand_idx = d.cand_idx + off * T1s * nb::kCandMax; dc.cand_dt = d.cand_dt + off * T1s * nb::kCandMax;
            dc.cand_cnt = d.cand_cnt + off * T1s;
            dc.flag_list = d.flag_list + off * T1s; dc.refine_list = d.refine_list + (size_t)2 * off * T1s;
            if (int rc = launch_dune(p, dc, s, dune_cta_limit)) return rc;
          }
        } else {
          if (int rc = launch_dune(p, d, s, dune_cta_limit)) return rc;
        }
      }
      nb::NrmpParams n{};
      n.nom_s = out_s + (size_t)lo * 3 * T1s; n.nom_u = out_u + (size_t)lo * 2 * T; n.ref_s = ref_s + (size_t)lo * 3 * T1s; n.ref_us = ref_us + (size_t)lo * T;
      if (with_dune) {
        n.sel_mu = p->sel_mu + (size_t)lo * T1s * Ms * Es; n.sel_lam = p->sel_lam + (size_t)lo * T1s * Ms * 2;
        n.sel_pts = p->sel_pts + (size_t)lo * T1s * Ms * 2; n.sel_count = p->sel_count + lo;
      }
      n.out_s = out_s + (size_t)lo * 3 * T1s; n.out_u = out_u + (size_t)lo * 2 * T; n.out_d = out_d + (size_t)lo * T;
      n.status = p->status + lo; n.iters = p->iters + lo; n.active = p->active + lo; n.ipm_iters = p->ipm_it + lo;
      n.prev_s = p->prev_s + (size_t)lo * 3 * T1s; n.prev_u = p->prev_u + (size_t)lo * 2 * T;
      n.prev_mu = p->prev_mu + (size_t)lo * T1s * Ms * Es; n.prev_lam = p->prev_lam + (size_t)lo * T1s * Ms * 2;
      n.prev_count = p->prev_count + lo; n.prev_valid = p->prev_valid + lo;
      if (p->differentiable && p->adj_rec && k < p->adj_iters) {
        n.adj_save = p->adj_rec + ((size_t)k * c.max_envs + lo) * nb::nrmp_adj_doubles(T, c.nrmp_max_num);
        n.adj_valid = p->adj_valid + (size_t)k * c.max_envs + lo;
      }
      if (p->nrmp_warm) {
        n.warm = p->warm + (size_t)lo * nb::nrmp_warm_floats(T, c.nrmp_max_num);
        n.warm_valid = p->warm_valid + lo;
      }
      n.B = nb_;
      if (int rc = launch_nrmp(p, n, s, counter_slot)) return rc;
    }
    return NB_OK;
  };
  const int parts = (p->overlap > 1 && with_dune && B >= 64 * p->overlap) ? p->overlap : 1;
  if (parts == 1) {
    if (int rc = run_range(0, B, st, 0, 0, 0, c.iter_num)) return rc;
  } else {
    // sub-batches on internal streams: the DUNE kernel of one part (issue / tensor / MUFU bound) shares the SMs with the
    // NRMP kernel of another (latency bound, few warps)
    NB_CUDA(cudaEventRecord(p->ev_fork, st));
    for (int i = 0; i < parts; ++i) NB_CUDA(cudaStreamWaitEvent(p->streams[i], p->ev_fork, 0));
    // enqueue order: iteration by iteration, alternating the streams (every sub-batch starts at once; NB_PAN_INTERLEAVE=0, a developer
    // switch, enqueues all K iterations of one sub-batch before the next: 19.29 vs 19.30-19.7 ms per C4 step)
    static int interleave = -1;
    if (interleave < 0) {
      const char* v = getenv("NB_PAN_INTERLEAVE");
      interleave = v ? atoi(v) : 1;
    }
    auto range_of = [&](int i, int& lo, int& hi) { lo = (int)((long long)B * i / parts); hi = (int)((long long)B * (i + 1) / parts); };
    if (interleave) {
      for (int k = 0; k < c.iter_num; ++k)
        for (int i = 0; i < parts; ++i) {
          int lo, hi;
          range_of(i, lo, hi);
          if (int rc = run_range(lo, hi, p->streams[i], 1, 1 + i, k, k + 1)) return rc;
        }
    } else {
      for (int i = 0; i < parts; ++i) {
        int lo, hi;
        range_of(i, lo, hi);
        if (int rc = run_range(lo, hi, p->streams[i], 1, 1 + i, 0, c.iter_num)) return rc;
      }
    }
    for (int i = 0; i < parts; ++i) {
      NB_CUDA(cudaEventRecord(p->ev_join[i], p->streams[i]));
      NB_CUDA(cudaStreamWaitEvent(st, p->ev_join[i], 0));
    }
  }
  finish_run_kernel<<<gb, tb, 0, st>>>(B, p->iters, p->status, p->min_dist, out_iters, out_status, out_min_distance);
  ++g_launches;
  NB_CUDA(cudaGetLastError());
  return NB_OK;
}
}  // namespace

namespace {
__global__ void adj_load_kernel(int n_s, int n_u, int n_d, int n_t, const float* gs, const float* gu, const float* gd, double* ds, double* du, double* dd,
                                double* dtheta) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n_s) ds[i] = gs ? (double)gs[i] : 0.0;
  if (i < n_u) du[i] = gu ? (double)gu[i] : 0.0;
  if (i < n_d) dd[i] = gd ? (double)gd[i] : 0.0;
  if (i < n_t) dtheta[i] = 0.0;
}
__global__ void adj_store_kernel(int n, const double* dtheta, float* out) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) out[i] = (float)dtheta[i];
}
}  // namespace

int nb_pan_backward(nb_pan_t* p, int32_t B, const float* ref_s, const float* ref_us, const float* grad_s, const float* grad_u, const float* grad_d,
                    float* grad_theta, void* stream) {
  if (int rc = check_forward_args(p, B, 0)) return rc;
  if (!p->differentiable || !p->adj_rec) return fail(NB_ERR_INVALID, "nb_pan_backward needs a forward in differentiable mode (NB_OPT_DIFFERENTIABLE = 1) first");
  if (!ref_s || !ref_us || !grad_theta) return fail(NB_ERR_INVALID, "null tensor argument");
  NB_CUDA(cudaSetDevice(p->cfg.device));
  cudaStream_t st = (cudaStream_t)stream;
  const nb_pan_config& c = p->cfg;
  const int T = c.receding, T1 = T + 1, nU = 2 * T;
  const int n_s = B * 3 * T1, n_u = B * 2 * T, n_d = B * T, n_t = B * 7;
  const int tb = 256, gb = (n_s + tb - 1) / tb;
  adj_load_kernel<<<gb, tb, 0, st>>>(n_s, n_u, n_d, n_t, grad_s, grad_u, grad_d, p->adj_gs, p->adj_gu, p->adj_gd, p->adj_gtheta);
  ++g_launches;
  nb::NrmpAdjParams a{};
  a.iters = p->iters; a.ref_s = ref_s; a.ref_us = ref_us;
  a.g_s = p->adj_gs; a.g_u = p->adj_gu; a.g_d = p->adj_gd; a.grad_theta = p->adj_gtheta;
  a.B = B; a.T = T; a.M = c.nrmp_max_num; a.kin = c.kinematics;
  for (int i = 0; i < 3; ++i) a.q[i] = c.q_s[i];
  a.p_u = c.p_u; a.d_min = c.d_min; a.bk = c.bk;
  const int wpc = 4;
  const size_t smem = (size_t)wpc * (((size_t)nU * (nU + 3)) / 2 + nU + 5 * T) * sizeof(double);
  if (smem > 48 * 1024) NB_CUDA(cudaFuncSetAttribute(nb::nrmp_adjoint_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  const int K = c.iter_num < p->adj_iters ? c.iter_num : p->adj_iters;
  for (int k = K - 1; k >= 0; --k) {  // reverse over the PAN iterations: the gradient w.r.t. para_s chains into the previous solve
    a.k = k;
    a.rec = p->adj_rec + (size_t)k * c.max_envs * nb::nrmp_adj_doubles(T, c.nrmp_max_num);
    a.rec_valid = p->adj_valid + (size_t)k * c.max_envs;
    nb::nrmp_adjoint_kernel<<<(B + wpc - 1) / wpc, wpc * 32, smem, st>>>(a);
    ++g_launches;
  }
  adj_store_kernel<<<(n_t + tb - 1) / tb, tb, 0, st>>>(n_t, p->adj_gtheta, grad_theta);
  ++g_launches;
  NB_CUDA(cudaGetLastError());
  return NB_OK;
}

int nb_pan_read_selection(nb_pan_t* p, int32_t B, float* sel_mu, float* sel_lam, float* sel_points, float* sel_distance,
                          int32_t* sel_count, void* stream) {
  if (int rc = check_forward_args(p, B, 0)) return rc;
  NB_CUDA(cudaSetDevice(p->cfg.device));
  cudaStream_t st = (cudaStream_t)stream;
  const size_t T1 = p->cfg.receding + 1, M = p->cfg.nrmp_max_num, E = p->cfg.edge_dim;
  if (sel_mu) NB_CUDA(cudaMemcpyAsync(sel_mu, p->sel_mu, (size_t)B * T1 * M * E * 4, cudaMemcpyDeviceToDevice, st));
  if (sel_lam) NB_CUDA(cudaMemcpyAsync(sel_lam, p->sel_lam, (size_t)B * T1 * M * 2 * 4, cudaMemcpyDeviceToDevice, st));
  if (sel_points) NB_CUDA(cudaMemcpyAsync(sel_points, p->sel_pts, (size_t)B * T1 * M * 2 * 4, cudaMemcpyDeviceToDevice, st));
  if (sel_distance) NB_CUDA(cudaMemcpyAsync(sel_distance, p->sel_dist, (size_t)B * T1 * M * 4, cudaMemcpyDeviceToDevice, st));
  if (sel_count) NB_CUDA(cudaMemcpyAsync(sel_count, p->sel_count, (size_t)B * 4, cudaMemcpyDeviceToDevice, st));
  return NB_OK;
}

int nb_pan_read_screen_stats(nb_pan_t* p, float* max_error_ratio, int32_t* counts, int32_t reset) {
  if (!p || !max_error_ratio || !counts) return fail(NB_ERR_INVALID, "nb_pan_read_screen_stats: null argument");
  if (!p->screen_stats) return fail(NB_ERR_INVALID, "handle was created in no_obs mode");
  NB_CUDA(cudaSetDevice(p->cfg.device));
  NB_CUDA(cudaDeviceSynchronize());
  unsigned h[4];
  NB_CUDA(cudaMemcpy(h, p->screen_stats, sizeof(h), cudaMemcpyDeviceToHost));
  memcpy(max_error_ratio, &h[0], 4);
  max_error_ratio[1] = p->c_mu;
  max_error_ratio[2] = p->screen_cal_ratio;
  counts[0] = (int32_t)h[1]; counts[1] = (int32_t)h[2]; counts[2] = (int32_t)h[3];
  if (reset) NB_CUDA(cudaMemset(p->screen_stats, 0, sizeof(h)));
  return NB_OK;
}

int nb_pan_read_diagnostics(nb_pan_t* p, int32_t B, int32_t* ipm_iterations, void* stream) {
  if (int rc = check_forward_args(p, B, 0)) return rc;
  NB_CUDA(cudaSetDevice(p->cfg.device));
  if (ipm_iterations) NB_CUDA(cudaMemcpyAsync(ipm_iterations, p->ipm_it, (size_t)B * 4, cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
  return NB_OK;
}

namespace {
// Upload of the host inputs into the handle's staging buffer on the copy stream, in env chunks, and the forward pass on `st` that
// consumes them chunk by chunk; outputs go to the device pointers given.  Nothing is synchronised here.
int pan_forward_from_host(nb_pan_t* p, int32_t B, int32_t N, const float* nom_s, const float* nom_u, const float* ref_s, const float* ref_us,
                          const float* points, const float* velocities, const int32_t* num_points, float* out_s, float* out_u, float* out_d,
                          float* out_min_distance, int32_t* out_iters, int32_t* out_status, cudaStream_t st) {
  const size_t T = p->cfg.receding, T1 = T + 1;
  const size_t n_s = (size_t)B * 3 * T1, n_u = (size_t)B * 2 * T, n_r = (size_t)B * T, n_p = (size_t)B * 2 * N;
  const size_t in_floats = 2 * n_s + n_u + n_r + 2 * n_p;
  if (!p->copy_stream) NB_CUDA(cudaStreamCreateWithFlags(&p->copy_stream, cudaStreamNonBlocking));
  if (!p->ev_inputs_free) NB_CUDA(cudaEventCreateWithFlags(&p->ev_inputs_free, cudaEventDisableTiming));
  for (int i = 0; i < nb_pan::kMaxChunks; ++i)
    if (!p->ev_chunk[i]) NB_CUDA(cudaEventCreateWithFlags(&p->ev_chunk[i], cudaEventDisableTiming));
  // whatever `st` still does with the staging buffer (the previous call) must be over before it is overwritten
  NB_CUDA(cudaEventRecord(p->ev_inputs_free, st));
  NB_CUDA(cudaStreamWaitEvent(p->copy_stream, p->ev_inputs_free, 0));
  if (in_floats > p->h_in_floats) {
    NB_CUDA(cudaStreamSynchronize(p->copy_stream));
    if (p->h_in) cudaFree(p->h_in);
    p->h_in = nullptr; p->h_in_floats = 0;
    NB_CUDA(dalloc(&p->h_in, in_floats));
    p->h_in_floats = in_floats;
  }
  if (!p->h_np) NB_CUDA(dalloc(&p->h_np, (size_t)p->cfg.max_envs));
  float* d = p->h_in;
  float* d_nom_s = d; d += n_s;
  float* d_ref_s = d; d += n_s;
  float* d_nom_u = d; d += n_u;
  float* d_ref_us = d; d += n_r;
  float* d_pts = d; d += n_p;
  float* d_vel = d;
  cudaStream_t cs = p->copy_stream;
  auto h2d = [&](void* dst, const void* src, size_t bytes) { return cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, cs); };
  NB_CUDA(h2d(d_nom_s, nom_s, n_s * 4));
  NB_CUDA(h2d(d_ref_s, ref_s, n_s * 4));
  NB_CUDA(h2d(d_nom_u, nom_u, n_u * 4));
  NB_CUDA(h2d(d_ref_us, ref_us, n_r * 4));
  if (num_points) NB_CUDA(h2d(p->h_np, num_points, (size_t)B * 4));
  const bool with_pts = points && N > 0;
  ChunkPlan plan;
  plan.n = (with_pts && B >= 64 * p->h2d_chunks) ? p->h2d_chunks : 1;
  if (with_pts && p->overlap > 1 && B >= 64 * p->overlap) {  // sub-batches on internal streams: chunk boundaries that contain theirs
    plan.n = p->overlap * (B >= 128 * p->overlap ? 2 : 1);
    if (plan.n > nb_pan::kMaxChunks) plan.n = p->overlap;
  }
  for (int c = 0; c <= plan.n; ++c) plan.bound[c] = (int)((long long)B * c / plan.n);
  for (int c = 0; c < plan.n; ++c) {
    const size_t lo = (size_t)plan.bound[c] * 2 * N, cnt = (size_t)(plan.bound[c + 1] - plan.bound[c]) * 2 * N;
    if (with_pts && cnt) NB_CUDA(h2d(d_pts + lo, points + lo, cnt * 4));
    if (with_pts && velocities && cnt) NB_CUDA(h2d(d_vel + lo, velocities + lo, cnt * 4));
    plan.ev[c] = p->ev_chunk[c];
    NB_CUDA(cudaEventRecord(plan.ev[c], cs));
  }
  return pan_forward_impl(p, B, N, d_nom_s, d_nom_u, d_ref_s, d_ref_us, with_pts ? d_pts : nullptr, (with_pts && velocities) ? d_vel : nullptr,
                          num_points ? p->h_np : nullptr, out_s, out_u, out_d, out_min_distance, out_iters, out_status, st, &plan);
}
}  // namespace

int nb_pan_forward_h2d(nb_pan_t* p, int32_t B, int32_t N, const float* nom_s, const float* nom_u, const float* ref_s, const float* ref_us,
                       const float* points, const float* velocities, const int32_t* num_points, float* out_s, float* out_u, float* out_d,
                       float* out_min_distance, int32_t* out_iters, int32_t* out_status, void* stream) {
  if (int rc = check_forward_args(p, B, N)) return rc;
  if (!nom_s || !nom_u || !ref_s || !ref_us || !out_s || !out_u || !out_d) return fail(NB_ERR_INVALID, "null tensor argument");
  NB_CUDA(cudaSetDevice(p->cfg.device));
  return pan_forward_from_host(p, B, N, nom_s, nom_u, ref_s, ref_us, points, velocities, num_points, out_s, out_u, out_d, out_min_distance, out_iters,
                               out_status, (cudaStream_t)stream);
}

int nb_pan_forward_host(nb_pan_t* p, int32_t B, int32_t N, const float* nom_s, const float* nom_u, const float* ref_s,
                        const float* ref_us, const float* points, const float* velocities, const int32_t* num_points, float* out_s,
                        float* out_u, float* out_d, float* out_min_distance, int32_t* out_iters, int32_t* out_status, void* stream) {
  if (int rc = check_forward_args(p, B, N)) return rc;
  if (!nom_s || !nom_u || !ref_s || !ref_us || !out_s || !out_u || !out_d) return fail(NB_ERR_INVALID, "null tensor argument");
  NB_CUDA(cudaSetDevice(p->cfg.device));
  cudaStream_t st = (cudaStream_t)stream;
  const size_t T = p->cfg.receding, T1 = T + 1;
  const size_t n_s = (size_t)B * 3 * T1, n_u = (size_t)B * 2 * T, n_r = (size_t)B * T;
  const size_t out_floats = n_s + n_u + n_r + (size_t)B;
  if (out_floats > p->h_out_floats) {
    if (p->h_out) cudaFree(p->h_out);
    p->h_out = nullptr; p->h_out_floats = 0;
    NB_CUDA(dalloc(&p->h_out, out_floats));
    p->h_out_floats = out_floats;
  }
  if (!p->h_io) NB_CUDA(dalloc(&p->h_io, 2 * (size_t)p->cfg.max_envs));
  float* o = p->h_out;
  float* o_s = o; o += n_s;
  float* o_u = o; o += n_u;
  float* o_d = o; o += n_r;
  float* o_md = o;
  int rc = pan_forward_from_host(p, B, N, nom_s, nom_u, ref_s, ref_us, points, velocities, num_points, o_s, o_u, o_d, o_md, p->h_io,
                                 p->h_io + p->cfg.max_envs, st);
  if (rc) return rc;
  auto d2h = [&](void* dst, const void* src, size_t bytes) { return cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToHost, st); };
  NB_CUDA(d2h(out_s, o_s, n_s * 4));
  NB_CUDA(d2h(out_u, o_u, n_u * 4));
  NB_CUDA(d2h(out_d, o_d, n_r * 4));
  if (out_min_distance) NB_CUDA(d2h(out_min_distance, o_md, (size_t)B * 4));
  if (out_iters) NB_CUDA(d2h(out_iters, p->h_io, (size_t)B * 4));
  if (out_status) NB_CUDA(d2h(out_status, p->h_io + p->cfg.max_envs, (size_t)B * 4));
  NB_CUDA(cudaStreamSynchronize(st));
  return NB_OK;
}

int nb_scan_to_points(int32_t B, int32_t R, const float* ranges, const float* velocity, const double* states,
                      const nb_scan_config* cfg, int32_t max_points, float* points, float* velocities_out,
                      int32_t* counts, void* stream) {
  if (!cfg || !ranges || !states || !points || !counts) return fail(NB_ERR_INVALID, "nb_scan_to_points: null argument");
  if (B < 0 || R < 1 || max_points < 1) return fail(NB_ERR_INVALID, "nb_scan_to_points: B=%d R=%d max_points=%d", B, R, max_points);
  if (cfg->down_sample < 1) return fail(NB_ERR_INVALID, "down_sample must be >= 1 (got %d)", cfg->down_sample);
  if ((size_t)R * sizeof(int32_t) > 200 * 1024) return fail(NB_ERR_CAPACITY, "R=%d beams exceed the shared-memory list (51200)", R);
  if (B == 0) return NB_OK;
  nb::ScanParams prm;
  prm.B = B; prm.R = R; prm.max_points = max_points;
  prm.ranges = ranges; prm.velocity = velocity; prm.states = states;
  prm.angle_min = cfg->angle_min; prm.angle_max = cfg->angle_max; prm.range_min = cfg->range_min; prm.range_max = cfg->range_max;
  prm.off_x = cfg->scan_offset[0]; prm.off_y = cfg->scan_offset[1]; prm.off_th = cfg->scan_offset[2];
  prm.angle_lo = cfg->angle_range[0]; prm.angle_hi = cfg->angle_range[1];
  prm.down_sample = cfg->down_sample; prm.velocity_mode = cfg->velocity_mode ? 1 : 0;
  prm.points = points; prm.vel_out = velocities_out; prm.counts = counts;
  const size_t smem = (size_t)R * sizeof(int32_t);
  static const bool generic_only = getenv("NB_SCAN_GENERIC") != nullptr;  // developer switch: force the chunked kernel
  if (R <= nb::kScanMaxChunks * 1024 && !generic_only) {  // all ranges of a thread in registers, one barrier
    int threads = 128;
    while (threads * nb::kScanMaxChunks < R) threads *= 2;
    if (R >= 512 && threads < 256) threads = 256;
    nb::scan_to_points_fast_kernel<<<B, threads, smem, (cudaStream_t)stream>>>(prm);
  } else {
    if (smem > 48 * 1024) NB_CUDA(cudaFuncSetAttribute(nb::scan_to_points_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    nb::scan_to_points_kernel<<<B, 256, smem, (cudaStream_t)stream>>>(prm);
  }
  ++g_launches;
  NB_CUDA(cudaGetLastError());
  return NB_OK;
}

// ---- DUNE training (SURVEY 8f row 4) -------------------------------------------------------------------------------
int nb_dune_labels(int32_t E, const float* G, const float* h, int64_t n, const double* points, float* points_f32, float* mu, float* dist, void* stream) {
  if (E < 3 || E > nb::kMaxEdges || !G || !h) return fail(NB_ERR_INVALID, "nb_dune_labels: edge_dim must be in 3..%d and G, h given", nb::kMaxEdges);
  if (n < 0 || (n > 0 && (!points || !points_f32 || !mu || !dist))) return fail(NB_ERR_INVALID, "nb_dune_labels: null argument");
  if (n == 0) return NB_OK;
  nb::DuneLabelParams prm;
  prm.n = (int)n; prm.E = E;
  for (int e = 0; e < E; ++e) { prm.G[e][0] = G[2 * e]; prm.G[e][1] = G[2 * e + 1]; prm.h[e] = h[e]; }
  prm.points = points; prm.points_f32 = points_f32; prm.mu = mu; prm.dist = dist;
  nb::dune_label_kernel<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(prm);
  ++g_launches;
  NB_CUDA(cudaGetLastError());
  return NB_OK;
}

int nb_dune_train_create(int32_t E, const float* G, const float* h, const float* weights, int64_t n_weights, int32_t device, nb_dune_train_t** out) {
  if (!out || !G || !h || !weights) return fail(NB_ERR_INVALID, "nb_dune_train_create: null argument");
  *out = nullptr;
  if (E < 3 || E > nb::kMaxEdges) return fail(NB_ERR_INVALID, "edge_dim must be in 3..%d", nb::kMaxEdges);
  if (n_weights != nb::WeightLayout::count(E)) return fail(NB_ERR_INVALID, "expected %d weights for edge_dim %d", nb::WeightLayout::count(E), E);
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0 || device < 0 || device >= ndev)
    return fail(NB_ERR_NO_DEVICE, "no CUDA device available: neupan_b200 has no CPU fallback");
  NB_CUDA(cudaSetDevice(device));
  nb_dune_train* t = new (std::nothrow) nb_dune_train();
  if (!t) return fail(NB_ERR_INVALID, "out of host memory");
  t->E = E; t->device = device; t->n_weights = (int)n_weights;
  for (int e = 0; e < E; ++e) { t->G[e][0] = G[2 * e]; t->G[e][1] = G[2 * e + 1]; t->h[e] = h[e]; }
  cudaError_t e = dalloc(&t->d_weights, (size_t)n_weights);
  if (e == cudaSuccess) e = dalloc(&t->d_m, (size_t)n_weights);
  if (e == cudaSuccess) e = dalloc(&t->d_v, (size_t)n_weights);
  if (e == cudaSuccess) e = dalloc(&t->d_losses, (size_t)4);
  if (e == cudaSuccess) e = cudaMemcpy(t->d_weights, weights, (size_t)n_weights * sizeof(float), cudaMemcpyHostToDevice);
  if (e == cudaSuccess) e = cudaMemset(t->d_m, 0, (size_t)n_weights * sizeof(float));
  if (e == cudaSuccess) e = cudaMemset(t->d_v, 0, (size_t)n_weights * sizeof(float));
  if (e != cudaSuccess) {
    nb_dune_train_destroy(t);
    return fail(NB_ERR_CUDA, "nb_dune_train_create: %s", cudaGetErrorString(e));
  }
  *out = t;
  return NB_OK;
}

int nb_dune_train_destroy(nb_dune_train_t* t) {
  if (!t) return NB_OK;
  cudaSetDevice(t->device);
  void* bufs[] = {t->d_weights, t->d_m, t->d_v, t->d_thetas, t->d_losses};
  for (void* b : bufs)
    if (b) cudaFree(b);
  delete t;
  return NB_OK;
}

int nb_dune_train_epoch(nb_dune_train_t* t, const float* pts, const float* mu, const float* dist, int64_t n, int32_t batch, const float* thetas,
                        float lr, int32_t validate, double* losses, void* stream) {
  if (!t || !pts || !mu || !dist || !thetas || !losses) return fail(NB_ERR_INVALID, "nb_dune_train_epoch: null argument");
  if (n < 1 || batch < 1 || batch > nb::kTrainThreads) return fail(NB_ERR_INVALID, "nb_dune_train_epoch: n >= 1 and 1 <= batch_size <= %d required", nb::kTrainThreads);
  NB_CUDA(cudaSetDevice(t->device));
  cudaStream_t st = (cudaStream_t)stream;
  const size_t nbatch = (size_t)((n + batch - 1) / batch);
  if (nbatch > t->thetas_cap) {
    if (t->d_thetas) cudaFree(t->d_thetas);
    t->d_thetas = nullptr; t->thetas_cap = 0;
    NB_CUDA(dalloc(&t->d_thetas, nbatch));
    t->thetas_cap = nbatch;
  }
  NB_CUDA(cudaMemcpyAsync(t->d_thetas, thetas, nbatch * sizeof(float), cudaMemcpyHostToDevice, st));
  nb::DuneTrainParams prm;
  prm.pts = pts; prm.mu = mu; prm.dist = dist; prm.thetas = t->d_thetas;
  prm.weights = t->d_weights; prm.adam_m = t->d_m; prm.adam_v = t->d_v; prm.losses = t->d_losses;
  prm.n = (int)n; prm.batch = batch; prm.E = t->E; prm.validate = validate ? 1 : 0;
  prm.step0 = t->steps;
  prm.lr = lr; prm.beta1 = 0.9f; prm.beta2 = 0.999f; prm.eps = 1e-8f; prm.weight_decay = 1e-4f;  // Adam(lr, weight_decay=1e-4), dune_train.py:72
  for (int e = 0; e < nb::kMaxEdges; ++e) { prm.G[e][0] = t->G[e][0]; prm.G[e][1] = t->G[e][1]; prm.h[e] = t->h[e]; }
  const size_t smem = nb::dune_train_smem_bytes(t->E);
  NB_CUDA(cudaFuncSetAttribute(nb::dune_train_epoch_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  nb::dune_train_epoch_kernel<<<1, nb::kTrainThreads, smem, st>>>(prm);
  ++g_launches;
  NB_CUDA(cudaGetLastError());
  double sums[4];
  NB_CUDA(cudaMemcpyAsync(sums, t->d_losses, sizeof(sums), cudaMemcpyDeviceToHost, st));
  NB_CUDA(cudaStreamSynchronize(st));
  for (int i = 0; i < 4; ++i) losses[i] = sums[i] / (double)nbatch;  // mean over the batches, like train_one_epoch (:322-327)
  if (!validate) t->steps += (long long)nbatch;
  return NB_OK;
}

int nb_dune_train_get_weights(nb_dune_train_t* t, float* weights) {
  if (!t || !weights) return fail(NB_ERR_INVALID, "nb_dune_train_get_weights: null argument");
  NB_CUDA(cudaSetDevice(t->device));
  NB_CUDA(cudaMemcpy(weights, t->d_weights, (size_t)t->n_weights * sizeof(float), cudaMemcpyDeviceToHost));
  return NB_OK;
}

// ---- initial path (SURVEY 8f row 1) ---------------------------------------------------------------------------------
int nb_ipath_create(const nb_ipath_config* cfg, nb_ipath_t** out) {
  if (!cfg || !out) return fail(NB_ERR_INVALID, "nb_ipath_create: null argument");
  if (cfg->receding < 1 || cfg->receding > nb::kIpathMaxT) return fail(NB_ERR_INVALID, "receding = %d outside [1, %d]", cfg->receding, nb::kIpathMaxT);
  if (cfg->kinematics < 0 || cfg->kinematics > 2) return fail(NB_ERR_INVALID, "kinematics currently only supports diff, acker or omni");
  if (cfg->kinematics == NB_KIN_ACKER && !(cfg->wheelbase > 0)) return fail(NB_ERR_INVALID, "acker needs a positive wheelbase");
  if (cfg->max_envs < 1 || !(cfg->step_time > 0)) return fail(NB_ERR_INVALID, "max_envs / step_time must be positive");
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0 || cfg->device >= ndev)
    return fail(NB_ERR_NO_DEVICE, "no CUDA device available: neupan_b200 has no CPU fallback");
  NB_CUDA(cudaSetDevice(cfg->device));
  nb_ipath* p = new nb_ipath();
  p->cfg = *cfg;
  cudaError_t e = dalloc(&p->d_env_curve_begin, (size_t)cfg->max_envs + 1);
  if (e == cudaSuccess) e = dalloc(&p->d_interval, (size_t)cfg->max_envs);
  if (e == cudaSuccess) e = dalloc(&p->d_curve_index, (size_t)cfg->max_envs);
  if (e == cudaSuccess) e = dalloc(&p->d_point_index, (size_t)cfg->max_envs);
  if (e == cudaSuccess) e = dalloc(&p->d_arrive_flag, (size_t)cfg->max_envs);
  if (e != cudaSuccess) {
    nb_ipath_destroy(p);
    return fail(NB_ERR_CUDA, "nb_ipath_create: %s", cudaGetErrorString(e));
  }
  *out = p;
  return NB_OK;
}

int nb_ipath_destroy(nb_ipath_t* p) {
  if (!p) return NB_OK;
  cudaSetDevice(p->cfg.device);
  void* bufs[] = {p->d_pts, p->d_curve_begin, p->d_env_curve_begin, p->d_interval, p->d_curve_index, p->d_point_index, p->d_arrive_flag};
  for (void* b : bufs)
    if (b) cudaFree(b);
  delete p;
  return NB_OK;
}

int nb_ipath_reset_async(nb_ipath_t* p, void* stream) {
  if (!p) return fail(NB_ERR_INVALID, "nb_ipath_reset: null handle");
  NB_CUDA(cudaSetDevice(p->cfg.device));
  cudaStream_t st = (cudaStream_t)stream;
  NB_CUDA(cudaMemsetAsync(p->d_curve_index, 0, sizeof(int32_t) * p->cfg.max_envs, st));
  NB_CUDA(cudaMemsetAsync(p->d_point_index, 0, sizeof(int32_t) * p->cfg.max_envs, st));
  NB_CUDA(cudaMemsetAsync(p->d_arrive_flag, 0, sizeof(int32_t) * p->cfg.max_envs, st));
  return NB_OK;
}

int nb_ipath_reset(nb_ipath_t* p) {
  if (int rc = nb_ipath_reset_async(p, nullptr)) return rc;
  NB_CUDA(cudaStreamSynchronize(nullptr));
  return NB_OK;
}

int nb_ipath_set_paths(nb_ipath_t* p, int32_t B, const double* points, int64_t P, const int32_t* curve_begin, int32_t C,
                       const int32_t* env_curve_begin, const double* interval) {
  if (!p || !points || !curve_begin || !env_curve_begin || !interval) return fail(NB_ERR_INVALID, "nb_ipath_set_paths: null argument");
  if (B < 1 || B > p->cfg.max_envs) return fail(NB_ERR_CAPACITY, "B = %d outside [1, max_envs = %d]", B, p->cfg.max_envs);
  if (P < 1 || C < B) return fail(NB_ERR_INVALID, "every environment needs at least one curve with one point (P = %lld, C = %d)", (long long)P, C);
  if (env_curve_begin[0] != 0 || env_curve_begin[B] != C || curve_begin[0] != 0 || curve_begin[C] != P)
    return fail(NB_ERR_INVALID, "curve_begin / env_curve_begin do not cover the points");
  for (int b = 0; b < B; ++b)
    if (env_curve_begin[b + 1] <= env_curve_begin[b]) return fail(NB_ERR_INVALID, "environment %d has no curve", b);
  for (int c = 0; c < C; ++c)
    if (curve_begin[c + 1] <= curve_begin[c]) return fail(NB_ERR_INVALID, "curve %d is empty", c);
  NB_CUDA(cudaSetDevice(p->cfg.device));
  if (p->d_pts) cudaFree(p->d_pts);
  if (p->d_curve_begin) cudaFree(p->d_curve_begin);
  p->d_pts = nullptr; p->d_curve_begin = nullptr;
  NB_CUDA(dalloc(&p->d_pts, (size_t)P * 4));
  NB_CUDA(dalloc(&p->d_curve_begin, (size_t)C + 1));
  NB_CUDA(cudaMemcpy(p->d_pts, points, sizeof(double) * 4 * P, cudaMemcpyHostToDevice));
  NB_CUDA(cudaMemcpy(p->d_curve_begin, curve_begin, sizeof(int32_t) * (C + 1), cudaMemcpyHostToDevice));
  NB_CUDA(cudaMemcpy(p->d_env_curve_begin, env_curve_begin, sizeof(int32_t) * (B + 1), cudaMemcpyHostToDevice));
  NB_CUDA(cudaMemcpy(p->d_interval, interval, sizeof(double) * B, cudaMemcpyHostToDevice));
  p->B = B; p->P = P;
  return nb_ipath_reset(p);
}

int nb_ipath_step(nb_ipath_t* p, int32_t B, const double* states, const float* cur_vel, double ref_speed,
                  float* nom_s, float* nom_u, float* ref_s, float* ref_us, int32_t* arrived, void* stream) {
  if (!p || !states || !cur_vel || !nom_s || !nom_u || !ref_s || !ref_us || !arrived) return fail(NB_ERR_INVALID, "nb_ipath_step: null argument");
  if (!p->d_pts) return fail(NB_ERR_INVALID, "initial path is not set (nb_ipath_set_paths)");
  if (B != p->B) return fail(NB_ERR_INVALID, "B = %d but the paths were set for %d environments", B, p->B);
  NB_CUDA(cudaSetDevice(p->cfg.device));
  nb::IpathParams prm;
  prm.B = B; prm.T = p->cfg.receding; prm.kinematics = p->cfg.kinematics; prm.loop = p->cfg.loop;
  prm.ind_range = p->cfg.ind_range; prm.arrive_index_threshold = p->cfg.arrive_index_threshold;
  prm.dt = p->cfg.step_time; prm.L = p->cfg.wheelbase; prm.arrive_threshold = p->cfg.arrive_threshold; prm.close_threshold = p->cfg.close_threshold;
  prm.ref_speed = ref_speed;
  prm.pts = p->d_pts; prm.curve_begin = p->d_curve_begin; prm.env_curve_begin = p->d_env_curve_begin; prm.interval = p->d_interval;
  prm.curve_index = p->d_curve_index; prm.point_index = p->d_point_index; prm.arrive_flag = p->d_arrive_flag;
  prm.states = states; prm.cur_vel = cur_vel; prm.nom_s = nom_s; prm.nom_u = nom_u; prm.ref_s = ref_s; prm.ref_us = ref_us; prm.arrived = arrived;
  nb::ipath_step_kernel<<<(B + 63) / 64, 64, 0, (cudaStream_t)stream>>>(prm);
  ++g_launches;
  NB_CUDA(cudaGetLastError());
  return NB_OK;
}

int nb_ipath_read_state(nb_ipath_t* p, int32_t B, int32_t* curve_index, int32_t* point_index, int32_t* arrive_flag,
                        double* points_host, void* stream) {
  if (!p) return fail(NB_ERR_INVALID, "nb_ipath_read_state: null handle");
  if (B != p->B) return fail(NB_ERR_INVALID, "B = %d but the paths were set for %d environments", B, p->B);
  NB_CUDA(cudaSetDevice(p->cfg.device));
  cudaStream_t st = (cudaStream_t)stream;
  if (curve_index) NB_CUDA(cudaMemcpyAsync(curve_index, p->d_curve_index, sizeof(int32_t) * B, cudaMemcpyDeviceToDevice, st));
  if (point_index) NB_CUDA(cudaMemcpyAsync(point_index, p->d_point_index, sizeof(int32_t) * B, cudaMemcpyDeviceToDevice, st));
  if (arrive_flag) NB_CUDA(cudaMemcpyAsync(arrive_flag, p->d_arrive_flag, sizeof(int32_t) * B, cudaMemcpyDeviceToDevice, st));
  if (points_host) {
    NB_CUDA(cudaMemcpyAsync(points_host, p->d_pts, sizeof(double) * 4 * p->P, cudaMemcpyDeviceToHost, st));
    NB_CUDA(cudaStreamSynchronize(st));
  }
  return NB_OK;
}

}  // extern "C"
