// Translation unit of the tcgen05 DUNE kernel: host-side operand image + launcher.
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <vector>

#include "dune_tc_kernel.cuh"
#include "dune_tc8_kernel.cuh"
#include "dune_screen_kernel.cuh"
#include "dune_screen_mma_kernel.cuh"

namespace nb {

static inline void split_half_tc(float v, uint16_t& hi, uint16_t& lo) {
  const __half h = __float2half_rn(v);
  const __half l = __float2half_rn(v - __half2float(h));
  memcpy(&hi, &h, 2);
  memcpy(&lo, &l, 2);
}

// packed checkpoint (WeightLayout order, E outputs) -> TcImage bytes (canonical K-major / no-swizzle UMMA layout)
// returns flags: bit 0 = every tanh argument of the network is bounded by 30 in exp2 units (|LN(x)_j| <= sqrt(32)), which
// allows the kernel's shared-reciprocal tanh (ln_tanh_split<true>)
// screen = true: the image of the screening network (dune_screen_kernel.cuh): the same layout, but tanh is NOT folded into the
// following layer (the screen kernel applies MUFU.TANH itself) and the LayerNorm gain / offset are the checkpoint's plain values;
// only the hi halves of the weights are used.
int build_tc_image(const float* w, int E, std::vector<unsigned char>& out, bool screen) {
  using L = WeightLayout;
  using I = TcImage;
  out.assign(I::kBytes, 0);
  auto put = [&](size_t off, uint16_t v) { memcpy(out.data() + off, &v, 2); };
  // element (n, k) of a K-major operand with `lbo` bytes between the two 8-half K groups and `kstep` bytes per 16 of K
  auto at = [](int n, int k, int lbo, int kstep) { return (size_t)(k / 16) * kstep + ((k % 16) / 8) * lbo + (n / 8) * 128 + (n % 8) * 16 + (k % 8) * 2; };
  float* fl = reinterpret_cast<float*>(out.data() + I::kFloatOff);
  // the five dense layers: MLP.3, .5, .8, .10 and the head MLP.13 (E rows, zero padded to N = 32).
  // Layers fed by a tanh (MLP.3, MLP.8, MLP.13) receive r = 1/(exp(2y)+1) instead of tanh(y) = 1 - 2r:
  //   W tanh + b = (b + rowsum(W)) + (-2 W) r
  const int dense_w[5] = {L::W3, L::W5, L::W8, L::W10, L::W13}, dense_b[5] = {L::B3, L::B5, L::B8, L::B10, L::b13(E)};
  const int rows[5] = {32, 32, 32, 32, E};
  const bool after_tanh[5] = {!screen, false, !screen, false, !screen};
  // Layers that feed a LayerNorm (MLP.0 -> LN1, MLP.5 -> LN6, MLP.10 -> LN11) are CENTRED here: LN subtracts the mean over
  // the 32 outputs, which is linear, so W - colmean(W) and b - mean(b) deliver mean-free pre-activations for free.
  const bool before_ln[5] = {false, true, false, true, false};
  for (int l = 0; l < 5; ++l) {
    const size_t base = (size_t)l * I::kLayerStride;
    std::vector<double> W(32 * 32, 0.0), bv(32, 0.0);
    for (int n = 0; n < rows[l]; ++n) {
      double rowsum = 0.0;
      for (int k = 0; k < 32; ++k) {
        const double wv = (double)w[dense_w[l] + n * 32 + k];
        rowsum += wv;
        W[n * 32 + k] = after_tanh[l] ? -2.0 * wv : wv;
      }
      bv[n] = (double)w[dense_b[l] + n] + (after_tanh[l] ? rowsum : 0.0);
    }
    if (before_ln[l]) {
      for (int k = 0; k < 32; ++k) {
        double m = 0.0;
        for (int n = 0; n < 32; ++n) m += W[n * 32 + k];
        for (int n = 0; n < 32; ++n) W[n * 32 + k] -= m / 32;
      }
      double m = 0.0;
      for (int n = 0; n < 32; ++n) m += bv[n];
      for (int n = 0; n < 32; ++n) bv[n] -= m / 32;
    }
    for (int n = 0; n < 32; ++n) {
      for (int k = 0; k < 32; ++k) {
        uint16_t hi, lo;
        split_half_tc((float)W[n * 32 + k], hi, lo);
        put(base + at(n, k, 512, 1024), hi);
        put(base + 2048 + at(n, k, 512, 1024), lo);
      }
      fl[I::BH + 32 * l + n] = (float)bv[n];
    }
  }
  for (int m = 0; m < 128; ++m)  // ONES(m, 0..2) = 1.0h, K-major with 2048 B between the two 8-wide K groups
    for (int k = 0; k < 3; ++k) put(I::kOnesOff + (size_t)(m / 8) * 128 + (m % 8) * 16 + k * 2, 0x3C00);
  for (int l = 0; l < 5; ++l)    // BIASB[l](n, 0..2) = three fp16 pieces of the (folded) bias
    for (int n = 0; n < 32; ++n) {
      float rest = fl[I::BH + 32 * l + n];
      for (int k = 0; k < 3; ++k) {
        const __half h = __float2half_rn(rest);
        rest -= __half2float(h);
        uint16_t bits;
        memcpy(&bits, &h, 2);
        put(I::kBiasBOff + (size_t)l * 1024 + at(n, k, 512, 1024), bits);
      }
    }
  {  // layer 0 (2 -> 32), centred for LN1; both layouts (row-major for the first kernel, columns for the packed one)
    double mx = 0.0, my = 0.0, mb = 0.0;
    for (int j = 0; j < 32; ++j) { mx += w[L::W0 + 2 * j]; my += w[L::W0 + 2 * j + 1]; mb += w[L::B0 + j]; }
    for (int j = 0; j < 32; ++j) {
      fl[I::W0X + j] = (float)((double)w[L::W0 + 2 * j] - mx / 32);
      fl[I::W0Y + j] = (float)((double)w[L::W0 + 2 * j + 1] - my / 32);
      fl[I::W0 + 2 * j] = fl[I::W0X + j];
      fl[I::W0 + 2 * j + 1] = fl[I::W0Y + j];
      fl[I::B0 + j] = (float)((double)w[L::B0 + j] - mb / 32);
    }
  }
  const int g_src[3] = {L::G1, L::G6, L::G11}, b_src[3] = {L::BE1, L::BE6, L::BE11};
  const int g_dst[3] = {I::G1, I::G6, I::G11}, b_dst[3] = {I::BE1, I::BE6, I::BE11};
  for (int q = 0; q < 3; ++q)
    for (int i = 0; i < 32; ++i) {  // pre-multiplied by 2*log2(e): tanh(y) = 1 - 2/(exp2(2*log2(e)*y) + 1)
      const double sc = screen ? 1.0 : 2.8853900817779268;
      fl[g_dst[q] + i] = (float)((double)w[g_src[q] + i] * sc);
      fl[b_dst[q] + i] = (float)((double)w[b_src[q] + i] * sc);
    }
  double amax = 0.0;
  for (int q = 0; q < 3; ++q)
    for (int i = 0; i < 32; ++i) {
      const double a = std::fabs((double)fl[g_dst[q] + i]) * 5.6568542494923806 + std::fabs((double)fl[b_dst[q] + i]);  // sqrt(32)
      if (!(a <= amax)) amax = a;  // NaN-propagating max
    }
  return amax <= 30.0 ? 1 : 0;
}

int launch_dune_tc(const DuneParams& prm_in, const unsigned char* d_image, const unsigned char* d_screen_image, int image_flags, int variant, int sm_count,
                   int max_smem_optin, cudaStream_t st, char* err, size_t errlen) {
  DuneParams prm = prm_in;
  if (variant == 4) {
    // screening: (1) interval pass over all points, (2) exact evaluation of the candidates, (3) the exact kernel for the items the
    // screen could not narrow down to 32 candidates (below, with only_flagged)
    if (!d_screen_image || !prm.cand_idx || !prm.cand_cnt || !prm.cand_dt || !prm.screen_stats || !prm.flag_list || !prm.flag_count || !prm.refine_list) {
      snprintf(err, errlen, "screening buffers are not allocated");
      return -1;
    }
    const int items_ = prm.B * (prm.T + 1);
    const size_t pad4 = (size_t)(233472 / 5) - 2048 + 512;  // never more than 4 CTAs (128 TMEM columns each) per SM
    size_t smem_s = dune_screen_smem_bytes(prm.N, prm.M);
    if ((long long)smem_s > max_smem_optin) {
      snprintf(err, errlen, "N=%d needs %zu B of shared memory (limit %d)", prm.N, smem_s, max_smem_optin);
      return -3;
    }
    if (smem_s < pad4) smem_s = pad4;
    size_t smem_r = TcImage::kBytes + 64;
    if (smem_r < pad4) smem_r = pad4;
    int per_s = (int)(233472 / (smem_s + 2048));
    per_s = per_s > 4 ? 4 : (per_s < 1 ? 1 : per_s);
    const int screen_mma = prm.screen_mma;
    cudaError_t e = cudaMemsetAsync(prm.flag_count, 0, 4 * sizeof(int32_t), st);
    // one warp per item where the launch has at least one item per resident warp; smaller batches keep the 4 warps of a CTA on one item
    // (an item's tiles would otherwise run one after another on a single warp while most warp slots idle).  2 / 3 force the CTA / warp shape.
    const int warp_slots = sm_count * (prm.N <= 512 ? NB_SMMA_BLOCKS : 4) * 4;
    const bool per_warp = screen_mma == 3 || (screen_mma != 2 && items_ >= warp_slots);
    const size_t smem_m = per_warp ? dune_screen_warp_smem_bytes(prm.N) : dune_screen_mma_smem_bytes(prm.N, prm.M);
    if (screen_mma && prm.N <= 1024 && (long long)smem_m <= max_smem_optin) {  // larger clouds: the tcgen05 screen kernel (key arrays in shared memory)
      // no TMEM in these kernels: residency is whatever registers and shared memory admit
      auto go = [&](auto kern, int& per_m, size_t& per_m_smem, int work) {
        if (e == cudaSuccess) e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_m);
        if (e == cudaSuccess && (per_m < 0 || per_m_smem != smem_m)) {
          e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_m, kern, 128, smem_m);
          per_m_smem = smem_m;
          if (per_m < 1) per_m = 1;
        }
        if (e == cudaSuccess) {
          static int cap = -1;  // NB_SCREEN_CTA_CAP (developer switch): fewer CTAs per SM, to leave room for a kernel of another stream (NB_OPT_OVERLAP)
          if (cap < 0) {
            const char* v = getenv("NB_SCREEN_CTA_CAP");
            cap = v ? atoi(v) : 0;
          }
          int grid = sm_count * ((cap > 0 && cap < per_m) ? cap : per_m);
          if (grid > work) grid = work;
          kern<<<grid, 128, smem_m, st>>>(prm, d_screen_image);
          e = cudaGetLastError();
        }
      };
      static int per4 = -1, per8 = -1, perw4 = -1, perw8 = -1;
      static size_t smem4 = 0, smem8 = 0, smemw4 = 0, smemw8 = 0;
      const int warp_ctas = (items_ + 3) / 4;  // one item per warp at a time
      if (per_warp && prm.N <= 512) go(dune_screen_warp_kernel<4>, perw4, smemw4, warp_ctas);
      else if (per_warp) go(dune_screen_warp_kernel<8>, perw8, smemw8, warp_ctas);
      else if (prm.N <= 512) go(dune_screen_mma_kernel<4>, per4, smem4, items_);
      else go(dune_screen_mma_kernel<8>, per8, smem8, items_);
    } else {
      if (e == cudaSuccess) e = cudaFuncSetAttribute(dune_screen_kernel<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_s);
      if (e == cudaSuccess) {
        int grid = sm_count * per_s;
        if (grid > items_) grid = items_;
        dune_screen_kernel<0><<<grid, 128, smem_s, st>>>(prm, d_screen_image);
        e = cudaGetLastError();
      }
    }
    const bool fast_r = (image_flags & 1) != 0;
    if (e == cudaSuccess) e = fast_r ? cudaFuncSetAttribute(dune_refine_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_r)
                                      : cudaFuncSetAttribute(dune_refine_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_r);
    if (e == cudaSuccess) {
      int grid = sm_count * 4;  // the number of work units is only known on the device: a persistent grid sized for the worst case
      const int groups = (items_ + 7) / 8;
      if (grid > groups) grid = groups;
      if (fast_r) dune_refine_kernel<true><<<grid, 128, smem_r, st>>>(prm, d_image);
      else dune_refine_kernel<false><<<grid, 128, smem_r, st>>>(prm, d_image);
      e = cudaGetLastError();
    }
    if (e != cudaSuccess) {
      snprintf(err, errlen, "dune screen / refine launch failed: %s", cudaGetErrorString(e));
      return -2;
    }
    prm.only_flagged = 1;
    variant = 2;
  }
  size_t smem = variant == 3 ? dune_tc8_smem_bytes(prm.N, prm.geo.E, prm.M) : dune_tc_smem_bytes(prm.N, prm.geo.E, prm.M);
  if ((long long)smem > max_smem_optin) {
    snprintf(err, errlen, "N=%d needs %zu B of shared memory (limit %d)", prm.N, smem, max_smem_optin);
    return -3;
  }
  const int items = prm.B * (prm.T + 1);
  static int force = -1;  // NB_DUNE_TC: developer switch, 1 = first (single-slot, scalar math) kernel, 2 = mbarrier hand-off
  if (force < 0) {
    const char* v = getenv("NB_DUNE_TC");
    force = v ? atoi(v) : 0;
  }
  static int blocks8 = -1;  // NB_DUNE_TC8_BLOCKS: CTAs per SM of the 8-warp kernel (3: <= 85 registers, 4: <= 64 registers)
  if (blocks8 < 0) {
    const char* v = getenv("NB_DUNE_TC8_BLOCKS");
    blocks8 = v ? atoi(v) : 3;
    if (blocks8 != 4) blocks8 = 3;
  }
  const bool single = force == 1 && variant != 3;
  const bool barrier_sync = force != 2;  // default: block barrier between operand stores and MMAs (2.19 ms vs 2.29 ms with the mbarrier hand-off)
  // TMEM columns are held by a CTA for its whole (persistent) lifetime: 512 / columns-per-CTA CTAs may share an SM, one
  // more would sit in tcgen05.alloc until another CTA exits, and the block scheduler knows nothing about TMEM
  // (observed: a 5th CTA with 128 columns landing on an SM turned 2.7 ms into 4.3 ms per launch).  The shared-memory
  // request is therefore padded so that never more CTAs fit than registers and TMEM admit.
  const int want = variant == 3 ? blocks8 : (single ? 5 : 4);  // two-slot kernel: 128 columns -> 4 CTAs;  single slot: 64 columns, 96 registers -> 5 CTAs
  // smallest request that keeps a (want+1)-th CTA out (anything larger only shrinks the L1 cache: 44 KB instead of 38 KB
  // per CTA cost 2.49 -> 3.50 ms per launch of the single-slot kernel)
  const size_t pad = (size_t)(233472 / (want + 1)) - 2048 + 512;
  if (smem < pad) smem = pad;
  const bool fast = (image_flags & 1) != 0 && force != 4;  // NB_DUNE_TC=4: plain reciprocals
  auto run = [&](auto kern, int threads) -> cudaError_t {
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    int per_sm = (int)(233472 / (smem + 2048));
    if (per_sm > want) per_sm = want;
    if (per_sm < 1) per_sm = 1;
    int grid = sm_count * per_sm;
    if (grid > items) grid = items;
    kern<<<grid, threads, smem, st>>>(prm, d_image);
    return cudaGetLastError();
  };
  cudaError_t e;
  if (variant == 3) {
    if (blocks8 == 4) e = fast ? run(dune_tc8_kernel<true, 4>, 256) : run(dune_tc8_kernel<false, 4>, 256);
    else e = fast ? run(dune_tc8_kernel<true, 3>, 256) : run(dune_tc8_kernel<false, 3>, 256);
  } else if (single) e = run(dune_tc_kernel, 128);
  else if (barrier_sync) e = fast ? run(dune_tcp_kernel<0, true>, 128) : run(dune_tcp_kernel<0, false>, 128);
  else e = fast ? run(dune_tcp_kernel<1, true>, 128) : run(dune_tcp_kernel<1, false>, 128);
  if (e != cudaSuccess) {
    snprintf(err, errlen, "dune_tc kernel launch failed: %s", cudaGetErrorString(e));
    return -2;
  }
  return 0;
}

}  // namespace nb
