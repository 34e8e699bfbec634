// Marching-plane weight gradient, one (32 input channels x 32 output channels) block per CTA column:
//   KT = 3: 3x3x3 s1 p1 convs            dW[kd,kh,kw][ci][co] = sum_v X[v + (kd,kh,kw) - 1][ci] * dY[v][co]
//   KT = 2: the 4x4x4 s2 p1 PatchGAN stem on its parity-planar space-to-depth source: for input parity
//           (pd,ph,pw) the conv is a 2x2x2-tap conv on the half-resolution grid,
//           dW[2s+1-p][ci][co] = sum_o X2[o + s + (p ? -1 : 0)][parity p][ci] * dY[o][co],   s in {0,1}^3.
//
// igemm_wgrad_kernel handles one depth tap per CTA with N = 32 (smem-bound UMMA, X planes re-loaded per
// tap). Here the depth taps are folded into N by shifting dY instead of X: for one X plane p,
//
//     D[kh][(kw, ci)][(j, co)] += sum_{h,w} X[p, h+kh, w+kw, ci] * dY[p + doff + j, h, w, co],   depth tap = KT-1-j
//
// so ONE UMMA (M = 128 = 4 kw-atoms x 32 ci, N = KT*32 = KT dY planes x 32 co, K = 16 voxels) covers
// KT*KT taps. Both operands are MN-major views of the tiles exactly as TMA delivered them:
//   A atoms (kw) are one halo row apart (LBO = 64 B), B atoms (j) are one dY plane apart
//   (LBO = 8 KB): the dY planes live in a ring whose first KT-1 slots are mirrored behind the last so
//   that KT consecutive planes are always contiguous. Out-of-range dY planes are out-of-bounds TMA
//   loads (zero fill) -- the conv padding in depth.
// A CTA marches along d through its share of (n, h-tile, w-tile, d-segment) items and keeps the KT
// kh accumulators (KT x KT*32 TMEM columns) for its whole lifetime (split-K over CTAs), then writes one
// fp32 partial record; wgrad_reduce_kernel sums the records in a fixed order.
#pragma once
#include "igemm_fwd.cuh"
#include "deferred_tile.cuh"

namespace ub {

struct WgradMarchParams {
  CUtensorMap tm_x[2];      // box (32, 8+KT-1, 16+KT-1, 1, 1)
  CUtensorMap tm_dy;        // box (32, 8, 16, 1, 1)
  int n_chunks_src0, n_chunks_total;
  int Nb, D, H, W;          // the dY grid (KT = 2: the half-resolution output grid)
  int tiles_w, tiles_h, nseg, seg_len;
  int ci_total;             // padded input channels (partial pitch)
  int co_total, n_cotiles;  // padded output channels, co_total / 32
  int ntaps;                // taps of the partial record (27 / 64)
  float* partial;           // [gridDim.x][ntaps][ci_total][co_total]
  // kTf (KT = 3): source 0 (one 32-channel chunk) is the raw fp16 output y of a conv -> norm block and `tf` its
  // deferred activation: the four epilogue warps, idle until the end, rewrite every X halo plane of chunk 0 in
  // shared memory (deferred_tile.cuh) before the MMA thread reads it.
  NormActArgs tf;
};

constexpr int kWmXStages = 4, kWmXBytes = 12288;
constexpr int kWmYSlots = 8, kWmYBytes = 8192;   // + KT-1 mirror slots

// Warps 0-3 epilogue (kTf: operand transform first), 4 TMA producer of the X planes, 5 MMA issuer, 6 TMA producer of the
// dY planes (two producer threads: the stem form has 16 UMMAs of 48 cycles per plane against two to three TMA boxes),
// 7 second MMA issuer: warp 5 takes the kh groups [0, KT - 1), warp 7 the last one (KT = 2: one each). The two issuers own
// DIFFERENT kh accumulators -- nothing orders them against each other, unlike two threads accumulating into one
// accumulator -- and walk the same barriers; one's per-plane hand-off (waits, fence, commits) runs while the other's UMMAs
// are in the pipe (the marching kernels spend ~450 cycles per plane on it beside UMMAs that run at their isolated rate,
// profiles/r02j_march_mma_ablation.txt). One issuer measured slower (profiles/r02j_wgrad_mma2.txt), removed.
constexpr int kWgradMarchThreads = kIgemmThreads + 64;
template <int KT, bool kTf>
__global__ void __launch_bounds__(kWgradMarchThreads, 1)
wgrad_march_kernel(const __grid_constant__ WgradMarchParams P) {
  static_assert(!kTf || KT == 3, "the operand transform serves the 3x3x3 layers");
  constexpr int BW = 8 + KT - 1, BH = 16 + KT - 1;     // halo box
  constexpr int NN = KT * 32;                          // UMMA N
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* sm = smem_raw + (base - smem_u32(smem_raw));
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t x_base = base;
  const uint32_t y_base = x_base + kWmXStages * kWmXBytes;
  const uint32_t bar_base = y_base + (kWmYSlots + KT - 1) * kWmYBytes;
  const uint32_t x_full = bar_base, x_empty = x_full + 8 * kWmXStages, y_full = x_empty + 8 * kWmXStages,
                 y_empty = y_full + 8 * kWmYSlots, acc_full = y_empty + 8 * kWmYSlots, x_ready = acc_full + 8;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(sm + (x_ready + 8 * kWmXStages - base));

  // blockIdx.y = ((parity) * chunks + chunk) * cotiles + cot   (parity only for KT = 2)
  int by = blockIdx.y;
  const int cot = by % P.n_cotiles; by /= P.n_cotiles;
  const int chunk = by % P.n_chunks_total; by /= P.n_chunks_total;
  const int parity = KT == 2 ? by : 0;
  const int pd = (parity >> 2) & 1, ph = (parity >> 1) & 1, pw = parity & 1;
  const bool s1 = chunk >= P.n_chunks_src0;
  const int c0 = (s1 ? chunk - P.n_chunks_src0 : chunk) * 32;
  const bool tf_cta = kTf && chunk == 0;     // this CTA's X planes are y planes of the deferred source
  // X tile origin relative to the dY tile origin, and the dY plane paired with atom j of X plane p: p + doff + j
  const int xoff_w = KT == 3 ? -1 : (pw ? -1 : 0), xoff_h = KT == 3 ? -1 : (ph ? -1 : 0);
  const int doff = KT == 3 ? -1 : pd - 1;
  // contiguous range of items for this CTA
  const int items = P.Nb * P.tiles_h * P.tiles_w * P.nseg;
  const int per = (items + gridDim.x - 1) / gridDim.x;
  const int i_begin = blockIdx.x * per;
  int i_end = i_begin + per; if (i_end > items) i_end = items;

  if (threadIdx.x == 0) {
    // both issuers commit the stage / slot / accumulator barriers
    for (int i = 0; i < kWmXStages; ++i) {
      mbar_init(x_full + 8 * i, 1); mbar_init(x_empty + 8 * i, 2); mbar_init(x_ready + 8 * i, 1);
    }
    for (int i = 0; i < kWmYSlots; ++i) { mbar_init(y_full + 8 * i, 1); mbar_init(y_empty + 8 * i, 2); }
    mbar_init(acc_full, 2);
    fence_mbar_init();
  }
  if (warp == 4 && lane == 0) tma_prefetch_desc(&P.tm_x[s1 ? 1 : 0]);
  if (warp == 6 && lane == 0) tma_prefetch_desc(&P.tm_dy);
  if (warp == 5) tmem_alloc_rt(smem_u32(tmem_slot), 512);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tmem_slot;

  if (warp == 4) {
    // =========================== TMA producer: X planes ===========================
    if (lane == 0) {
      const CUtensorMap* tmx = &P.tm_x[s1 ? 1 : 0];
      int xs = 0; uint32_t xp = 0;    // X ring
      for (int it = i_begin; it < i_end; ++it) {
        int t = it;
        const int seg = t % P.nseg; t /= P.nseg;
        const int w0 = (t % P.tiles_w) * 8; t /= P.tiles_w;
        const int h0 = (t % P.tiles_h) * 16; t /= P.tiles_h;
        const int nb = t;
        const int d0 = seg * P.seg_len;
        int d1 = d0 + P.seg_len; if (d1 > P.D) d1 = P.D;
        for (int p = d0; p < d1; ++p) {
          mbar_wait(x_empty + 8 * xs, xp ^ 1);
          mbar_expect_tx(x_full + 8 * xs, BW * BH * 64);
          tma_load_5d(x_base + xs * kWmXBytes, tmx, x_full + 8 * xs, c0, w0 + xoff_w, h0 + xoff_h, p,
                      KT == 2 ? nb * 8 + parity : nb);
          if (++xs == kWmXStages) { xs = 0; xp ^= 1; }
        }
      }
    }
    __syncwarp();
  } else if (warp == 6) {
    // =========================== TMA producer: dY planes ===========================
    if (lane == 0) {
      int ys = 0; uint32_t yp = 0;    // dY ring
      auto load_dy = [&](int q, int nb, int h0, int w0) {
        mbar_wait(y_empty + 8 * ys, yp ^ 1);
        const bool mirror = ys < KT - 1;
        mbar_expect_tx(y_full + 8 * ys, mirror ? 2 * kWmYBytes : kWmYBytes);
        tma_load_5d(y_base + ys * kWmYBytes, &P.tm_dy, y_full + 8 * ys, cot * 32, w0, h0, q, nb);
        if (mirror) tma_load_5d(y_base + (kWmYSlots + ys) * kWmYBytes, &P.tm_dy, y_full + 8 * ys, cot * 32, w0, h0, q, nb);
        if (++ys == kWmYSlots) { ys = 0; yp ^= 1; }
      };
      for (int it = i_begin; it < i_end; ++it) {
        int t = it;
        const int seg = t % P.nseg; t /= P.nseg;
        const int w0 = (t % P.tiles_w) * 8; t /= P.tiles_w;
        const int h0 = (t % P.tiles_h) * 16; t /= P.tiles_h;
        const int nb = t;
        const int d0 = seg * P.seg_len;
        int d1 = d0 + P.seg_len; if (d1 > P.D) d1 = P.D;
        // the item owns X planes [d0, d1) and pairs each with the dY planes p+doff .. p+doff+KT-1; planes
        // outside [0, D) are out-of-bounds TMA coordinates (zero fill = the conv padding in depth)
#pragma unroll
        for (int j = 0; j < KT - 1; ++j) load_dy(d0 + doff + j, nb, h0, w0);
        for (int p = d0; p < d1; ++p) load_dy(p + doff + KT - 1, nb, h0, w0);
      }
    }
    __syncwarp();
  } else if (warp == 5 || warp == 7) {
    // =========================== MMA issuer(s) ===========================
    const int kh_begin = warp == 7 ? KT - 1 : 0;
    const int kh_end = warp == 5 ? KT - 1 : KT;
    const uint32_t idesc = make_idesc_bf16(128, NN, 1, 1);
    const uint64_t a_desc0 = make_smem_desc(0, /*lbo: next kw atom = next halo row*/ 64, /*sbo: next h row*/ BW * 64, SWZ_64B);
    const uint64_t b_desc0 = make_smem_desc(0, /*lbo: next dY plane*/ kWmYBytes, /*sbo: next 8 voxel rows*/ 8 * 64, SWZ_64B);
    const uint32_t a_hi = (uint32_t)(a_desc0 >> 32), b_hi = (uint32_t)(b_desc0 >> 32);
    const uint32_t a_lo0 = (uint32_t)a_desc0, b_lo0 = (uint32_t)b_desc0;
    const bool leader = elect_one();
    int xs = 0; uint32_t xp = 0;
    int ys = 0; uint32_t yp = 0;       // slot / phase of the OLDEST of the KT live dY planes
    uint32_t first = 1;
    for (int it = i_begin; it < i_end; ++it) {
      const int seg = it % P.nseg;
      const int d0 = seg * P.seg_len;
      int d1 = d0 + P.seg_len; if (d1 > P.D) d1 = P.D;
      // the first KT-1 dY planes of the item
      {
        int s = ys; uint32_t ph_ = yp;
        for (int k = 0; k < KT - 1; ++k) {
          mbar_wait(y_full + 8 * s, ph_);
          if (++s == kWmYSlots) { s = 0; ph_ ^= 1; }
        }
      }
      for (int p = d0; p < d1; ++p) {
        // newest plane (oldest + KT-1)
        {
          int s = ys + KT - 1; uint32_t ph_ = yp;
          if (s >= kWmYSlots) { s -= kWmYSlots; ph_ ^= 1; }
          mbar_wait(y_full + 8 * s, ph_);
        }
        mbar_wait((tf_cta ? x_ready : x_full) + 8 * xs, xp);
        tc_fence_after();
        const bool last = p + 1 == d1;
        if (leader) {
          const uint32_t a_lo = a_lo0 + ((x_base + xs * kWmXBytes) >> 4);
          const uint32_t b_lo = b_lo0 + ((y_base + ys * kWmYBytes) >> 4);
#pragma unroll
          for (int kh = 0; kh < KT; ++kh)
#pragma unroll
            for (int ks = 0; ks < 8; ++ks)
              if (kh >= kh_begin && kh < kh_end) umma_bf16_lohi(tmem + kh * NN, a_lo + (uint32_t)((kh * BW + ks * 2 * BW) * 64 >> 4), a_hi,
                             b_lo + (uint32_t)(ks * 16 * 64 >> 4), b_hi, idesc, (ks == 0 ? (first ^ 1u) : 1u));
          umma_commit(x_empty + 8 * xs);
          umma_commit(y_empty + 8 * ys);           // the oldest plane is dead after this step
          if (last) {                              // ... and so are the others at the end of an item
#pragma unroll
            for (int k = 1; k < KT; ++k) {
              int s = ys + k; if (s >= kWmYSlots) s -= kWmYSlots;
              umma_commit(y_empty + 8 * s);
            }
          }
        }
        __syncwarp();
        first = 0;
        if (++xs == kWmXStages) { xs = 0; xp ^= 1; }
        const int adv = last ? KT : 1;
        ys += adv;
        if (ys >= kWmYSlots) { ys -= kWmYSlots; yp ^= 1; }
      }
    }
    if (leader) umma_commit(acc_full);
    __syncwarp();
  } else {
    if (tf_cta) {
      // =========================== operand transform (warps 0-3), then the epilogue ===========================
      HaloTransform<128> T;
      const unsigned long long plane_vox = (unsigned long long)P.H * P.W;
      int xs = 0; uint32_t xp = 0;
      for (int it = i_begin; it < i_end; ++it) {
        int t = it;
        const int seg = t % P.nseg; t /= P.nseg;
        const int w0 = (t % P.tiles_w) * 8; t /= P.tiles_w;
        const int h0 = (t % P.tiles_h) * 16; t /= P.tiles_h;
        const int nb = t;
        const int d0 = seg * P.seg_len;
        int d1 = d0 + P.seg_len; if (d1 > P.D) d1 = P.D;
        T.setup((int)threadIdx.x, P.tf, nb, h0, w0, P.H, P.W);
        for (int p = d0; p < d1; ++p) {
          mbar_wait(x_full + 8 * xs, xp);
          T.apply(sm + (x_base - base) + xs * kWmXBytes, ((unsigned long long)nb * P.D + p) * plane_vox);
          fence_proxy_async();
          named_bar_sync(1, 128);
          if (threadIdx.x == 0) mbar_arrive(x_ready + 8 * xs);
          if (++xs == kWmXStages) { xs = 0; xp ^= 1; }
        }
      }
    }
    // =========================== epilogue: TMEM -> partial record ===========================
    mbar_wait(acc_full, 0);
    tc_fence_after();
    const bool any = i_end > i_begin;
    const size_t tap_elems = (size_t)P.ci_total * P.co_total;
    float* outb = P.partial + (size_t)blockIdx.x * P.ntaps * tap_elems;
    for (int kh = 0; kh < KT; ++kh) {
#pragma unroll 1
      for (int j = 0; j < KT; ++j) {
        uint32_t rr[32];
        tmem_ld_32x32b_x32(tmem + ((uint32_t)(warp * 32) << 16) + kh * NN + j * 32, rr);
        tmem_ld_wait();
        if (warp < KT) {   // warp = kw atom (the other atoms are unused), lane = ci
          int tap;
          if (KT == 3) tap = ((2 - j) * 3 + kh) * 3 + warp;
          else tap = ((2 * (1 - j) + 1 - pd) * 4 + (2 * kh + 1 - ph)) * 4 + (2 * warp + 1 - pw);
          float4* d4 = reinterpret_cast<float4*>(outb + (size_t)tap * tap_elems +
                                                 (size_t)(chunk * 32 + lane) * P.co_total + cot * 32);
#pragma unroll
          for (int q = 0; q < 8; ++q)
            d4[q] = any ? make_float4(__uint_as_float(rr[4 * q]), __uint_as_float(rr[4 * q + 1]),
                                      __uint_as_float(rr[4 * q + 2]), __uint_as_float(rr[4 * q + 3]))
                        : make_float4(0.f, 0.f, 0.f, 0.f);
        }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 5) tmem_dealloc_rt(tmem, 512);
}

}  // namespace ub
