// Marching-plane implicit GEMM for the 3x3x3 s1 p1 convolutions with 32 output channels -- the
// full-resolution layers that hold 57 % of the generator FLOPs (SURVEY.md Appendix B).
//
// Why a second kernel: with N = C_out = 32 a 128x32x16 UMMA reads 5 KB of shared memory in 16 tensor
// cycles (320 B/clk against 128 B/clk of smem bandwidth), so igemm_fwd_kernel tops out below 50 % of
// tensor peak on these layers. Here the depth taps are folded into N:
//
//     P[d'][(kd, co)][h, w] = sum_{kh, kw, c} X[d', h+kh-1, w+kw-1, c] * W[kd, kh, kw][co][c]      (N = 96)
//     out[d][co][h, w]      = P[d-1][(0, co)] + P[d][(1, co)] + P[d+1][(2, co)]
//
// One CTA owns a 16x8 (h, w) column and *marches* along d: every input plane is loaded once (TMA halo
// tile, 18x10 rows), multiplied by the 9 (kh, kw) weight tiles of N = 96 rows (18 UMMAs per 32-channel
// chunk instead of 54), and lands in one of four TMEM accumulators. The epilogue warps, one plane
// behind, add the three 32-column slices that belong to output plane d -- same thread, three TMEM
// loads, no cross-lane traffic -- while the MMA thread already works on the next planes (TMEM ring of
// 5 x 96 columns). Eight epilogue warps (two per TMEM lane quarter, 16 output channels each) read every
// accumulator once, as soon as it completes, and roll the partial output planes through registers.
// The full weight set (9 x 96 x C_in bf16, <= 162 KB for the 96->32 skip-concat conv)
// stays resident in shared memory for the CTA's lifetime.
#pragma once
#include "igemm_fwd.cuh"
#include "pointwise.cuh"
#include "deferred_tile.cuh"

namespace ub {

struct MarchParams {
  CUtensorMap tm_src[2];
  CUtensorMap tm_w;                 // [9 * 96][Kpad] bf16, box (32, 96); pair mode: box (32, 48)
  int n_chunks_src0, n_chunks_total;
  int Nb, D, H, W;
  int tiles_w, tiles_h, nseg, seg_len;
  void* out;                        // [N][D][H][W][32] bf16
  const float* bias;
  int bias_n;
  float* stats;                     // [item][2][32] or nullptr
  int nsa;                          // A (plane, chunk) stages
  // kNormBwd instantiation (dgrad of the conv that consumes a norm block's activations): the tensor
  // written here is dA of that block; the epilogue also accumulates its norm-backward reductions
  //   S1[n,c] = sum dz,  S2[n,c] = sum dz * xhat,  dz = dA * lrelu'(y*scale+shift) * dropout,
  // into `stats` (same per-CTA record format), so the separate reduction pass over dA and y is not run.
  const void* nb_y;                 // raw conv output of the producer block [N][D][H][W][32] bf16
  const float* nb_scale;            // [N][32] gamma * rstd
  const float* nb_shift;            // [N][32]
  const float* nb_mean;             // [N][32]
  const float* nb_rstd;             // [N][32]
  float nb_slope, nb_drop_p;
  uint32_t nb_drop_seed, nb_drop_thresh;
  // kTf instantiation: source 0 (one 32-channel chunk) is the raw fp16 output y of a conv -> norm block and `tf`
  // its deferred activation; two extra warps rewrite every halo plane of chunk 0 in shared memory
  // (deferred_tile.cuh) between the TMA arrival and the MMAs.
  int src0_f16;                     // source 0 is a MATERIALISED fp16 activation tensor (its chunks are fp16 x fp16 MMAs
                                    // against weight columns packed as fp16, UB_PACK_F16_SRC0)
  NormActArgs tf;
  int tf_f16;                       // the transformed chunk is an fp16 operand (its weight columns are packed as fp16)
};

constexpr int kMarchPlaneBytes = 12288;   // 180 rows x 64 B, padded to a multiple of 1024
constexpr int kMarchWTileBytes = 96 * 64;  // one (chunk, kh, kw) weight tile

constexpr int kMarchRing = 5;       // TMEM accumulator ring: 5 x 96 columns
constexpr int kMarchEpiWarps = 8;
constexpr int kMarchThreads = (kMarchEpiWarps + 2) * 32;   // warps 0-7 epilogue, warp 8 TMA producer, warp 9 MMA issuer (+ warp 10: second issuer, kMarchThreads2)
// kTf: + two operand-transform warps. Two, not four: the epilogue warps need ~166 registers and a scheduler
// partition holds 16 K of them, so the CTA must stay at <= 3 warps per partition (12 warps). Role order in a kTf
// CTA: warps 0-7 epilogue, 8-9 transform, 10 TMA producer, 11 MMA issuer -- the warp scheduler prefers the
// highest warp id among the ready warps of a partition, and the MMA thread is the one that must never wait.
constexpr int kMarchTfThreads = 64;
constexpr int kMarchThreadsTf = kMarchThreads + kMarchTfThreads;

// One MMA issuer of the single-CTA, untransformed kernel taking planes p_first + me, + step, ...: ring slot, stage and
// barrier phases follow from the plane index alone, so several issuers need no shared state.
__device__ __forceinline__ void march_issue_planes(const MarchParams& P, int me, int step, int p_first, int p_last, int nch,
                                                   uint32_t tmem, uint32_t w_base, uint32_t a_base, uint32_t w_full,
                                                   uint32_t a_full, uint32_t a_empty, uint32_t acc_full, uint32_t acc_empty) {
  const uint32_t idesc_bf = make_idesc_bf16(128, 96, 0, 0);
  const uint32_t idesc_h = idesc_f16_operands(idesc_bf);
  const uint32_t a_hi = (uint32_t)(make_smem_desc(0, 16, 10 * 64, SWZ_64B) >> 32);
  const uint32_t b_hi = (uint32_t)(make_smem_desc(0, 16, 8 * 64, SWZ_64B) >> 32);
  const uint32_t lbo_lo = 1u << 16;
  const bool leader = elect_one();
  const int n_f16 = P.src0_f16 ? P.n_chunks_src0 : 0;
  mbar_wait(w_full, 0);
  tc_fence_after();
  for (int p = p_first + me; p <= p_last; p += step) {
    const int pi = p - p_first;
    const int slot = pi % kMarchRing;
    mbar_wait(acc_empty + 8 * slot, (((uint32_t)(pi / kMarchRing)) & 1u) ^ 1u);
    tc_fence_after();
    const uint32_t acc = tmem + slot * 96;
    for (int c = 0; c < nch; ++c) {
      const int si = pi * nch + c;
      const int sa = si % P.nsa;
      mbar_wait(a_full + 8 * sa, ((uint32_t)(si / P.nsa)) & 1u);
      tc_fence_after();
      if (leader) {
        const uint32_t idesc = c < n_f16 ? idesc_h : idesc_bf;
        const uint32_t a_lo = lbo_lo | ((a_base + sa * kMarchPlaneBytes) >> 4);
        const uint32_t b_lo = lbo_lo | ((w_base + c * 9 * kMarchWTileBytes) >> 4);
#pragma unroll
        for (int kh = 0; kh < 3; ++kh)
#pragma unroll
          for (int kw = 0; kw < 3; ++kw) {
            const uint32_t ao = (uint32_t)((kh * 10 + kw) * 64) >> 4;
            const uint32_t bo = (uint32_t)((kh * 3 + kw) * kMarchWTileBytes) >> 4;
            umma_bf16_lohi(acc, a_lo + ao, a_hi, b_lo + bo, b_hi, idesc, (uint32_t)((c | kh | kw) != 0));
            umma_bf16_lohi(acc, a_lo + ao + 2, a_hi, b_lo + bo + 2, b_hi, idesc, 1u);
          }
        umma_commit(a_empty + 8 * sa);
      }
      __syncwarp();
    }
    if (leader) umma_commit(acc_full + 8 * slot);
    __syncwarp();
  }
}

// kPair: two CTAs of a cluster (cta_group::2) own two neighbouring 16x8 columns and march together; every
// UMMA is M = 256 x N = 96 with the 96 weight rows split 48 / 48 between the two CTAs' shared memories,
// so each SM reads 4 KB (A) + 1.5 KB (B) per instruction instead of 4 + 3 KB -- the shared-memory pipe is
// what bounds the single-CTA kernel (ncu: 81 % l1tex data-pipe, 69 % tensor-pipe active). The leader
// (rank 0) issues the MMAs and owns w_full / a_full / acc_empty; the peer's TMA loads and epilogue arrive
// on them remotely; tcgen05.commit multicasts a_empty / acc_full to both CTAs.
// kTf (forward only): chunk 0 arrives as y and is transformed in place. Its TMA completes on a CTA-local barrier
// a_loc[stage] (pair mode: each CTA waits for its own plane), the transform warps hand the stage to the MMA thread
// through a_ready[stage] in the leader CTA (one arrival per CTA). Untransformed chunks keep the a_full path. A
// stage alternates between the two paths, so the barrier phases are tracked per stage in bit masks.
// !kPair && !kTf: warp kMmaWarp + 1 is a second MMA issuer. The two warps take alternating planes -- different
// accumulator slots and different A stages, so nothing orders them against each other -- and one warp's per-plane
// hand-off (two barrier waits, two fences, two commits) runs while the other one's UMMAs are in the pipe. Measured
// (profiles/r02j_march_mma2.txt): one-chunk 32 -> 32 forward 0.875 -> 0.71 ms, its dgrad 0.85 -> 0.70, 24 -> 32
// 0.85 -> 0.68, three chunks without CTA pairs 2.18 -> 2.05. In the CTA-pair kernel a second issuer measured neutral
// (profiles/r02j_march_pair_mma2.txt), removed: warp kMmaWarp + 1 idles there.
constexpr int kMarchThreads2 = kMarchThreads + 32;
template <bool kNormBwd, bool kPair, bool kTf>
__global__ void __launch_bounds__(kTf ? kMarchThreadsTf : kMarchThreads2, 1)
igemm_march_kernel(const __grid_constant__ MarchParams P) {
  static_assert(!(kNormBwd && kTf), "the operand transform is a forward-path feature");
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* sm = smem_raw + (base - smem_u32(smem_raw));
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int nch = P.n_chunks_total;
  constexpr int kTfWarps = kTf ? kMarchTfThreads / 32 : 0;
  constexpr int kTmaWarp = kMarchEpiWarps + kTfWarps, kMmaWarp = kTmaWarp + 1;
  const uint32_t rank = kPair ? cluster_ctarank() : 0u;
  constexpr int kWTile = kPair ? kMarchWTileBytes / 2 : kMarchWTileBytes;   // this CTA's share of a weight tile

  const uint32_t w_base = base;
  const uint32_t a_base = w_base + nch * 9 * kWTile;
  const uint32_t bar_base = a_base + P.nsa * kMarchPlaneBytes;
  // barriers: w_full | a_full[nsa] | a_empty[nsa] | acc_full[ring] | acc_empty[ring] | a_loc[nsa] | a_ready[nsa]
  const uint32_t w_full = bar_base, a_full = w_full + 8, a_empty = a_full + 8 * P.nsa,
                 acc_full = a_empty + 8 * P.nsa, acc_empty = acc_full + 8 * kMarchRing,
                 a_loc = acc_empty + 8 * kMarchRing, a_ready = a_loc + 8 * P.nsa, bar_end = a_ready + 8 * P.nsa;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(sm + (bar_end - base));
  float* red = reinterpret_cast<float*>(sm + (((bar_end + 16 + 15) & ~15u) - base));  // [8][2][32] + bias[32] + consts[4][32], 16-B aligned

  // ---- work item: (n, h tile, w tile, d segment); a CTA pair takes the w tiles 2k and 2k+1
  int t = kPair ? (int)(blockIdx.x >> 1) : (int)blockIdx.x;
  const int seg = t % P.nseg; t /= P.nseg;
  const int tiles_wp = kPair ? P.tiles_w / 2 : P.tiles_w;
  const int tw_i = kPair ? (t % tiles_wp) * 2 + (int)rank : t % tiles_wp; t /= tiles_wp;
  const int th_i = t % P.tiles_h; t /= P.tiles_h;
  const int nb = t;
  const int item = ((nb * P.tiles_h + th_i) * P.tiles_w + tw_i) * P.nseg + seg;   // statistics record
  const int w0 = tw_i * 8, h0 = th_i * 16;
  const int d_begin = seg * P.seg_len;
  int d_end = d_begin + P.seg_len; if (d_end > P.D) d_end = P.D;
  const int p_first = d_begin > 0 ? d_begin - 1 : 0;           // input planes [p_first, p_last]
  const int p_last = d_end < P.D ? d_end : P.D - 1;

  if (threadIdx.x == 0) {
    mbar_init(w_full, 1);
    for (int i = 0; i < P.nsa; ++i) { mbar_init(a_full + 8 * i, 1); mbar_init(a_empty + 8 * i, 1); }
    for (int i = 0; i < kMarchRing; ++i) {
      mbar_init(acc_full + 8 * i, 1);
      // single CTA: one arrival per epilogue warp and plane; pair: ONE arrival per CTA and plane (the eight
      // warps meet at a named barrier first -- remote mbarrier arrivals are expensive)
      mbar_init(acc_empty + 8 * i, kPair ? 2 : kMarchEpiWarps);
    }
    for (int i = 0; i < P.nsa; ++i) { mbar_init(a_loc + 8 * i, 1); mbar_init(a_ready + 8 * i, kPair ? 2 : 1); }
    fence_mbar_init();
  }
  if (warp == kTmaWarp && lane == 0) {
    tma_prefetch_desc(&P.tm_src[0]);
    if (nch > P.n_chunks_src0) tma_prefetch_desc(&P.tm_src[1]);
    tma_prefetch_desc(&P.tm_w);
  }
  if (warp == kMmaWarp) {
    if (kPair) tmem_alloc_pair(smem_u32(tmem_slot), 512);
    else tmem_alloc_rt(smem_u32(tmem_slot), 512);
  }
  tc_fence_before();
  __syncthreads();
  if (kPair) cluster_sync_all();   // the peer's barriers are initialised before anything signals them
  tc_fence_after();
  const uint32_t tmem = *tmem_slot;
  // barriers that live in the leader CTA, as shared::cluster addresses usable from both CTAs
  const uint32_t w_full_ld = kPair ? mapa_shared(w_full, 0) : w_full;
  const uint32_t a_full_ld = kPair ? mapa_shared(a_full, 0) : a_full;
  const uint32_t acc_empty_ld = kPair ? mapa_shared(acc_empty, 0) : acc_empty;
  const uint32_t a_ready_ld = kPair ? mapa_shared(a_ready, 0) : a_ready;

  if (warp == kTmaWarp) {
    // =========================== TMA producer ===========================
    if (lane == 0) {
      const uint32_t w_bytes = (uint32_t)(nch * 9 * kWTile);
      if (rank == 0) mbar_expect_tx(w_full, kPair ? 2 * w_bytes : w_bytes);
      for (int c = 0; c < nch; ++c)
        for (int tp = 0; tp < 9; ++tp) {
          if (kPair) tma_load_2d_pair(w_base + (c * 9 + tp) * kWTile, &P.tm_w, w_full_ld, c * 32, tp * 96 + (int)rank * 48);
          else tma_load_2d(w_base + (c * 9 + tp) * kWTile, &P.tm_w, w_full, c * 32, tp * 96);
        }
      int sa = 0;
      uint32_t pa = 0;
      for (int p = p_first; p <= p_last; ++p) {
        for (int c = 0; c < nch; ++c) {
          mbar_wait(a_empty + 8 * sa, pa ^ 1);
          if (kTf && c == 0) {
            // y plane of the deferred source: completes on this CTA's own barrier, the transform warps take over
            mbar_expect_tx(a_loc + 8 * sa, 180 * 64);
            tma_load_5d(a_base + sa * kMarchPlaneBytes, &P.tm_src[0], a_loc + 8 * sa, 0, w0 - 1, h0 - 1, p, nb);
            if (++sa == P.nsa) { sa = 0; pa ^= 1; }
            continue;
          }
          if (rank == 0) mbar_expect_tx(a_full + 8 * sa, kPair ? 2 * 180 * 64 : 180 * 64);
          const bool s1 = c >= P.n_chunks_src0;
          if (kPair)
            tma_load_5d_pair(a_base + sa * kMarchPlaneBytes, &P.tm_src[s1 ? 1 : 0], a_full_ld + 8 * sa,
                             (s1 ? c - P.n_chunks_src0 : c) * 32, w0 - 1, h0 - 1, p, nb);
          else
            tma_load_5d(a_base + sa * kMarchPlaneBytes, &P.tm_src[s1 ? 1 : 0], a_full + 8 * sa,
                        (s1 ? c - P.n_chunks_src0 : c) * 32, w0 - 1, h0 - 1, p, nb);
          if (++sa == P.nsa) { sa = 0; pa ^= 1; }
        }
      }
    }
    __syncwarp();
  } else if (warp == kMmaWarp) {
    // =========================== MMA issuer (leader CTA only in pair mode) ===========================
    if (!kPair && !kTf) {
      march_issue_planes(P, 0, 2, p_first, p_last, nch, tmem, w_base, a_base, w_full, a_full, a_empty, acc_full, acc_empty);
    } else if (rank == 0) {
      const uint32_t idesc_bf = make_idesc_bf16(kPair ? 256 : 128, 96, 0, 0);
      const uint32_t idesc_h = idesc_f16_operands(idesc_bf);
      const uint32_t idesc_tf = (kTf && P.tf_f16) ? idesc_h : idesc_bf;   // chunk 0 of a kTf CTA
      const uint32_t a_hi = (uint32_t)(make_smem_desc(0, 16, 10 * 64, SWZ_64B) >> 32);
      const uint32_t b_hi = (uint32_t)(make_smem_desc(0, 16, 8 * 64, SWZ_64B) >> 32);
      const uint32_t lbo_lo = 1u << 16;
      const bool leader = elect_one();
      mbar_wait(w_full, 0);
      tc_fence_after();
      int sa = 0;
      uint32_t pa = 0;                      // !kTf: every stage use completes a_full -- one ring parity
      uint32_t ph_full = 0, ph_ready = 0;   // kTf: a stage alternates between a_full and a_ready -- per-stage phase bits
      const int n_f16 = P.src0_f16 ? P.n_chunks_src0 : 0;   // chunks of a materialised fp16 source 0
      int slot = 0;
      uint32_t pacc = 0;
      for (int p = p_first; p <= p_last; ++p) {
        mbar_wait(acc_empty + 8 * slot, pacc ^ 1);
        tc_fence_after();
        const uint32_t acc = tmem + slot * 96;
        for (int c = 0; c < nch; ++c) {
          if (!kTf) {
            mbar_wait(a_full + 8 * sa, pa);
          } else if (c == 0) {
            mbar_wait(a_ready + 8 * sa, (ph_ready >> sa) & 1u);
            ph_ready ^= 1u << sa;
          } else {
            mbar_wait(a_full + 8 * sa, (ph_full >> sa) & 1u);
            ph_full ^= 1u << sa;
          }
          tc_fence_after();
          if (leader) {
            const uint32_t idesc = kTf ? (c == 0 ? idesc_tf : idesc_bf) : (c < n_f16 ? idesc_h : idesc_bf);
            const uint32_t a_lo = lbo_lo | ((a_base + sa * kMarchPlaneBytes) >> 4);
            const uint32_t b_lo = lbo_lo | ((w_base + c * 9 * kWTile) >> 4);
#pragma unroll
            for (int kh = 0; kh < 3; ++kh)
#pragma unroll
              for (int kw = 0; kw < 3; ++kw) {
                const uint32_t ao = (uint32_t)((kh * 10 + kw) * 64) >> 4;
                const uint32_t bo = (uint32_t)((kh * 3 + kw) * kWTile) >> 4;
                if (kPair) {
                  umma_bf16_lohi_pair(acc, a_lo + ao, a_hi, b_lo + bo, b_hi, idesc, (uint32_t)((c | kh | kw) != 0));
                  umma_bf16_lohi_pair(acc, a_lo + ao + 2, a_hi, b_lo + bo + 2, b_hi, idesc, 1u);
                } else {
                  umma_bf16_lohi(acc, a_lo + ao, a_hi, b_lo + bo, b_hi, idesc, (uint32_t)((c | kh | kw) != 0));
                  umma_bf16_lohi(acc, a_lo + ao + 2, a_hi, b_lo + bo + 2, b_hi, idesc, 1u);
                }
              }
            if (kPair) umma_commit_pair(a_empty + 8 * sa);
            else umma_commit(a_empty + 8 * sa);
          }
          __syncwarp();
          if (++sa == P.nsa) { sa = 0; pa ^= 1; }
        }
        if (leader) {
          if (kPair) umma_commit_pair(acc_full + 8 * slot);
          else umma_commit(acc_full + 8 * slot);
        }
        __syncwarp();
        if (++slot == kMarchRing) { slot = 0; pacc ^= 1; }
      }
    }
  } else if (!kTf && warp == kMmaWarp + 1) {
    // =========================== second MMA issuer (single CTA): odd planes ===========================
    if (!kPair) march_issue_planes(P, 1, 2, p_first, p_last, nch, tmem, w_base, a_base, w_full, a_full, a_empty, acc_full, acc_empty);
  } else if (kTf && warp >= kMarchEpiWarps) {
    // =========================== operand transform (warps 8-9) ===========================
    const int t = (int)threadIdx.x - kMarchEpiWarps * 32;
    const unsigned long long plane_vox = (unsigned long long)P.H * P.W;
    auto run = [&](auto& T) {
      T.setup(t, P.tf, nb, h0, w0, P.H, P.W);
      int sa = 0;
      uint32_t ph_loc = 0;
      for (int p = p_first; p <= p_last; ++p) {
        // chunk 0 of plane p sits in stage sa; the other chunks of the plane only advance the ring
        mbar_wait(a_loc + 8 * sa, (ph_loc >> sa) & 1u);
        ph_loc ^= 1u << sa;
        T.apply(sm + (a_base - base) + sa * kMarchPlaneBytes, ((unsigned long long)nb * P.D + p) * plane_vox);
        fence_proxy_async();                       // generic-proxy writes -> visible to the tensor core's async proxy
        named_bar_sync(3, kMarchTfThreads);
        if (t == 0) {
          if (kPair) mbar_arrive_cluster(a_ready_ld + 8 * sa, 1u);
          else mbar_arrive(a_ready + 8 * sa);
        }
        sa = (sa + nch) % P.nsa;
      }
    };
    if (P.tf_f16) {
      HaloTransform<kMarchTfThreads, true> T;
      run(T);
    } else {
      HaloTransform<kMarchTfThreads, false> T;
      run(T);
    }
  } else {
    // =========================== epilogue (warps 0-7) ===========================
    // warp w reads TMEM lanes 32*(w%4)..+31 (accumulator rows); warp group w/4 takes the output channels
    // [16*(w/4), +16). Every input plane's accumulator is read ONCE, right when it completes, and handed
    // back to the MMA thread immediately: its three depth slices are contributions to the output planes
    // p+1 (kd=0), p (kd=1), p-1 (kd=2), which roll through two register sets (ra: plane p-1 so far,
    // rb: plane p so far). The MMA thread can therefore run ring-1 planes ahead of the epilogue.
    const int q = warp & 3, half = warp >> 2;
    const int r = q * 32 + lane;
    const int h = h0 + (r >> 3), w = w0 + (r & 7);
    const bool valid_hw = (h < P.H) && (w < P.W);
    const bool do_stats = P.stats != nullptr;
    float* bias_s = red + kMarchEpiWarps * 2 * 32;
    float* nbc = bias_s + 32;   // [scale*inv | shift*inv | rstd | -mean*rstd][32] of this CTA's sample (folded like the forward)
    if (threadIdx.x < 32)
      bias_s[threadIdx.x] = (P.bias != nullptr && threadIdx.x < P.bias_n) ? __ldg(P.bias + threadIdx.x) : 0.f;
    if (kNormBwd && threadIdx.x >= 32 && threadIdx.x < 64) {
      const int c = threadIdx.x - 32;
      const float rs = P.nb_rstd[nb * 32 + c];
      const float finv = P.nb_drop_p > 0.f ? 1.f / (1.f - P.nb_drop_p) : 1.f;
      nbc[c] = fold_inv(P.nb_scale[nb * 32 + c], finv);
      nbc[32 + c] = fold_inv(P.nb_shift[nb * 32 + c], finv);
      nbc[64 + c] = rs;
      nbc[96 + c] = -P.nb_mean[nb * 32 + c] * rs;
    }
    named_bar_sync(1, kMarchEpiWarps * 32);
    const bool has_drop = kNormBwd && P.nb_drop_p > 0.f;
    const float nb_inv = has_drop ? 1.f / (1.f - P.nb_drop_p) : 1.f;
    const int cb = half * 16;           // first channel of this thread
    float bias_r[16];
#pragma unroll
    for (int j = 0; j < 16; ++j) bias_r[j] = bias_s[cb + j];
    float st_a[16], st_b[16];           // per-thread channel sums over the CTA's planes; transposed once at the end
    float ra[16], rb[16];
#pragma unroll
    for (int j = 0; j < 16; ++j) { st_a[j] = 0.f; st_b[j] = 0.f; ra[j] = 0.f; rb[j] = 0.f; }
    __nv_bfloat16* outp = reinterpret_cast<__nv_bfloat16*>(P.out);
    const uint32_t lane_base = tmem + ((uint32_t)(q * 32) << 16) + (uint32_t)cb;
    const size_t plane_vox = (size_t)P.H * P.W;
    const size_t vox0 = (((size_t)nb * P.D) * P.H + h) * P.W + w;     // voxel of plane 0

    // finish output plane d from `fin` (all three depth contributions summed): bias, bf16, store, statistics
    auto finish_plane = [&](int d, const float (&fin)[16], const uint4 (&yv)[2]) {
      uint32_t pk[8];
      // with statistics the tensor written here is the raw output of a conv -> norm block: fp16, never an MMA operand
      const bool y16 = !kNormBwd && do_stats;
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const float x0 = fin[2 * j] + bias_r[2 * j], x1 = fin[2 * j + 1] + bias_r[2 * j + 1];
        pk[j] = y16 ? pack_f16x2_sat(x0, x1) : pack_bf16x2(x0, x1);
      }
      const size_t vox = vox0 + (size_t)d * plane_vox;
      if (valid_hw) {
        // 16 channels = 32 bytes = one whole sector of this voxel row
        uint4* dst = reinterpret_cast<uint4*>(outp + vox * 32 + cb);
        __stcs(dst, make_uint4(pk[0], pk[1], pk[2], pk[3]));
        __stcs(dst + 1, make_uint4(pk[4], pk[5], pk[6], pk[7]));
      }
      if (!kNormBwd && do_stats && valid_hw) {
        // statistics from the fp32 accumulators
#pragma unroll
        for (int j = 0; j < 16; ++j) {
          const float x = fin[j] + bias_r[j];
          st_a[j] += x;
          st_b[j] = fmaf(x, x, st_b[j]);
        }
      }
      if (kNormBwd && valid_hw) {
        // dz from the ROUNDED gradient (what the apply pass will read back) and the forward's own fma.
        // st_a accumulates sum dz, st_b accumulates sum dz * y; xhat = y * rstd - mean * rstd is applied
        // once per thread after the loop.
        const uint32_t* yw = reinterpret_cast<const uint32_t*>(yv);
#pragma unroll
        for (int o8 = 0; o8 < 2; ++o8) {
          float f[8];
          if (has_drop) {
            dropout_factors8((unsigned long long)vox * 32ull + cb + o8 * 8, P.nb_drop_seed, P.nb_drop_thresh, nb_inv, f);
          } else {
#pragma unroll
            for (int k = 0; k < 8; ++k) f[k] = 1.f;
          }
#pragma unroll
          for (int k = 0; k < 8; ++k) {
            const int c = o8 * 8 + k;
            const uint32_t dw = pk[c >> 1], yy = yw[c >> 1];
            const float da = __uint_as_float((c & 1) ? (dw & 0xFFFF0000u) : (dw << 16));
            const float yf = __half2float(__ushort_as_half((unsigned short)((c & 1) ? (yy >> 16) : (yy & 0xFFFFu))));   // y is fp16
            const float dz = da * (fmaf(yf, nbc[cb + c], nbc[32 + cb + c]) > 0.f ? f[k] : f[k] * P.nb_slope);
            st_a[c] += dz;
            st_b[c] = fmaf(dz, yf, st_b[c]);
          }
        }
      }
    };

    for (int p = p_first; p <= p_last; ++p) {
      const int pi = p - p_first;
      const int slot = pi % kMarchRing;
      // the output plane this step completes is p-1: fetch its producer-block row early (kNormBwd)
      const int dfin = p - 1;
      const bool fin_ok = dfin >= d_begin && dfin < d_end;
      uint4 yv[2];
      if (kNormBwd && valid_hw && fin_ok) {
        const uint4* yp = reinterpret_cast<const uint4*>(P.nb_y) + (vox0 + (size_t)dfin * plane_vox) * 4 + half * 2;
        yv[0] = __ldg(yp);
        yv[1] = __ldg(yp + 1);
        if (dfin + 1 < d_end) asm volatile("prefetch.global.L2 [%0];" ::"l"(yp + plane_vox * 4));
      }
      mbar_wait(acc_full + 8 * slot, (uint32_t)(pi / kMarchRing) & 1u);
      tc_fence_after();
      uint32_t v0[16], v1[16], v2[16];
      const uint32_t ta = lane_base + (uint32_t)(slot * 96);
      tmem_ld_32x32b_x16(ta, v0);           // kd = 0 -> output plane p+1
      tmem_ld_32x32b_x16(ta + 32, v1);      // kd = 1 -> output plane p
      tmem_ld_32x32b_x16(ta + 64, v2);      // kd = 2 -> output plane p-1
      tmem_ld_wait();
      // the accumulator is in registers: hand the slot back before doing anything else
      tc_fence_before();
      if (kPair) {
        named_bar_sync(2, kMarchEpiWarps * 32);
        if (threadIdx.x == 0) mbar_arrive_cluster(acc_empty_ld + 8 * slot, 1u);
      } else {
        __syncwarp();
        if (lane == 0) mbar_arrive(acc_empty + 8 * slot);
      }
      float fin[16];
#pragma unroll
      for (int j = 0; j < 16; ++j) {
        fin[j] = ra[j] + __uint_as_float(v2[j]);
        ra[j] = rb[j] + __uint_as_float(v1[j]);
        rb[j] = __uint_as_float(v0[j]);
      }
      if (fin_ok) finish_plane(dfin, fin, yv);
    }
    // the last output plane of the volume has no plane behind it: ra already holds its full sum
    if (p_last == d_end - 1) {
      uint4 yv[2];
      if (kNormBwd && valid_hw) {
        const uint4* yp = reinterpret_cast<const uint4*>(P.nb_y) + (vox0 + (size_t)p_last * plane_vox) * 4 + half * 2;
        yv[0] = __ldg(yp);
        yv[1] = __ldg(yp + 1);
      }
      finish_plane(p_last, ra, yv);
    }
    if (kNormBwd) {
      // S2 = sum dz * xhat = rstd * sum dz*y - mean*rstd * sum dz
#pragma unroll
      for (int c = 0; c < 16; ++c) st_b[c] = fmaf(nbc[64 + cb + c], st_b[c], nbc[96 + cb + c] * st_a[c]);
    }
    if (do_stats || kNormBwd) {
      float ta_[32], tb_[32];
#pragma unroll
      for (int j = 0; j < 32; ++j) { ta_[j] = j < 16 ? st_a[j] : 0.f; tb_[j] = j < 16 ? st_b[j] : 0.f; }
      const float s_acc = warp_transpose_reduce32(ta_, lane);   // lane l < 16: total of channel cb + l
      const float q_acc = warp_transpose_reduce32(tb_, lane);
      if (lane < 16) {
        red[(warp * 2 + 0) * 32 + lane] = s_acc;
        red[(warp * 2 + 1) * 32 + lane] = q_acc;
      }
      named_bar_sync(1, kMarchEpiWarps * 32);
      if (threadIdx.x < 32) {
        const int hh = lane >> 4, cl = lane & 15;     // channel lane = hh * 16 + cl, summed over the 4 lane quarters
        float s = 0.f, qq = 0.f;
#pragma unroll
        for (int wq = 0; wq < 4; ++wq) {
          s += red[((hh * 4 + wq) * 2 + 0) * 32 + cl];
          qq += red[((hh * 4 + wq) * 2 + 1) * 32 + cl];
        }
        float* st = P.stats + (size_t)item * 64;
        st[lane] = s;
        st[32 + lane] = qq;
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (kPair) cluster_sync_all();   // neither CTA leaves (or frees TMEM) while the other may still signal it
  if (warp == kMmaWarp) {
    if (kPair) tmem_dealloc_pair(tmem, 512);
    else tmem_dealloc_rt(tmem, 512);
  }
}

}  // namespace ub
