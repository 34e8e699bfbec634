// Tap-table implicit-GEMM convolution for sm_100a: TMA halo tiles -> shifted UMMA views -> TMEM.
//
// One kernel serves every "activation x weights -> activation" contraction on the hot path:
//   * Conv3d 3x3x3 s1 p1 forward and its dgrad (flipped/transposed weight pack)   ref:model.py:22-28 (BasicUNet)
//   * Conv3d 4x4x4 s2 p1 forward (8 parity tiles loaded with TMA elementStrides=2)  ref:model.py:50,72-82
//     and its dgrad (8 output parity classes, scatter store)
//   * ConvTranspose3d k2 s2 forward (1 tap, scatter store) and dgrad (8 parity tiles) ref:BasicUNet UpCat
//   * 1x1x1 convs (heads, final convs)                                            ref:model.py:19-21,83
//
// Geometry: an output tile is TD planes x 16 (h) x 8 (w) voxels. Every plane is one UMMA M=128
// accumulator of NT fp32 columns in TMEM. For each K chunk (kIgemmKc = 32 input channels, one
// 64-byte swizzle span per voxel row) the producer loads the *halo* of the tile once per A-tile
// ((16+KH-1) x (8+KW-1) rows per plane) and the MMA thread addresses each filter tap as a
// row-shifted view of that halo (start address + row offset, SBO = box-width rows) -- no im2col
// re-load per tap. The skip concatenation is a second tensor map: chunks [0,n0) come from source 0,
// the rest from source 1, so the concat tensor never exists. Weights stream through a TMA ring,
// one [NT x kc] tile per (chunk, tap), shared by the TD planes.
//
// The kernel is persistent: one CTA per SM walks the tile list (stride gridDim.x); the TMA rings run
// across tile boundaries and the accumulators are double-buffered in TMEM whenever two sets fit in
// 512 columns, so the epilogue of tile i overlaps the loads and MMAs of tile i+1.
//
// Epilogue (8 warps, two per TMEM lane quarter, thread <-> accumulator row): tcgen05.ld -> +bias ->
// optional LeakyReLU -> per-channel sum / sum-of-squares partials (register transpose-reduce with
// shuffles, one partial record per tile, no atomics) -> bf16 -> 16-byte global stores; neighbouring
// lanes exchange half rows first so that every store instruction writes whole 32-byte sectors.
#pragma once
#include "sm100_ptx.cuh"

namespace ub {

constexpr int kMaxTaps = 64;
constexpr int kIgemmKc = 32;     // input channels per K chunk of the generic kernel (64-byte rows, two K = 16 UMMAs)
constexpr int kMaxAccSets = 2;   // TMEM accumulator sets of the generic kernel (tiles whose epilogue may be pending)
constexpr int kMaxATiles = 8;
constexpr int kMaxNTiles = 16;

struct IgemmTap {
  uint16_t atile;      // which A tile of the stage
  uint16_t row_off;    // row offset inside the tile plane (kh * box_w + kw)
  uint16_t plane_off;  // plane offset (kd)
  uint16_t wblock;     // weight row block (rows [wblock * w_rows_per_block + n0, ...))
};

struct IgemmNTile {
  int n0;             // first output column (row inside a weight block)
  int nt;             // columns in this tile (multiple of 16, <= 128)
  void* out;          // destination tensor (bf16, NDHWC)
  int out_cpitch;     // channels per voxel in the destination
  int out_coff;       // channel offset inside the destination voxel
  int split;          // columns [split, nt) go to out2 instead (split == nt: single destination)
  void* out2;         // second destination (dgrad of a skip-concat conv: [d skip | d upsampled])
  int out2_cpitch;
  int wblock_add;     // added to every tap's weight block (transposed conv: the sub-position's tap)
  int tapset;         // tap table / tile-origin set of this N tile (stride-2 dgrad: the input parity class)
  int out_p[3];       // destination voxel = tile-space voxel * out_s + out_p (w,h,d)
};

struct IgemmParams {
  CUtensorMap tm_src[2];
  CUtensorMap tm_w;
  int n_chunks_src0, n_chunks_total;
  int n_atiles, bw, bh, n_in_planes, in_stride;
  // chunks_per_group > 0 ("group mode", space-to-depth sources): chunk ch belongs to group
  // g = ch / chunks_per_group (the input parity class); the stage holds ONE tile whose origin offset
  // is atile_off[g] and the taps of that chunk are taps[g * ntaps + tp]. The source is parity-planar
  // ([N * groups][D][H][W][chunks_per_group * kc]): channel coordinate (ch % chunks_per_group) * kc,
  // batch coordinate nb * groups + g. The weight K coordinate is (ch % chunks_per_group) * kc (kc = kIgemmKc).
  int chunks_per_group;
  int atile_off[kMaxATiles][3];  // (w, h, d) added to in_stride * tile origin
  int ntaps;
  IgemmTap taps[kMaxTaps];
  int w_rows_per_block;
  // kd_fold = f > 0 (3x3x3, one N tile of nt columns, f * nt <= 256): the weight tile of a (chunk, kh, kw)
  // tap holds the three depth taps stacked as rows [(2 - kd) * nt + n]; input plane p of the halo
  // feeds the output planes p-2 .. p of the tile with UMMAs of N = up to f * nt (their accumulators
  // are adjacent TMEM columns), so the A operand is read from shared memory once per f depth taps.
  int kd_fold;
  int fold_nd;                   // depth taps folded (3: 3x3x3; 2: the stride-2 stem on its space-to-depth source)
  int fold_row_step;             // weight-tensor rows between the depth-tap blocks j = 0 .. fold_nd-1 of a tile
                                 // (block j holds depth tap fold_nd-1-j)
  int b_block_rows;              // rows of one weight block in the packed tensor (nt, or 3 * nt when folded)
  int td;
  int Nb, Do, Ho, Wo;            // tile space (output voxels before the optional scatter)
  int tiles_w, tiles_h, tiles_d;
  int n_ntiles;
  IgemmNTile ntile[kMaxNTiles];
  int out_s;                     // destination voxel = tile-space voxel * out_s + ntile.out_p
  int oD, oH, oW;                // destination tensor dims
  const float* bias;             // [bias_n] real output channels, or nullptr
  int bias_n;
  int bias_wrap;                 // see the epilogue's bias load (0: plain)
  int act;                       // 0 none, 1 LeakyReLU(act_slope)
  float act_slope;
  float* stats;                  // [tile][2][w_rows_per_block] partial sum / sumsq, or nullptr
  // shared memory plan (bytes)
  int plane_stride, a_stage_bytes, b_stage_bytes, nsa, nsb, tmem_cols;
  int box_planes;                // > 1: ONE TMA box carries all n_in_planes planes of an A tile (planes bh * bw * pitch apart)
  int nacc;                      // TMEM accumulator sets (>= 2: the epilogue of a tile overlaps the next tiles' MMAs; <= kMaxAccSets)
  int total_tiles;
};

__device__ __forceinline__ void tmem_alloc_rt(uint32_t smem_slot, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_slot),
               "r"(ncols)
               : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc_rt(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}

__device__ __forceinline__ void named_bar_sync(int id, int nthreads) {
  asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}

// Sum over the 32 lanes of a warp of 32 per-lane values; lane l ends with the total of v[l].
__device__ __forceinline__ float warp_transpose_reduce32(float (&v)[32], int lane) {
#pragma unroll
  for (int off = 16, n = 32; off >= 1; off >>= 1, n >>= 1) {
    const bool hi = (lane & off) != 0;
#pragma unroll
    for (int i = 0; i < 16; ++i) {
      if (i < n / 2) {
        const float send = hi ? v[i] : v[i + n / 2];
        const float keep = hi ? v[i + n / 2] : v[i];
        v[i] = keep + __shfl_xor_sync(0xffffffffu, send, off);
      }
    }
  }
  return v[0];
}

__device__ __forceinline__ uint32_t pack_bf16x2(float lo, float hi) {
  __nv_bfloat162 t = __floats2bfloat162_rn(lo, hi);
  return *reinterpret_cast<uint32_t*>(&t);
}

constexpr int kIgemmThreads = 192;  // marching / wgrad kernels: warps 0-3 epilogue, warp 4 TMA producer, warp 5 MMA issuer
// Epilogue warps of the generic kernel. With statistics (forward convs in front of a norm) a thread carries 64
// per-channel accumulators. WITHOUT statistics -- every dgrad, the transposed convs, the PatchGAN stem -- a separate
// instantiation drops that code and its registers (168 -> 120): ncu showed the output-heavy launches of that group
// (transposed conv 64 -> 64: 2.1 GB written for 16 UMMAs per tile) bound by the epilogue's instruction stream, not by
// HBM or L2 (profiles/r02g_deconv_pair.txt). Sixteen epilogue warps for that instantiation were measured, removed: they
// do not pay (profiles/r02g_epi16.txt).
constexpr int kFwdEpiWarps = 8;
constexpr int kFwdThreads = (kFwdEpiWarps + 3) * 32;  // warps 0-7 epilogue, 8 TMA producer (A), 9 MMA issuer, 10 TMA producer (B)
constexpr int kFwdRedFloats = 2 * kFwdEpiWarps * 2 * 128 + 128;  // [parity][warp][sum|sumsq][128] + bias[128]

struct IgemmTileCoord {
  int w0, h0, d0, nb, planes;
};
__device__ __forceinline__ IgemmTileCoord igemm_tile(const IgemmParams& P, int t) {
  IgemmTileCoord c;
  const int tw_i = t % P.tiles_w; t /= P.tiles_w;
  const int th_i = t % P.tiles_h; t /= P.tiles_h;
  const int td_i = t % P.tiles_d; t /= P.tiles_d;
  c.nb = t;
  c.w0 = tw_i * 8; c.h0 = th_i * 16; c.d0 = td_i * P.td;
  c.planes = P.Do - c.d0; if (c.planes > P.td) c.planes = P.td;
  return c;
}

// First tap of a full folded tile: every output plane's first contribution (kd = 0) overwrites its accumulator, so
// the depth taps cannot share an instruction; same compile-time schedule, N = nt per UMMA.
template <int ND, int PL>
__device__ __forceinline__ void issue_first_tap(uint32_t acc0, uint32_t a_tap, uint32_t a_hi, uint32_t b_lo0, uint32_t b_hi,
                                                uint32_t ntc, uint32_t plane16, uint32_t kd_rows16, uint32_t idesc) {
  constexpr int ndm1 = ND - 1;
#pragma unroll
  for (int p_in = 0; p_in < PL + ndm1; ++p_in) {
    const int o_lo = p_in - ndm1 > 0 ? p_in - ndm1 : 0;
    const int o_hi = p_in < PL - 1 ? p_in : PL - 1;
#pragma unroll
    for (int o = o_lo; o <= o_hi; ++o) {
      const int kd = p_in - o;
      const uint32_t d = acc0 + (uint32_t)o * ntc;
      const uint32_t a = a_tap + (uint32_t)p_in * plane16;
      const uint32_t b = b_lo0 + (uint32_t)(ndm1 - kd) * kd_rows16;
      umma_bf16_lohi(d, a, a_hi, b, b_hi, idesc, (uint32_t)(kd != 0));
      umma_bf16_lohi(d, a + 2, a_hi, b + 2, b_hi, idesc, 1u);
    }
  }
}

template <int V> struct IntC { static constexpr int value = V; };

// Straight-line issue of one non-overwriting tap of a FULL folded tile (ND depth taps, FOLD of them per UMMA, PL output
// planes): the schedule of (halo plane, output-plane group) entries is a compile-time constant, so every operand is a
// constant multiple of three warp-uniform strides on top of three bases and the compiler keeps the whole run in the
// uniform datapath. The generic per-tile table (fs_* below) costs ~9 instructions per UMMA, most of them vector ->
// uniform register moves: 113 cycles per N = 64 UMMA against ~50 for its operands (profiles/r02f_stem_fwd_ncu_summary.txt).
template <int ND, int FOLD, int PL>
__device__ __forceinline__ void issue_folded_tap(uint32_t acc0, uint32_t a_tap, uint32_t a_hi, uint32_t b_lo0, uint32_t b_hi,
                                                 uint32_t ntc, uint32_t plane16, uint32_t kd_rows16,
                                                 const uint32_t (&idesc_blk)[3]) {
  constexpr int ndm1 = ND - 1;
#pragma unroll
  for (int p_in = 0; p_in < PL + ndm1; ++p_in) {
    const int o_lo = p_in - ndm1 > 0 ? p_in - ndm1 : 0;
    const int o_hi = p_in < PL - 1 ? p_in : PL - 1;
#pragma unroll
    for (int oa = o_lo; oa <= o_hi; oa += FOLD) {
      const int ob = oa + FOLD - 1 < o_hi ? oa + FOLD - 1 : o_hi;
      const uint32_t d = acc0 + (uint32_t)oa * ntc;
      const uint32_t a = a_tap + (uint32_t)p_in * plane16;
      const uint32_t b = b_lo0 + (uint32_t)(ndm1 - (p_in - oa)) * kd_rows16;
      const uint32_t id = idesc_blk[ob - oa];
      umma_bf16_lohi(d, a, a_hi, b, b_hi, id, 1u);
      umma_bf16_lohi(d, a + 2, a_hi, b + 2, b_hi, id, 1u);
    }
  }
}

// kMma = 2: TWO MMA-issuing warps that split the PLANES of a tile, each on its own accumulators. The host launches it
// for folded tiles only (launch_igemm: the four-plane schedule with three depth taps per UMMA). Why: the issue loop costs
// ~8 instructions per UMMA (each operand crosses from vector to uniform registers, R2UR), 113 cycles per N = 64 UMMA
// measured against ~50 for its shared-memory operands (profiles/r02f_stem_fwd_ncu_summary.txt), so every launch with
// N <= 128 per instruction is bound by ONE thread's issue rate. The stage / accumulator barriers count two commits.
// (Two warps issuing the two K = 16 halves of every instruction into the SAME accumulators were 8-35 % slower,
// profiles/r02g_mma2.txt: measured, removed.)
// Warp roles: 0 .. kFwdEpiWarps-1 epilogue, kFwdEpiWarps: TMA producer of the activation (A) stages, kFwdEpiWarps+1
// (.. +kMma): MMA issuer(s), last warp: TMA producer of the weight (B) ring. Two producers because ONE thread issuing every TMA operation bound the
// launches with little MMA work per box: the stem forward needs 40 A + 64 B boxes per tile, ~290 cycles each
// = the 30 k cycles per tile the launch took, against 16 k cycles of UMMAs (profiles/r02i_producer_ab.txt).
template <bool kStats, int kMma>
__global__ void __launch_bounds__((kFwdEpiWarps + 2 + kMma) * 32, 1)
igemm_fwd_kernel(const __grid_constant__ IgemmParams P) {
  constexpr int kEpi = kFwdEpiWarps;
  static_assert(kMma == 1 || kMma == 2, "one or two MMA-issuing warps");
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* sm = smem_raw + (base - smem_u32(smem_raw));
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

  const uint32_t a_base = base;
  const uint32_t b_base = a_base + P.nsa * P.a_stage_bytes;
  const uint32_t bar_base = b_base + P.nsb * P.b_stage_bytes;  // 8-byte mbarriers
  // barrier layout: a_full[nsa] a_empty[nsa] b_full[nsb] b_empty[nsb] acc_full[kMaxAccSets] acc_empty[kMaxAccSets]
  const uint32_t a_full = bar_base, a_empty = a_full + 8 * P.nsa, b_full = a_empty + 8 * P.nsa,
                 b_empty = b_full + 8 * P.nsb, acc_full = b_empty + 8 * P.nsb, acc_empty = acc_full + 8 * kMaxAccSets;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(sm + (acc_empty + 8 * kMaxAccSets - base));
  float* red = reinterpret_cast<float*>(sm + (((acc_empty + 8 * kMaxAccSets + 16 + 15) & ~15u) - base));  // kFwdRedFloats, 16-B aligned

  const IgemmNTile NT = P.ntile[blockIdx.y];
  const int ntc = (NT.nt + 31) & ~31;  // TMEM columns per plane accumulator
  const int acc_cols = P.td * ntc;     // columns of one accumulator set

  if (threadIdx.x == 0) {
    for (int i = 0; i < P.nsa; ++i) { mbar_init(a_full + 8 * i, 1); mbar_init(a_empty + 8 * i, kMma); }
    for (int i = 0; i < P.nsb; ++i) { mbar_init(b_full + 8 * i, 1); mbar_init(b_empty + 8 * i, kMma); }
    for (int i = 0; i < kMaxAccSets; ++i) { mbar_init(acc_full + 8 * i, kMma); mbar_init(acc_empty + 8 * i, kEpi); }
    fence_mbar_init();
  }
  if (warp == kEpi && lane == 0) {
    tma_prefetch_desc(&P.tm_src[0]);
    if (P.n_chunks_total > P.n_chunks_src0) tma_prefetch_desc(&P.tm_src[1]);
  }
  if (warp == kEpi + 1 + kMma && lane == 0) tma_prefetch_desc(&P.tm_w);
  if (warp == kEpi + 1) tmem_alloc_rt(smem_u32(tmem_slot), P.tmem_cols);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tmem_slot;
  constexpr int pitch = kIgemmKc * 2;

  if (warp == kEpi) {
    // =========================== TMA producer: activation stages ===========================
    if (lane == 0) {
      const uint32_t a_bytes = (uint32_t)(P.n_atiles * P.n_in_planes * P.bh * P.bw * pitch);
      int sa = 0;
      uint32_t pa = 0;
      for (int t = blockIdx.x; t < P.total_tiles; t += gridDim.x) {
        const IgemmTileCoord T = igemm_tile(P, t);
        for (int ch = 0; ch < P.n_chunks_total; ++ch) {
          mbar_wait(a_empty + 8 * sa, pa ^ 1);
          mbar_expect_tx(a_full + 8 * sa, a_bytes);
          const bool s1 = ch >= P.n_chunks_src0;
          const CUtensorMap* tm = &P.tm_src[s1 ? 1 : 0];
          const int grp = P.chunks_per_group ? ch / P.chunks_per_group : 0;
          const int c0 = P.chunks_per_group ? (ch % P.chunks_per_group) * kIgemmKc : (s1 ? ch - P.n_chunks_src0 : ch) * kIgemmKc;
          const int nb5 = P.chunks_per_group ? T.nb * (P.n_chunks_total / P.chunks_per_group) + grp : T.nb;
          uint32_t dst = a_base + sa * P.a_stage_bytes;
          for (int at = 0; at < P.n_atiles; ++at) {
            const int oi = P.chunks_per_group ? grp : at + NT.tapset;
            const int cw = T.w0 * P.in_stride + P.atile_off[oi][0];
            const int chh = T.h0 * P.in_stride + P.atile_off[oi][1];
            if (P.box_planes > 1) {
              // one box for all the planes of the tile (out-of-volume planes are zero-filled like the halo rows)
              tma_load_5d(dst, tm, a_full + 8 * sa, c0, cw, chh, T.d0 * P.in_stride + P.atile_off[oi][2], nb5);
              dst += P.n_in_planes * P.plane_stride;
            } else {
              for (int p = 0; p < P.n_in_planes; ++p, dst += P.plane_stride) {
                const int cd = (T.d0 + p) * P.in_stride + P.atile_off[oi][2];
                tma_load_5d(dst, tm, a_full + 8 * sa, c0, cw, chh, cd, nb5);
              }
            }
          }
          if (++sa == P.nsa) { sa = 0; pa ^= 1; }
        }
      }
    }
    __syncwarp();
  } else if (warp == kEpi + 1 + kMma) {
    // =========================== TMA producer: weight ring ===========================
    if (lane == 0) {
      const uint32_t b_bytes = (uint32_t)((P.kd_fold ? P.fold_nd : 1) * NT.nt * pitch);
      int sb = 0;
      uint32_t pb = 0;
      for (int t = blockIdx.x; t < P.total_tiles; t += gridDim.x) {
        for (int ch = 0; ch < P.n_chunks_total; ++ch) {
          const int grp = P.chunks_per_group ? ch / P.chunks_per_group : 0;
          const int wk = (P.chunks_per_group ? ch % P.chunks_per_group : ch) * kIgemmKc;
          const IgemmTap* taps = P.taps + (P.chunks_per_group ? grp : NT.tapset) * P.ntaps;
          for (int tp = 0; tp < P.ntaps; ++tp) {
            mbar_wait(b_empty + 8 * sb, pb ^ 1);
            mbar_expect_tx(b_full + 8 * sb, b_bytes);
            const int brow = (taps[tp].wblock + NT.wblock_add) * P.b_block_rows + NT.n0;
            tma_load_2d(b_base + sb * P.b_stage_bytes, &P.tm_w, b_full + 8 * sb, wk, brow);
            // the other depth-tap blocks of the folded tile, one box each (TMA boxes hold <= 256 rows). The blocks of a
            // 3x3x3 tile are adjacent in the pack; one merged box for them measured neutral, removed
            // (profiles/r02i_wbox_ab.txt: these launches are not bound by the producer's issue rate).
            if (P.kd_fold) {
              for (int j = 1; j < P.fold_nd; ++j)
                tma_load_2d(b_base + sb * P.b_stage_bytes + j * NT.nt * pitch, &P.tm_w, b_full + 8 * sb, wk,
                            brow + j * P.fold_row_step);
            }
            if (++sb == P.nsb) { sb = 0; pb ^= 1; }
          }
        }
      }
    }
    __syncwarp();
  } else if (warp >= kEpi + 1) {
    // =========================== MMA issuer(s): warps kEpi+1 .. kEpi+kMma ===========================
    // The whole warp walks the pipeline (uniform control flow); one elected lane issues.
    const int ph = kMma == 2 ? warp - (kEpi + 1) : 0;        // this warp's index among the issuers (its half of the planes)
    const uint32_t idesc = make_idesc_bf16(128, NT.nt, 0, 0);
    const uint32_t a_hi = (uint32_t)(make_smem_desc(0, 16, P.bw * pitch, SWZ_64B) >> 32);
    const uint32_t b_hi = (uint32_t)(make_smem_desc(0, 16, 8 * pitch, SWZ_64B) >> 32);
    const uint32_t lbo_lo = 1u << 16;  // LBO field (16 bytes) lives in the low word
    const uint32_t plane16 = (uint32_t)P.plane_stride >> 4;
    const bool leader = elect_one();
    // depth-tap folding constants
    const int fold = P.kd_fold, ndm1 = P.fold_nd - 1;
    const uint32_t kd_rows16 = (uint32_t)(NT.nt * pitch) >> 4;   // one depth-tap block of the weight tile
    uint32_t idesc_blk[3];
#pragma unroll
    for (int i = 0; i < 3; ++i) idesc_blk[i] = make_idesc_bf16(128, (i + 1) * NT.nt <= 256 ? (i + 1) * NT.nt : NT.nt, 0, 0);
    int sa = 0, sb = 0, slot = 0;
    uint32_t pa = 0, pb = 0, pacc = 0;
    for (int t = blockIdx.x; t < P.total_tiles; t += gridDim.x) {
      const IgemmTileCoord T = igemm_tile(P, t);
      const int n_pin = T.planes + ndm1;
      // folded schedule of this tile: entry e = (halo plane p_in, UMMA group gi): accumulator column
      // offset, A plane offset, weight block offset, instruction descriptor (N = 1..3 depth blocks)
      uint32_t fs_d[12], fs_a[12], fs_b[12], fs_i[12], fs_valid = 0;
      // 1: (3 depth taps, 3 per UMMA, 4 planes)  2: (3, 2, 2)  3: (2, 2, 4)  0: the table
      const int sched = !fold ? 0
                        : (P.fold_nd == 3 && fold == 3 && T.planes == 4) ? 1
                        : (P.fold_nd == 3 && fold == 2 && T.planes == 2) ? 2
                        : (P.fold_nd == 2 && fold == 2 && T.planes == 4) ? 3 : 0;
      if (fold && sched == 0 && ph == 0) {   // (a second issuer leaves such tiles to the first)
#pragma unroll
        for (int p_in = 0; p_in < 6; ++p_in) {
#pragma unroll
          for (int gi = 0; gi < 2; ++gi) {
            const int e = p_in * 2 + gi;
            const int o_lo = p_in - ndm1 > 0 ? p_in - ndm1 : 0;
            const int o_hi = p_in < T.planes - 1 ? p_in : T.planes - 1;
            const int oa = o_lo + gi * fold;
            const int ob = oa + fold - 1 < o_hi ? oa + fold - 1 : o_hi;
            const bool v = p_in < n_pin && oa <= o_hi;
            const int nb_ = ob - oa;
            fs_d[e] = (uint32_t)(oa * ntc);
            fs_a[e] = (uint32_t)p_in * plane16;
            fs_b[e] = (uint32_t)(ndm1 - (p_in - oa)) * kd_rows16;
            fs_i[e] = nb_ <= 0 ? idesc_blk[0] : (nb_ == 1 ? idesc_blk[1] : idesc_blk[2]);
            fs_valid |= (v ? 1u : 0u) << e;
          }
        }
      }
      mbar_wait(acc_empty + 8 * slot, pacc ^ 1);
      tc_fence_after();
      const uint32_t acc0 = tmem + slot * acc_cols;
      for (int ch = 0; ch < P.n_chunks_total; ++ch) {
        mbar_wait(a_full + 8 * sa, pa);
        tc_fence_after();
        const uint32_t a_stage = a_base + sa * P.a_stage_bytes;
        const int tbase = (P.chunks_per_group ? ch / P.chunks_per_group : NT.tapset) * P.ntaps;
        for (int tp = 0; tp < P.ntaps; ++tp) {
          mbar_wait(b_full + 8 * sb, pb);
          tc_fence_after();
          if (leader && P.kd_fold) {
            const IgemmTap Tp = P.taps[tbase + tp];
            const uint32_t a_tap = lbo_lo | ((a_stage + Tp.row_off * pitch) >> 4);
            const uint32_t b_lo0 = lbo_lo | ((b_base + sb * P.b_stage_bytes) >> 4);
            if (kMma == 2 && sched != 0) {
              // plane-split issuers: each warp runs the schedule of HALF the tile's planes on its own accumulators --
              // (3, 3, 4) -> two (3, 2, 2) halves, (3, 2, 2) -> two (3, 1, 1), (2, 2, 4) -> two (2, 2, 2)
              const uint32_t nh = sched == 2 ? 1u : 2u;                       // output planes per issuer
              const uint32_t accp = acc0 + (uint32_t)ph * nh * (uint32_t)ntc, a_p = a_tap + (uint32_t)ph * nh * plane16;
              if ((ch | tp) != 0) {
                if (sched == 1) issue_folded_tap<3, 2, 2>(accp, a_p, a_hi, b_lo0, b_hi, (uint32_t)ntc, plane16, kd_rows16, idesc_blk);
                else if (sched == 2) issue_folded_tap<3, 1, 1>(accp, a_p, a_hi, b_lo0, b_hi, (uint32_t)ntc, plane16, kd_rows16, idesc_blk);
                else issue_folded_tap<2, 2, 2>(accp, a_p, a_hi, b_lo0, b_hi, (uint32_t)ntc, plane16, kd_rows16, idesc_blk);
              } else {
                if (sched == 1) issue_first_tap<3, 2>(accp, a_p, a_hi, b_lo0, b_hi, (uint32_t)ntc, plane16, kd_rows16, idesc);
                else if (sched == 2) issue_first_tap<3, 1>(accp, a_p, a_hi, b_lo0, b_hi, (uint32_t)ntc, plane16, kd_rows16, idesc);
                else issue_first_tap<2, 2>(accp, a_p, a_hi, b_lo0, b_hi, (uint32_t)ntc, plane16, kd_rows16, idesc);
              }
            } else if (kMma == 2 && ph == 1) {
              // ragged tile: the first issuer runs the whole table, this one only commits
            } else if ((ch | tp) != 0 && sched != 0) {
              // full tile of one of the three shapes the step uses: compile-time schedule
              if (sched == 1) issue_folded_tap<3, 3, 4>(acc0, a_tap, a_hi, b_lo0, b_hi, (uint32_t)ntc, plane16, kd_rows16, idesc_blk);
              else if (sched == 2) issue_folded_tap<3, 2, 2>(acc0, a_tap, a_hi, b_lo0, b_hi, (uint32_t)ntc, plane16, kd_rows16, idesc_blk);
              else issue_folded_tap<2, 2, 4>(acc0, a_tap, a_hi, b_lo0, b_hi, (uint32_t)ntc, plane16, kd_rows16, idesc_blk);
            } else if ((ch | tp) != 0) {
              // any other tile (ragged depth, other fold shapes): the per-tile schedule table (fs_*)
#pragma unroll
              for (int e = 0; e < 12; ++e) {
                if ((fs_valid >> e) & 1u) {
                  umma_bf16_lohi(acc0 + fs_d[e], a_tap + fs_a[e], a_hi, b_lo0 + fs_b[e], b_hi, fs_i[e], 1u);
                  umma_bf16_lohi(acc0 + fs_d[e], a_tap + fs_a[e] + 2, a_hi, b_lo0 + fs_b[e] + 2, b_hi, fs_i[e], 1u);
                }
              }
            } else if (sched != 0) {
              if (sched == 1) issue_first_tap<3, 4>(acc0, a_tap, a_hi, b_lo0, b_hi, (uint32_t)ntc, plane16, kd_rows16, idesc);
              else if (sched == 2) issue_first_tap<3, 2>(acc0, a_tap, a_hi, b_lo0, b_hi, (uint32_t)ntc, plane16, kd_rows16, idesc);
              else issue_first_tap<2, 4>(acc0, a_tap, a_hi, b_lo0, b_hi, (uint32_t)ntc, plane16, kd_rows16, idesc);
            } else {
              // first tap of the tile: each output plane's first contribution (kd = 0) overwrites
              for (int p_in = 0; p_in < n_pin; ++p_in) {
                const int o_lo = p_in - ndm1 > 0 ? p_in - ndm1 : 0;
                const int o_hi = p_in < T.planes - 1 ? p_in : T.planes - 1;
                const uint32_t a_lo = a_tap + p_in * plane16;
                for (int o = o_lo; o <= o_hi; ++o) {
                  const int kd = p_in - o;
                  const uint32_t b_lo = b_lo0 + (uint32_t)(ndm1 - kd) * kd_rows16;
                  umma_bf16_lohi(acc0 + o * ntc, a_lo, a_hi, b_lo, b_hi, idesc, (uint32_t)(kd != 0));
                  umma_bf16_lohi(acc0 + o * ntc, a_lo + 2, a_hi, b_lo + 2, b_hi, idesc, 1u);
                }
              }
            }
            umma_commit(b_empty + 8 * sb);
          } else if (leader) {
            const IgemmTap Tp = P.taps[tbase + tp];
            const uint32_t a_lo = lbo_lo | ((a_stage + (Tp.atile * P.n_in_planes + Tp.plane_off) * P.plane_stride +
                                             Tp.row_off * pitch) >> 4);
            const uint32_t b_lo = lbo_lo | ((b_base + sb * P.b_stage_bytes) >> 4);
            const uint32_t acc = (ch | tp) != 0;
            // one branch per tap, not per plane: the planes of a tap are then one straight run of UMMAs (every branch
            // in between makes the compiler move all seven operands to uniform registers again)
            auto planes = [&](auto pl) {
              constexpr int PL = decltype(pl)::value;
#pragma unroll
              for (int o = 0; o < PL; ++o) {
                umma_bf16_lohi(acc0 + o * ntc, a_lo + o * plane16, a_hi, b_lo, b_hi, idesc, acc);
                umma_bf16_lohi(acc0 + o * ntc, a_lo + o * plane16 + 2, a_hi, b_lo + 2, b_hi, idesc, 1u);
              }
            };
            if (T.planes == 4) planes(IntC<4>{});
            else if (T.planes == 2) planes(IntC<2>{});
            else if (T.planes == 1) planes(IntC<1>{});
            else planes(IntC<3>{});
            umma_commit(b_empty + 8 * sb);
          }
          __syncwarp();
          if (++sb == P.nsb) { sb = 0; pb ^= 1; }
        }
        if (leader) umma_commit(a_empty + 8 * sa);
        __syncwarp();
        if (++sa == P.nsa) { sa = 0; pa ^= 1; }
      }
      if (leader) umma_commit(acc_full + 8 * slot);
      __syncwarp();
      if (++slot == P.nacc) { slot = 0; pacc ^= 1; }
    }
  } else {
    // =========================== epilogue (warps 0 .. kEpi-1) ===========================
    // warp w reads TMEM lanes 32*(w%4)..+31 (accumulator rows); the kEpi / 4 warps of a lane quarter split
    // the (plane, 32-column chunk) units of a tile between them.
    const int q = warp & 3, grp = warp >> 2;
    constexpr int kGroups = kEpi / 4;
    const int r = q * 32 + lane;
    const bool do_stats = kStats && P.stats != nullptr;
    const bool do_act = P.act == 1;
    const float slope = P.act_slope;
    const int nchunks = (NT.nt + 31) >> 5;
    // bias of this N tile -> smem (zero where there is none), read back as broadcast float4
    float* bias_s = red + 2 * kFwdEpiWarps * 2 * 128;  // [128]
    if (threadIdx.x < 128) {
      const int c = threadIdx.x;
      // bias_wrap > 0: the N tile holds several copies of the output channels (two sub-positions of a transposed conv
      // side by side): column c carries channel (n0 + c) mod bias_wrap
      const int bc = P.bias_wrap > 0 ? (NT.n0 + c) % P.bias_wrap : NT.n0 + c;
      bias_s[c] = (P.bias != nullptr && c < NT.nt && bc < P.bias_n) ? __ldg(P.bias + bc) : 0.f;
    }
    named_bar_sync(1, kEpi * 32);
    __nv_bfloat16* outp = reinterpret_cast<__nv_bfloat16*>(NT.out);
    __nv_bfloat16* outp2 = reinterpret_cast<__nv_bfloat16*>(NT.out2);
    const bool odd = (lane & 1) != 0;
    int slot = 0, it = 0;
    uint32_t pacc = 0;
    // per-thread channel sums (statistics variant). With ONE 32-column chunk per tile (the 1x1x1 input head) they are
    // carried over the CTA's consecutive tiles of a sample and transposed / written only when the sample changes or the
    // CTA runs out of tiles -- the other tiles write a zero record. That launch has 8 UMMAs per tile and was bound by
    // the epilogue's per-tile transpose-reduce (2 x 31 shuffle steps, a block barrier and a shared-memory round trip).
    float st_a[kStats ? 32 : 1], st_b[kStats ? 32 : 1];
#pragma unroll
    for (int j = 0; j < (kStats ? 32 : 1); ++j) { st_a[j] = 0.f; st_b[j] = 0.f; }
    const bool carry = kStats && do_stats && nchunks == 1;
    for (int t = blockIdx.x; t < P.total_tiles; t += gridDim.x, ++it) {
      const IgemmTileCoord T = igemm_tile(P, t);
      const int h = T.h0 + (r >> 3), w = T.w0 + (r & 7);
      const bool valid_hw = (h < P.Ho) && (w < P.Wo);
      const bool valid_pair = (h < P.Ho) && ((w ^ 1) < P.Wo);   // the partner lane's row (w +- 1)
      // rows of the lane pair: even lane's row first
      const bool valid_e = odd ? valid_pair : valid_hw, valid_o = odd ? valid_hw : valid_pair;
      const size_t vox_hw = (size_t)(h * P.out_s + NT.out_p[1]) * P.oW + (size_t)((w & ~1) * P.out_s + NT.out_p[0]);
      float s_acc[4] = {0.f, 0.f, 0.f, 0.f}, q_acc[4] = {0.f, 0.f, 0.f, 0.f};
      mbar_wait(acc_full + 8 * slot, pacc);
      tc_fence_after();
      const uint32_t acc0 = tmem + ((uint32_t)(q * 32) << 16) + slot * acc_cols;

      // one (32-column chunk cc, plane o) unit of the tile: TMEM -> bias / activation -> 16-bit -> global
      auto unit = [&](int cc, int o, float (&st_a)[kStats ? 32 : 1], float (&st_b)[kStats ? 32 : 1]) {
        const bool full32 = (NT.nt - cc * 32) >= 32;
        const bool to2 = cc * 32 >= NT.split;
        const float4* b4 = reinterpret_cast<const float4*>(bias_s + cc * 32);
        const int d = T.d0 + o;
        const size_t vox_e = ((size_t)T.nb * P.oD + (size_t)(d * P.out_s + NT.out_p[2])) * P.oH * P.oW + vox_hw;
        uint32_t rr[32];
        const uint32_t taddr = acc0 + o * ntc + cc * 32;
        if (full32) {
          tmem_ld_32x32b_x32(taddr, rr);
        } else {
          uint32_t r16[16];
          tmem_ld_32x32b_x16(taddr, r16);
#pragma unroll
          for (int j = 0; j < 16; ++j) { rr[j] = r16[j]; rr[j + 16] = 0u; }
        }
        tmem_ld_wait();
        uint32_t pk[16];
        const bool acc_stats = do_stats && valid_hw;
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          const float4 bv = b4[j];
          float x0 = __uint_as_float(rr[4 * j + 0]) + bv.x, x1 = __uint_as_float(rr[4 * j + 1]) + bv.y;
          float x2 = __uint_as_float(rr[4 * j + 2]) + bv.z, x3 = __uint_as_float(rr[4 * j + 3]) + bv.w;
          if (do_act) {
            x0 = x0 > 0.f ? x0 : x0 * slope; x1 = x1 > 0.f ? x1 : x1 * slope;
            x2 = x2 > 0.f ? x2 : x2 * slope; x3 = x3 > 0.f ? x3 : x3 * slope;
          }
          if (kStats && do_stats) {
            // the raw output of a conv -> norm block: stored as fp16 (never an MMA operand), statistics from
            // the fp32 accumulators
            pk[2 * j] = pack_f16x2_sat(x0, x1);
            pk[2 * j + 1] = pack_f16x2_sat(x2, x3);
            if (acc_stats) {
              if constexpr (kStats) {
                st_a[4 * j] += x0; st_a[4 * j + 1] += x1; st_a[4 * j + 2] += x2; st_a[4 * j + 3] += x3;
                st_b[4 * j] = fmaf(x0, x0, st_b[4 * j]); st_b[4 * j + 1] = fmaf(x1, x1, st_b[4 * j + 1]);
                st_b[4 * j + 2] = fmaf(x2, x2, st_b[4 * j + 2]); st_b[4 * j + 3] = fmaf(x3, x3, st_b[4 * j + 3]);
              }
            }
          } else {
            pk[2 * j] = pack_bf16x2(x0, x1);
            pk[2 * j + 1] = pack_bf16x2(x2, x3);
          }
        }
        // ---- stores: the lane pair (2k, 2k+1) owns two neighbouring voxel rows (w, w+1). Exchange half
        // rows so that instruction j writes one whole 32-byte sector per lane pair:
        //   even lane: row_e chunk 0 | row_e chunk 2 | row_o chunk 0 | row_o chunk 2
        //   odd  lane: row_e chunk 1 | row_e chunk 3 | row_o chunk 1 | row_o chunk 3
        uint32_t sx[8], rx[8];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          sx[j] = odd ? pk[j] : pk[4 + j];            // odd sends chunk 0, even sends chunk 1
          sx[4 + j] = odd ? pk[8 + j] : pk[12 + j];   // odd sends chunk 2, even sends chunk 3
        }
#pragma unroll
        for (int j = 0; j < 8; ++j) rx[j] = __shfl_xor_sync(0xffffffffu, sx[j], 1);
        __nv_bfloat16* be = to2 ? outp2 + vox_e * NT.out2_cpitch + (cc * 32 - NT.split)
                                : outp + vox_e * NT.out_cpitch + NT.out_coff + cc * 32;
        const size_t row_step = (size_t)P.out_s * (to2 ? NT.out2_cpitch : NT.out_cpitch);
        uint4* de = reinterpret_cast<uint4*>(be) + (odd ? 1 : 0);
        uint4* d_o = reinterpret_cast<uint4*>(be + row_step) + (odd ? 1 : 0);
        if (valid_e) {
          __stcs(de + 0, odd ? make_uint4(rx[0], rx[1], rx[2], rx[3]) : make_uint4(pk[0], pk[1], pk[2], pk[3]));
          if (full32) __stcs(de + 2, odd ? make_uint4(rx[4], rx[5], rx[6], rx[7]) : make_uint4(pk[8], pk[9], pk[10], pk[11]));
        }
        if (valid_o) {
          __stcs(d_o + 0, odd ? make_uint4(pk[4], pk[5], pk[6], pk[7]) : make_uint4(rx[0], rx[1], rx[2], rx[3]));
          if (full32) __stcs(d_o + 2, odd ? make_uint4(pk[12], pk[13], pk[14], pk[15]) : make_uint4(rx[4], rx[5], rx[6], rx[7]));
        }
      };

      bool flush = true;       // this tile writes a real statistics record (always, unless the sums are carried on)
      if constexpr (kStats) {
        // the two warps of a lane quarter split the tile by 32-column chunk when their number is even,
        // else by plane; per-channel statistics are summed in registers over the planes of a chunk and
        // transposed once per (chunk, tile)
        const bool by_chunk = (nchunks & 1) == 0;
        if (carry) {
          const int tn = t + (int)gridDim.x;
          flush = tn >= P.total_tiles || igemm_tile(P, tn).nb != T.nb;
        }
        for (int cc = by_chunk ? grp : 0; cc < nchunks; cc += by_chunk ? 2 : 1) {
          if (!carry) {
#pragma unroll
            for (int j = 0; j < 32; ++j) { st_a[j] = 0.f; st_b[j] = 0.f; }
          }
          for (int o = by_chunk ? 0 : grp; o < T.planes; o += by_chunk ? 1 : 2) unit(cc, o, st_a, st_b);
          if (do_stats && flush) {
            const float sa_ = warp_transpose_reduce32(st_a, lane);     // (destroys its argument)
            const float sq_ = warp_transpose_reduce32(st_b, lane);
#pragma unroll
            for (int k = 0; k < 4; ++k)
              if (k == cc) { s_acc[k] = sa_; q_acc[k] = sq_; }
            if (carry) {
#pragma unroll
              for (int j = 0; j < 32; ++j) { st_a[j] = 0.f; st_b[j] = 0.f; }
            }
          }
        }
      } else {
        // no statistics: the (chunk, plane) units go round-robin over the kEpi / 4 warps of the lane quarter
        float dummy_a[1], dummy_b[1];
        const int nunits = nchunks * T.planes;
        for (int u = grp; u < nunits; u += kGroups) unit(u % nchunks, u / nchunks, dummy_a, dummy_b);
      }
      // all TMEM reads of this tile are done: hand the accumulator set back to the MMA warp
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(acc_empty + 8 * slot);
      if (++slot == P.nacc) { slot = 0; pacc ^= 1; }
      if constexpr (kStats) {
        if (do_stats && !flush) {
          // sums carried on to the CTA's next tile of this sample: this tile's record is zero
          const int c = threadIdx.x;
          if (c < NT.nt) {
            float* st = P.stats + (size_t)t * 2 * P.w_rows_per_block;
            st[NT.n0 + c] = 0.f;
            st[P.w_rows_per_block + NT.n0 + c] = 0.f;
          }
        } else if (do_stats) {
          float* rd = red + (it & 1) * (kFwdEpiWarps * 2 * 128);
          for (int cc = 0; cc < nchunks; ++cc) {
            float s = 0.f, qq = 0.f;
#pragma unroll
            for (int k = 0; k < 4; ++k)
              if (k == cc) { s = s_acc[k]; qq = q_acc[k]; }
            rd[(warp * 2 + 0) * 128 + cc * 32 + lane] = s;
            rd[(warp * 2 + 1) * 128 + cc * 32 + lane] = qq;
          }
          named_bar_sync(1, kEpi * 32);
          const int c = threadIdx.x;
          if (c < NT.nt) {
            float s = 0.f, qq = 0.f;
#pragma unroll
            for (int wq = 0; wq < kFwdEpiWarps; ++wq) { s += rd[(wq * 2 + 0) * 128 + c]; qq += rd[(wq * 2 + 1) * 128 + c]; }
            float* st = P.stats + (size_t)t * 2 * P.w_rows_per_block;
            st[NT.n0 + c] = s;
            st[P.w_rows_per_block + NT.n0 + c] = qq;
          }
        }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == kEpi + 1) tmem_dealloc_rt(tmem, P.tmem_cols);
}

}  // namespace ub
