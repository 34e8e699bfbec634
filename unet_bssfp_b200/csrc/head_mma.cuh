// Output head of the generator on warp-level tensor-core MMAs (mma.sync, sm_100a):
//   forward   out[co][v] = b[co] + sum_ch W[co][ch] * u[v][ch]          ref: monai BasicUNet.final_conv (Conv3d(32, 6, 1)),
//   backward  du[v][ch]  = sum_co g[co][v] * W[co][ch]                   ref:model.py:22-28; u = the deferred activations of
//             dW[co][ch] = sum_v g[co][v] * u[v][ch],  db[co] = sum_v g[co][v]        upcat_1.conv_1 (conv -> IN -> dropout -> LReLU)
//
// Why: these are HBM-bound ops by their bytes (24 B of result per 64 B voxel row), but the CUDA-core kernels in
// pointwise.cuh were ISSUE-bound -- ncu (profiles/r02b_head_*_ncu_summary.txt): 217 / 331 warp instructions per 16-byte
// vector, sm throughput 68 % / 48 % at 2.4 / 2.0 TB/s of DRAM traffic -- because a 6 x 32 matvec per voxel costs 48
// FFMA + 12 SHFL per thread. A warp-level m16n8k16 / m16n8k8 bf16 MMA does the same contraction for 8 (forward) or 16
// (backward) voxels in ONE instruction, and the fragment layouts can be chosen so that no data moves between lanes:
//
//   lane = (gid, tig) = (lane >> 2, lane & 3) owns the channel octet `tig` of voxel `gid` of a group of 8 consecutive
//   voxels -- the same 16-byte vectors the pointwise kernels load (a warp reads 512 contiguous bytes). Its four packed
//   registers U[r] = channels (8 tig + 2r, 8 tig + 2r + 1) ARE the B fragment of the forward MMA (k <-> the lane's own
//   channels, n <-> its voxel), and the D fragment of the backward MMA du = g^T W (m <-> voxel, n <-> channel) lands
//   as du[own voxel][own octet] when the weight fragment's columns are permuted accordingly. Only the weight-gradient
//   MMA (k <-> voxel) needs its operands transposed, which is one `movmatrix` per register.
//
// The backward is fused with the norm backward of the block in front of the head (the block is never materialised,
// section 3.7 of DESIGN.md): kernel 1 accumulates dW, db AND that block's reductions S1 = sum dz, S2 = sum dz * xhat
// from du without writing du; after the finalize, kernel 2 recomputes du and writes the block's dy directly.
// HBM traffic of the chain: (0.4 + 1.07) + (0.4 + 1.07 + 1.07) GB instead of 7.9 GB in three passes.
#pragma once
#include "pointwise.cuh"

namespace ub {

__device__ __forceinline__ uint32_t movmatrix_trans(uint32_t a) {
  uint32_t d;
  asm volatile("movmatrix.sync.aligned.m8n8.trans.b16 %0, %1;" : "=r"(d) : "r"(a));
  return d;
}
// D (16x8 fp32) += A (16x16 bf16, row) * B (16x8 bf16, col)
__device__ __forceinline__ void mma_bf16_16816(float (&c)[4], uint32_t a0, uint32_t a1, uint32_t a2, uint32_t a3,
                                               uint32_t b0, uint32_t b1) {
  asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
               : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
               : "r"(a0), "r"(a1), "r"(a2), "r"(a3), "r"(b0), "r"(b1));
}
// D (16x8 fp32) += A (16x8 bf16, row) * B (8x8 bf16, col)
__device__ __forceinline__ void mma_bf16_1688(float (&c)[4], uint32_t a0, uint32_t a1, uint32_t b0) {
  asm volatile("mma.sync.aligned.m16n8k8.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5}, {%6}, {%0,%1,%2,%3};"
               : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
               : "r"(a0), "r"(a1), "r"(b0));
}
__device__ __forceinline__ uint32_t pack_bf16_pair(float lo, float hi) {
  const __nv_bfloat162 t = __floats2bfloat162_rn(lo, hi);
  return *reinterpret_cast<const uint32_t*>(&t);
}

// ------------------------------------------------------------------------------------------------
// forward. grid = (blocks, N), block = 256 (8 warps); a warp walks groups of 8 voxels, kHeadFwdUnroll loads in flight.
// V % 8 == 0. The fp32 weights enter as three bf16 terms hi + mid + lo (three MMAs per k-step): W is reproduced exactly,
// so the result matches the fp32-weight CUDA-core kernel to fp32 summation order.
// ------------------------------------------------------------------------------------------------
constexpr int kHeadFwdUnroll = 4;
template <int CO, bool DEFERRED>
__global__ void __launch_bounds__(256)
head_fwd_mma_kernel(const __nv_bfloat16* __restrict__ u, float* __restrict__ out, const Conv1x1Weights* __restrict__ Wg,
                    uint32_t V, NormActArgs A) {
  const int n = blockIdx.y;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int gid = lane >> 2, tig = lane & 3;
  // A fragments (row = co = gid; rows 8..15 are padding): k-step s, register h: W[gid][8 tig + 4 s + 2 h + {0, 1}]
  uint32_t ah[2][2], am[2][2], al[2][2];     // W = hi + mid + lo, three bf16 terms: 24 significand bits, i.e. exact
#pragma unroll
  for (int s = 0; s < 2; ++s)
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      const int c = 8 * tig + 4 * s + 2 * h;
      const float w0 = gid < CO ? Wg->w[gid][c] : 0.f, w1 = gid < CO ? Wg->w[gid][c + 1] : 0.f;
      const float h0 = __bfloat162float(__float2bfloat16_rn(w0)), h1 = __bfloat162float(__float2bfloat16_rn(w1));
      const float r0 = w0 - h0, r1 = w1 - h1;
      const float m0 = __bfloat162float(__float2bfloat16_rn(r0)), m1 = __bfloat162float(__float2bfloat16_rn(r1));
      ah[s][h] = pack_bf16_pair(h0, h1);
      am[s][h] = pack_bf16_pair(m0, m1);
      al[s][h] = pack_bf16_pair(r0 - m0, r1 - m1);
    }
  const float br = gid < CO ? Wg->b[gid] : 0.f;
  DeferredOctet K;
  if (DEFERRED) K.load(A, n, 32, tig * 8);
  const bf16x8* up = reinterpret_cast<const bf16x8*>(u) + (size_t)n * V * 4;
  float* op = out + (size_t)n * CO * V;
  const uint32_t ngroups = V >> 3;
  const uint32_t gstep = gridDim.x * 8u * kHeadFwdUnroll;
  for (uint32_t g0 = (blockIdx.x * 8u + warp) * kHeadFwdUnroll; g0 < ngroups; g0 += gstep) {   // warp-uniform
    bf16x8 raw[kHeadFwdUnroll];
#pragma unroll
    for (int q = 0; q < kHeadFwdUnroll; ++q)
      if (g0 + q < ngroups) raw[q] = ld_stream(up + (size_t)((g0 + q) * 8u + gid) * 4 + tig);
#pragma unroll
    for (int q = 0; q < kHeadFwdUnroll; ++q) {
      const uint32_t g = g0 + q;
      if (g >= ngroups) break;                                                               // warp-uniform
      const uint32_t v = g * 8u + gid;
      const bf16x8 a8 = DEFERRED ? K.apply(raw[q], ((unsigned long long)n * V + v) * 32ull + tig * 8) : raw[q];
      const uint32_t* U = reinterpret_cast<const uint32_t*>(&a8);
      float c[4] = {0.f, 0.f, 0.f, 0.f};
      mma_bf16_16816(c, al[0][0], 0u, al[0][1], 0u, U[0], U[1]);      // smallest terms first
      mma_bf16_16816(c, al[1][0], 0u, al[1][1], 0u, U[2], U[3]);
      mma_bf16_16816(c, am[0][0], 0u, am[0][1], 0u, U[0], U[1]);
      mma_bf16_16816(c, am[1][0], 0u, am[1][1], 0u, U[2], U[3]);
      mma_bf16_16816(c, ah[0][0], 0u, ah[0][1], 0u, U[0], U[1]);
      mma_bf16_16816(c, ah[1][0], 0u, ah[1][1], 0u, U[2], U[3]);
      // D[row = co = gid][col = voxel 2 tig + {0, 1}]: 8 bytes per lane, 32 contiguous bytes per channel plane
      if (gid < CO) __stcs(reinterpret_cast<float2*>(op + (size_t)gid * V + g * 8u + 2 * tig), make_float2(c[0] + br, c[1] + br));
    }
  }
}

// ------------------------------------------------------------------------------------------------
// backward, shared pieces. A unit = 16 voxels = group a (rows 0..7 of the MMA) + group b (rows 8..15).
// ------------------------------------------------------------------------------------------------
// B fragments of du = g^T W for the four column blocks nb: rows k = co = 2 tig + {0, 1}, column n = gid <-> channel
// 8 (gid >> 1) + 2 nb + (gid & 1), so that D[voxel gid][2 tig + e] is channel 8 tig + 2 nb + e: the lane's own octet.
template <int CO>
__device__ __forceinline__ void head_du_weights(const Conv1x1Weights* __restrict__ Wg, int gid, int tig, uint32_t (&bw)[4]) {
#pragma unroll
  for (int nb = 0; nb < 4; ++nb) {
    const int ch = 8 * (gid >> 1) + 2 * nb + (gid & 1);
    const float w0 = 2 * tig < CO ? Wg->w[2 * tig][ch] : 0.f, w1 = 2 * tig + 1 < CO ? Wg->w[2 * tig + 1][ch] : 0.f;
    bw[nb] = pack_bf16_pair(w0, w1);
  }
}
struct HeadUnitLoad {
  bf16x8 ya, yb;        // the lane's y octet of its voxel in group a / b
  float g[4];           // dout[2 tig][va], dout[2 tig + 1][va], dout[2 tig][vb], dout[2 tig + 1][vb]
};
template <int CO>
__device__ __forceinline__ void head_unit_load(HeadUnitLoad& L, const float* __restrict__ gp, const bf16x8* __restrict__ yp,
                                               uint32_t V, uint32_t va, int tig) {
  L.ya = ld_stream(yp + (size_t)va * 4 + tig);
  L.yb = ld_stream(yp + (size_t)(va + 8) * 4 + tig);
  const int c0 = 2 * tig;
  L.g[0] = c0 < CO ? __ldg(gp + (size_t)c0 * V + va) : 0.f;
  L.g[1] = c0 + 1 < CO ? __ldg(gp + (size_t)(c0 + 1) * V + va) : 0.f;
  L.g[2] = c0 < CO ? __ldg(gp + (size_t)c0 * V + va + 8) : 0.f;
  L.g[3] = c0 + 1 < CO ? __ldg(gp + (size_t)(c0 + 1) * V + va + 8) : 0.f;
}

// ------------------------------------------------------------------------------------------------
// backward kernel 1: dW / db partials of the head and the norm-backward reductions of the block in front of it.
// grid = (blocks, N), block = 256. V % 16 == 0.
//   part_w[(n * gridDim.x + b)][kC1MaxCo][33]   (column 32 = db; format of conv1x1_bwd_finish_kernel)
//   part_n[(n * gridDim.x + b)][2][32]          (S1 | S2; format of norm_bwd_finalize_kernel)
// ------------------------------------------------------------------------------------------------
template <int CO>
__global__ void __launch_bounds__(256, 2)
head_bwd_sums_mma_kernel(const float* __restrict__ dout, const __nv_bfloat16* __restrict__ y,
                         const Conv1x1Weights* __restrict__ Wg, uint32_t V, NormActArgs A, const float* __restrict__ mean,
                         const float* __restrict__ rstd, int want_w, float* __restrict__ part_w, float* __restrict__ part_n) {
  __shared__ float red_w[8][kC1MaxCo][33];
  __shared__ float red_n[8][2][32];
  const int n = blockIdx.y;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int gid = lane >> 2, tig = lane & 3;
  uint32_t bw[4];
  head_du_weights<CO>(Wg, gid, tig, bw);
  DeferredOctet K;
  K.load(A, n, 32, tig * 8);
  const float inv = K.has_drop ? 1.f / (1.f - A.drop_p) : 1.f;
  const float sinv = K.slope * inv;
  const float* gp = dout + (size_t)n * CO * V;
  const bf16x8* yp = reinterpret_cast<const bf16x8*>(y) + (size_t)n * V * 4;
  float dw[4][4];
#pragma unroll
  for (int r = 0; r < 4; ++r)
#pragma unroll
    for (int j = 0; j < 4; ++j) dw[r][j] = 0.f;
  float gbs[2] = {0.f, 0.f}, s1[8], s2[8];
#pragma unroll
  for (int k = 0; k < 8; ++k) { s1[k] = 0.f; s2[k] = 0.f; }
  const uint32_t nunits = V >> 4;
  const uint32_t ustep = gridDim.x * 8u;
  uint32_t unit = blockIdx.x * 8u + warp;                      // warp-uniform
  HeadUnitLoad L;
  if (unit < nunits) head_unit_load<CO>(L, gp, yp, V, unit * 16u + gid, tig);
  while (unit < nunits) {
    const HeadUnitLoad C = L;
    const uint32_t va = unit * 16u + gid;
    unit += ustep;
    if (unit < nunits) head_unit_load<CO>(L, gp, yp, V, unit * 16u + gid, tig);   // next unit in flight
    const uint32_t a0 = pack_bf16_pair(C.g[0], C.g[1]), a1 = pack_bf16_pair(C.g[2], C.g[3]);
    float du[4][4];
#pragma unroll
    for (int nb = 0; nb < 4; ++nb) {
      du[nb][0] = du[nb][1] = du[nb][2] = du[nb][3] = 0.f;
      mma_bf16_1688(du[nb], a0, a1, bw[nb]);
    }
    uint32_t Ua[4], Ub[4];
#pragma unroll
    for (int grp = 0; grp < 2; ++grp) {
      const bf16x8& yraw = grp ? C.yb : C.ya;
      const unsigned long long e0 = ((unsigned long long)n * V + va + 8u * grp) * 32ull + tig * 8;
      uint32_t keep[4];
      const bf16x8 a8 = K.apply(yraw, e0, nullptr, keep);
      const uint32_t* aw = reinterpret_cast<const uint32_t*>(&a8);
#pragma unroll
      for (int r = 0; r < 4; ++r) (grp ? Ub : Ua)[r] = aw[r];
      // d act / d pre-activation: the sign of the forward's own fma (the one deferred_act8 just evaluated), times the
      // dropout mask of that same evaluation (no second hash). A pre-activation of exactly 0 takes the slope branch,
      // as in every other backward pass and in kernel 2 below; the sign of the stored bf16 activation cannot tell it
      // (or a positive value below bf16's smallest subnormal) from a dropped element.
      float yy[8];
      unpack8h(yraw, yy);
#pragma unroll
      for (int k = 0; k < 8; ++k) {
        const float d_ = du[k >> 1][2 * grp + (k & 1)];
        const bool kept = (keep[k >> 1] >> (16 * (k & 1))) & 1u;
        const float fac = kept ? (fmaf(yy[k], K.sc[k], K.sh[k]) > 0.f ? inv : sinv) : 0.f;
        const float dz = d_ * fac;
        s1[k] += dz;
        s2[k] = fmaf(dz, yy[k], s2[k]);
      }
    }
    if (want_w) {
      gbs[0] += C.g[0] + C.g[2];
      gbs[1] += C.g[1] + C.g[3];
      // dW[co][ch] += sum over the unit's 16 voxels: A = g[co][voxel] (the du fragment transposed), B = u[voxel][ch]
      const uint32_t ta = movmatrix_trans(a0), tb = movmatrix_trans(a1);
#pragma unroll
      for (int r = 0; r < 4; ++r) {
        const uint32_t b0 = movmatrix_trans(Ua[r]), b1 = movmatrix_trans(Ub[r]);
        mma_bf16_16816(dw[r], ta, 0u, tb, 0u, b0, b1);
      }
    }
  }
  // ---- block reduction ----
  // S2 = sum dz * xhat = rstd * sum dz*y - mean*rstd * sum dz; then over the 8 voxel lanes (gid) of the warp
#pragma unroll
  for (int k = 0; k < 8; ++k) {
    const float r = rstd[(size_t)n * 32 + tig * 8 + k], m = mean[(size_t)n * 32 + tig * 8 + k];
    float a = s1[k], b = fmaf(r, s2[k], -m * r * s1[k]);
#pragma unroll
    for (int o = 4; o < 32; o <<= 1) {
      a += __shfl_xor_sync(0xffffffffu, a, o);
      b += __shfl_xor_sync(0xffffffffu, b, o);
    }
    if (gid == 0) { red_n[warp][0][tig * 8 + k] = a; red_n[warp][1][tig * 8 + k] = b; }
  }
  if (want_w) {
    // D fragment of dW block r: row co = gid, columns 2 tig + e <-> channel 8 tig + 2 r + e (rows 8..15 are padding)
    if (gid < CO) {
#pragma unroll
      for (int r = 0; r < 4; ++r) {
        red_w[warp][gid][8 * tig + 2 * r] = dw[r][0];
        red_w[warp][gid][8 * tig + 2 * r + 1] = dw[r][1];
      }
    }
#pragma unroll
    for (int e = 0; e < 2; ++e) {
      float a = gbs[e];
#pragma unroll
      for (int o = 4; o < 32; o <<= 1) a += __shfl_xor_sync(0xffffffffu, a, o);
      if (gid == 0 && 2 * tig + e < CO) red_w[warp][2 * tig + e][32] = a;
    }
  }
  __syncthreads();
  const size_t rec = (size_t)n * gridDim.x + blockIdx.x;
  if (threadIdx.x < 64) {
    float a = 0.f;
#pragma unroll
    for (int wq = 0; wq < 8; ++wq) a += red_n[wq][threadIdx.x >> 5][threadIdx.x & 31];
    part_n[rec * 64 + threadIdx.x] = a;
  }
  if (want_w) {
    float* pb = part_w + rec * kC1MaxCo * 33;
    for (int i = threadIdx.x; i < CO * 33; i += blockDim.x) {
      float a = 0.f;
#pragma unroll
      for (int wq = 0; wq < 8; ++wq) a += red_w[wq][i / 33][i % 33];
      pb[i] = a;
    }
  }
}

// ------------------------------------------------------------------------------------------------
// backward kernel 2: dy of the block in front of the head, straight from dout:
//   du = g^T W (recomputed), dz = du * lrelu'(y sc + sh) * keep / (1 - p), dy = ka dz + kc y + kb   (NormBwdArgs as in
//   norm_act_bwd_apply_y_kernel). grid = (blocks, N), block = 256. V % 16 == 0.
// ------------------------------------------------------------------------------------------------
template <int CO, bool DROP>
__global__ void __launch_bounds__(256, 2)
head_bwd_apply_mma_kernel(const float* __restrict__ dout, const __nv_bfloat16* __restrict__ y,
                          __nv_bfloat16* __restrict__ dy, const Conv1x1Weights* __restrict__ Wg, uint32_t V, NormBwdArgs B) {
  __shared__ __align__(16) float ks[5][32];
  const int n = blockIdx.y;
  const float finv = DROP ? 1.f / (1.f - B.drop_p) : 1.f;
  if (threadIdx.x < 32) {
    const int c = threadIdx.x;
    const size_t o = (size_t)n * 32 + c;
    const float g = B.gscale[o], r = B.rstd[o], m = B.mean[o];
    const float kc = -g * r * B.c2[o];
    ks[0][c] = g;
    ks[1][c] = -g * B.c1[o] - kc * m;
    ks[2][c] = kc;
    ks[3][c] = fold_inv(g, finv);
    ks[4][c] = fold_inv(B.fshift[o], finv);
  }
  __syncthreads();
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int gid = lane >> 2, tig = lane & 3;
  float ka[8], kb[8], kc[8], sc[8], sh[8];
#pragma unroll
  for (int k = 0; k < 8; ++k) {
    ka[k] = ks[0][tig * 8 + k]; kb[k] = ks[1][tig * 8 + k]; kc[k] = ks[2][tig * 8 + k];
    sc[k] = ks[3][tig * 8 + k]; sh[k] = ks[4][tig * 8 + k];
  }
  uint32_t bw[4];
  head_du_weights<CO>(Wg, gid, tig, bw);
  const float* gp = dout + (size_t)n * CO * V;
  const bf16x8* yp = reinterpret_cast<const bf16x8*>(y) + (size_t)n * V * 4;
  bf16x8* dyp = reinterpret_cast<bf16x8*>(dy) + (size_t)n * V * 4;
  const uint32_t nunits = V >> 4;
  const uint32_t ustep = gridDim.x * 8u;
  uint32_t unit = blockIdx.x * 8u + warp;
  HeadUnitLoad L;
  if (unit < nunits) head_unit_load<CO>(L, gp, yp, V, unit * 16u + gid, tig);
  while (unit < nunits) {
    const HeadUnitLoad C = L;
    const uint32_t va = unit * 16u + gid;
    unit += ustep;
    if (unit < nunits) head_unit_load<CO>(L, gp, yp, V, unit * 16u + gid, tig);
    const uint32_t a0 = pack_bf16_pair(C.g[0], C.g[1]), a1 = pack_bf16_pair(C.g[2], C.g[3]);
    float du[4][4];
#pragma unroll
    for (int nb = 0; nb < 4; ++nb) {
      du[nb][0] = du[nb][1] = du[nb][2] = du[nb][3] = 0.f;
      mma_bf16_1688(du[nb], a0, a1, bw[nb]);
    }
#pragma unroll
    for (int grp = 0; grp < 2; ++grp) {
      const bf16x8& yraw = grp ? C.yb : C.ya;
      const uint32_t v = va + 8u * grp;
      float f[8], yy[8], o[8];
      if (DROP) {
        dropout_factors8(((unsigned long long)n * V + v) * 32ull + tig * 8, B.drop_seed, B.drop_thresh, finv, f);
      } else {
#pragma unroll
        for (int k = 0; k < 8; ++k) f[k] = 1.f;
      }
      unpack8h(yraw, yy);
#pragma unroll
      for (int k = 0; k < 8; ++k) {
        const float d_ = du[k >> 1][2 * grp + (k & 1)];
        const float dz = d_ * (fmaf(yy[k], sc[k], sh[k]) > 0.f ? f[k] : f[k] * B.slope);
        o[k] = fmaf(ka[k], dz, fmaf(kc[k], yy[k], kb[k]));
      }
      st_stream(dyp + (size_t)v * 4 + tig, pack8(o));
    }
  }
}

}  // namespace ub
