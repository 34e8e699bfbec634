// Memory-bound kernels of the hot path (sm_100a): layout pack/unpack, norm statistics finalisation,
// fused norm-apply + dropout + LeakyReLU (+ 2x2x2 max-pool), their backward passes, max-pool
// backward, weight packing, split-K reduction of weight gradients, the L1 / BCE-with-logits losses
// and the evaluation's relative-error map + ROI reduction.
// Activations are NDHWC bf16 with the channel count padded to a multiple of 16; every kernel moves
// 16-byte vectors (8 channels) per thread and is bounded by HBM bandwidth.
#pragma once
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <stdint.h>
#include "sm100_ptx.cuh"

namespace ub {

// ------------------------------------------------------------------------------------------------
// small helpers
// ------------------------------------------------------------------------------------------------
struct alignas(16) bf16x8 {
  __nv_bfloat162 v[4];
};

// streaming 16-byte accesses (ld.global.cs / st.global.cs): every pass touches each byte once and the
// tensors are far larger than L2, so they should not displace what little is re-used
__device__ __forceinline__ bf16x8 ld_stream(const bf16x8* p) {
  const uint4 v = __ldcs(reinterpret_cast<const uint4*>(p));
  bf16x8 r;
  *reinterpret_cast<uint4*>(&r) = v;
  return r;
}
__device__ __forceinline__ void st_stream(bf16x8* p, const bf16x8& v) {
  __stcs(reinterpret_cast<uint4*>(p), *reinterpret_cast<const uint4*>(&v));
}

__device__ __forceinline__ void unpack8(const bf16x8& p, float (&f)[8]) {
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const float2 t = __bfloat1622float2(p.v[i]);
    f[2 * i] = t.x;
    f[2 * i + 1] = t.y;
  }
}
__device__ __forceinline__ bf16x8 pack8(const float (&f)[8]) {
  bf16x8 p;
#pragma unroll
  for (int i = 0; i < 4; ++i) p.v[i] = __floats2bfloat162_rn(f[2 * i], f[2 * i + 1]);
  return p;
}

// The raw conv output y of a conv -> norm block is never an MMA operand: it is stored as IEEE fp16 (11-bit
// significand instead of bf16's 8) so that the block's activations are rounded to bf16 ONCE, when they become the
// next conv's operand. Same 16-byte vectors; conversion saturates at +-65504 instead of producing inf.
__device__ __forceinline__ void unpack8h(const bf16x8& p, float (&f)[8]) {
  const __half2* h = reinterpret_cast<const __half2*>(&p);
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const float2 t = __half22float2(h[i]);
    f[2 * i] = t.x;
    f[2 * i + 1] = t.y;
  }
}

// Counter-based dropout mask (replaces torch's Philox stream, which cannot be reproduced bit-exactly;
// ref: monai ADN "D" = nn.Dropout(p), element-wise). Eight consecutive elements (one 16-byte vector)
// share one counter = the vector index; two rounds of 32x32->64-bit multiply-fold (a "mum" hash) give
// 128 bits = eight 16-bit lanes, of which 15 bits each are compared against round(p * 32768).
__device__ __forceinline__ uint32_t mulfold(uint32_t a, uint32_t b) {
  const unsigned long long m = (unsigned long long)a * b;
  return (uint32_t)m ^ (uint32_t)(m >> 32);
}
__device__ __forceinline__ void dropout_bits8(unsigned long long e0, uint32_t seed, uint32_t (&u)[4]) {
  const uint32_t idx = (uint32_t)(e0 >> 3);                     // vector index (low 32 bits)
  const uint32_t salt = seed ^ ((uint32_t)(e0 >> 35) * 0x7FEB352Du);
  const uint32_t m = mulfold(idx ^ 0x9E3779B9u, 0x85EBCA6Bu ^ (salt << 1 | 1u)) ^ salt;
  const unsigned long long p0 = (unsigned long long)(m ^ 0xC2B2AE35u) * 0x27D4EB2Fu;
  const unsigned long long p1 = (unsigned long long)(m ^ 0x165667B1u) * 0x9E3779B1u;
  const uint32_t q = mulfold(m + 0x632BE5ABu, 0xD2B74407u);
  u[0] = (uint32_t)p0 ^ q;
  u[1] = (uint32_t)(p0 >> 32) ^ (q >> 7 | q << 25);
  u[2] = (uint32_t)p1 ^ (q >> 13 | q << 19);
  u[3] = (uint32_t)(p1 >> 32) ^ (q >> 21 | q << 11);
}
// Keep decision per element: its 15-bit uniform (low 15 bits of its 16-bit lane) >= t15 = round(p * 32768).
// `thresh` carries t15 in BOTH 16-bit lanes. Lane-wise compare without unpacking: setting bit 15 of every lane
// before subtracting the threshold confines the borrow to the lane and leaves bit 15 = (u15 >= t15); PRMT's
// sign-replication mode spreads that bit over the lane. One mask word per packed bf16x2 word: 0xFFFF keeps,
// 0 drops -- applied with a single AND on the packed data (4 integer ops per 2 elements).
__device__ __forceinline__ void dropout_maskw(unsigned long long e0, uint32_t seed, uint32_t thresh, uint32_t (&mw)[4]) {
  uint32_t u[4];
  dropout_bits8(e0, seed, u);
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const uint32_t d = ((u[i] & 0x7FFF7FFFu) | 0x80008000u) - thresh;
    // prmt, generic mode: selector nibble = byte index | 8 -> replicate that byte's sign over the target byte
    // (inline PTX: __byte_perm documents only the three index bits of each nibble)
    asm("prmt.b32 %0, %1, %2, %3;" : "=r"(mw[i]) : "r"(d), "r"(0u), "r"(0xBB99u));
  }
}
__device__ __forceinline__ void apply_maskw(bf16x8& v, const uint32_t (&mw)[4]) {
  uint32_t* w = reinterpret_cast<uint32_t*>(&v);
#pragma unroll
  for (int i = 0; i < 4; ++i) w[i] &= mw[i];
}
// keep mask for the 8 consecutive elements starting at element index e0 (multiple of 8), bit i = element i
__device__ __forceinline__ uint32_t dropout_keep8(unsigned long long e0, uint32_t seed, uint32_t thresh) {
  uint32_t mw[4];
  dropout_maskw(e0, seed, thresh, mw);
  uint32_t m = 0;
#pragma unroll
  for (int i = 0; i < 4; ++i) m |= ((mw[i] & 1u) | ((mw[i] >> 15) & 2u)) << (2 * i);
  return m;
}

struct NormActArgs;
// Same mask as dropout_maskw, delivered as per-element factors f[i] = keep ? inv : 0.
__device__ __forceinline__ void dropout_factors8(unsigned long long e0, uint32_t seed, uint32_t thresh, float inv,
                                                 float (&f)[8]) {
  uint32_t mw[4];
  dropout_maskw(e0, seed, thresh, mw);
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    f[2 * i] = (mw[i] & 0xFFFFu) ? inv : 0.f;
    f[2 * i + 1] = (mw[i] >> 16) ? inv : 0.f;
  }
}
// LeakyReLU for slope <= 1 is max(x, slope * x); the general form keeps the select.
__device__ __forceinline__ float lrelu(float x, float slope, bool slope_le1) {
  const float t = x * slope;
  return slope_le1 ? fmaxf(x, t) : (x > 0.f ? x : t);
}

struct NormActArgs {
  const float* scale;   // [N][Cp]  gamma * rstd          (or nullptr: identity)
  const float* shift;   // [N][Cp]  beta - mean * scale
  float slope;          // LeakyReLU negative slope (1.0f = no activation)
  float drop_p;         // 0 = no dropout
  uint32_t drop_seed;
  uint32_t drop_thresh; // round(p * 32768) in both 16-bit lanes
};

// THE definition of a block's activations from its raw conv output (fp16 bits in `yraw`):
//   a = bf16( LeakyReLU_slope( y * (scale / (1-p)) + shift / (1-p) ) ) with dropped lanes cleared on the packed words
// -- the inverted-dropout factor 1 / (1 - p) is folded into the affine constants (sc = scale * inv, sh = shift * inv,
// both rounded once in fp32), so an element costs one fma, one multiply and one max.
// Every consumer of a deferred activation (conv operand transform, weight-gradient operand transform, max-pool
// forward / backward, the 1x1x1 output head), the materialising pass (norm_act_fwd) AND the backward passes (which
// need the sign of the same fma) use these constants and this function, so they all see bit-identical values.
// e0 = element index of the vector's first channel in the y tensor (dropout counter).
// `o16` (optional): the SAME fp32 values rounded to fp16 instead of bf16 -- the operand copy a forward conv
// multiplies with fp16-packed weights (11-bit significand: the forward pass then carries 1/8 of bf16's operand
// rounding); the bf16 form is what a weight gradient pairs with its bf16 gradients.
__device__ __forceinline__ bf16x8 deferred_act8(const bf16x8& yraw, const float (&sc)[8], const float (&sh)[8],
                                                float slope, bool slope_le1, bool has_drop, unsigned long long e0,
                                                uint32_t seed, uint32_t thresh, bf16x8* o16 = nullptr,
                                                uint32_t* keep_words = nullptr) {
  float x[8];
  unpack8h(yraw, x);
#pragma unroll
  for (int k = 0; k < 8; ++k) {
    const float hi = fmaf(x[k], sc[k], sh[k]);
    const float lo = hi * slope;
    x[k] = slope_le1 ? fmaxf(hi, lo) : (hi > 0.f ? hi : lo);
  }
  bf16x8 o = pack8(x);
  uint32_t mw[4];
  if (has_drop) {
    dropout_maskw(e0, seed, thresh, mw);
    apply_maskw(o, mw);
  }
  if (o16 != nullptr) {
    uint32_t* w16 = reinterpret_cast<uint32_t*>(o16);
#pragma unroll
    for (int k = 0; k < 4; ++k) w16[k] = pack_f16x2_sat(x[2 * k], x[2 * k + 1]);
    if (has_drop) apply_maskw(*o16, mw);
  }
  if (keep_words != nullptr) {   // the dropout mask words (0xFFFF per kept lane), for a backward that needs keep
#pragma unroll
    for (int k = 0; k < 4; ++k) keep_words[k] = has_drop ? mw[k] : 0xFFFFFFFFu;
  }
  return o;
}
// The fp16-OPERAND form of the same activations, for a conv that multiplies them as an fp16 x fp16 tensor-core
// operand (no backward pass will need them in bf16): packed half2 arithmetic straight on the fp16 y -- one HFMA2,
// one HMUL2 and one HMNMX2 per PAIR of elements, no conversions -- with the affine constants rounded to fp16.
// Relative error ~3 * 2^-12, i.e. tighter than the bf16 rounding of the canonical form.
__device__ __forceinline__ bf16x8 deferred_act8_f16(const bf16x8& yraw, const __half2 (&sc)[4], const __half2 (&sh)[4],
                                                    __half2 slope2, bool slope_le1, bool has_drop,
                                                    unsigned long long e0, uint32_t seed, uint32_t thresh) {
  bf16x8 o;
  const __half2* y2 = reinterpret_cast<const __half2*>(&yraw);
  __half2* o2 = reinterpret_cast<__half2*>(&o);
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    const __half2 hi = __hfma2(y2[k], sc[k], sh[k]);
    const __half2 lo = __hmul2(hi, slope2);
    if (slope_le1) {
      o2[k] = __hmax2(hi, lo);
    } else {
      const __half2 pos = __hgt2(hi, __float2half2_rn(0.f));     // 1.0 / 0.0 per lane
      o2[k] = __hfma2(pos, __hsub2(hi, lo), lo);
    }
  }
  if (has_drop) {
    uint32_t mw[4];
    dropout_maskw(e0, seed, thresh, mw);
    apply_maskw(o, mw);
  }
  return o;
}

// folded affine constant: the one place that defines the rounding of scale * inv / shift * inv
__device__ __forceinline__ float fold_inv(float v, float inv) { return v * inv; }
// per-thread constants of a deferred activation for the channel octet starting at c0 of sample n
struct DeferredOctet {
  float sc[8], sh[8];
  float slope;
  bool slope_le1, has_drop;
  uint32_t seed, thresh;
  __device__ __forceinline__ void load(const NormActArgs& A, int n, int Cp, int c0) {
    const bool has_norm = A.scale != nullptr;
    has_drop = A.drop_p > 0.f;
    const float inv = has_drop ? 1.f / (1.f - A.drop_p) : 1.f;
#pragma unroll
    for (int k = 0; k < 8; ++k) {
      sc[k] = fold_inv(has_norm ? __ldg(A.scale + (size_t)n * Cp + c0 + k) : 1.f, inv);
      sh[k] = fold_inv(has_norm ? __ldg(A.shift + (size_t)n * Cp + c0 + k) : 0.f, inv);
    }
    slope = A.slope;
    slope_le1 = A.slope <= 1.f;
    seed = A.drop_seed;
    thresh = A.drop_thresh;
  }
  __device__ __forceinline__ bf16x8 apply(const bf16x8& yraw, unsigned long long e0, bf16x8* o16 = nullptr,
                                          uint32_t* keep_words = nullptr) const {
    return deferred_act8(yraw, sc, sh, slope, slope_le1, has_drop, e0, seed, thresh, o16, keep_words);
  }
};

// ------------------------------------------------------------------------------------------------
// layout: NCDHW fp32 <-> NDHWC bf16 (channel padded)
// ------------------------------------------------------------------------------------------------
// thread = (voxel, channel octet): a warp covers 8 (CP = 32) or 4 (CP = 64) consecutive voxels x all
// octets, so every load instruction reads whole 32-byte sectors of the channel planes and every store
// instruction writes one contiguous run of CP*2-byte voxel rows (no partial sectors on either side).
// Two optional inputs a (ca channels) and b (cb channels) are concatenated: this is the torch.cat of
// the PatchGAN input (ref: model.py:86) folded into the layout change.
// S2D: the destination is the parity-planar space-to-depth layout [N][(pd,ph,pw)][D/2][H/2][W/2][CP]
// (eight dense half-resolution sub-volumes per sample) that the stride-2 PatchGAN stem reads with
// plain, unstrided TMA boxes whose rows are contiguous in memory.
// a_bf16: input a is NCDHW bf16 instead of fp32 (a host pipeline that ships the network input in bf16 halves the
// host-to-device bytes; the packed result is bit-identical, since fp32 inputs are rounded to bf16 here anyway).
template <int CP, bool S2D, int UNROLL, bool A16>
__global__ void __launch_bounds__(256)
pack_ncdhw_kernel(const void* __restrict__ a_raw, int ca, const float* __restrict__ b, int cb,
                  __nv_bfloat16* __restrict__ dst, long long V, int D, int H, int W) {
  constexpr int OCT = CP / 8;            // octets per voxel
  constexpr int VPB = 256 / OCT;         // voxels per block pass
  const int n = blockIdx.y;
  const int oct = threadIdx.x % OCT;
  const long long v0 = (long long)blockIdx.x * (VPB * UNROLL) + threadIdx.x / OCT;
  // source plane of channel k: a (fp32, or bf16 when A16) for c < ca, b (fp32) for ca <= c < ca + cb, else nullptr.
  // With A16 the planes of a are addressed in 2-byte elements; `from_a` tells the two apart.
  const void* src[8];
  bool from_a[8];
#pragma unroll
  for (int k = 0; k < 8; ++k) {
    const int c = oct * 8 + k;
    const size_t off_a = ((size_t)n * ca + c) * V;
    from_a[k] = c < ca;
    if (c < ca) src[k] = A16 ? (const void*)(reinterpret_cast<const __nv_bfloat16*>(a_raw) + off_a)
                             : (const void*)(reinterpret_cast<const float*>(a_raw) + off_a);
    else src[k] = c < ca + cb ? (const void*)(b + ((size_t)n * cb + (c - ca)) * V) : nullptr;
  }
  float g[UNROLL][8];
#pragma unroll
  for (int u = 0; u < UNROLL; ++u) {
    const long long v = v0 + (long long)u * VPB;
#pragma unroll
    for (int k = 0; k < 8; ++k) {
      float val = 0.f;
      if (src[k] != nullptr && v < V) {
        if (A16 && from_a[k]) val = __bfloat162float(__ldg(reinterpret_cast<const __nv_bfloat16*>(src[k]) + v));
        else val = __ldg(reinterpret_cast<const float*>(src[k]) + v);
      }
      g[u][k] = val;
    }
  }
#pragma unroll
  for (int u = 0; u < UNROLL; ++u) {
    const long long v = v0 + (long long)u * VPB;
    if (v >= V) continue;
    size_t row;
    if (S2D) {
      // 32-bit index math (the host checks voxels per sample < 2^31): 64-bit divisions by run-time values cost
      // ~100 instructions each and made the space-to-depth pack 25 % slower than the plain one
      const uint32_t v32 = (uint32_t)v;
      const int w = (int)(v32 % (uint32_t)W);
      const uint32_t t = v32 / (uint32_t)W;
      const int h = (int)(t % (uint32_t)H), d = (int)(t / (uint32_t)H);
      const size_t par = (size_t)n * 8 + ((d & 1) * 4 + (h & 1) * 2 + (w & 1));
      row = ((par * (D >> 1) + (d >> 1)) * (H >> 1) + (h >> 1)) * (W >> 1) + (w >> 1);
    } else {
      row = (size_t)n * V + v;
    }
    st_stream(reinterpret_cast<bf16x8*>(dst + row * CP) + oct, pack8(g[u]));
  }
}

// The same pack for a bf16 input `a` (NCDHW bf16: the transport format of the conditioning input), two voxels per
// thread: a 4-byte load per channel plane covers the voxel pair (v, v + 1), so a warp reads whole 32-byte sectors
// like the fp32 kernel does (one bf16 per lane would touch twice the sectors per byte). V (and for S2D: W) even.
template <int CP, bool S2D, int UNROLL>
__global__ void __launch_bounds__(256)
pack_ncdhw_a16_kernel(const __nv_bfloat16* __restrict__ a, int ca, const float* __restrict__ b, int cb,
                      __nv_bfloat16* __restrict__ dst, long long V, int D, int H, int W) {
  constexpr int OCT = CP / 8;
  constexpr int PPB = 256 / OCT;         // voxel pairs per block pass
  const int n = blockIdx.y;
  const int oct = threadIdx.x % OCT;
  const long long p0 = (long long)blockIdx.x * (PPB * UNROLL) + threadIdx.x / OCT;
  const __nv_bfloat16* sa[8];
  const float* sb[8];
#pragma unroll
  for (int k = 0; k < 8; ++k) {
    const int c = oct * 8 + k;
    sa[k] = c < ca ? a + ((size_t)n * ca + c) * V : nullptr;
    sb[k] = (c >= ca && c < ca + cb) ? b + ((size_t)n * cb + (c - ca)) * V : nullptr;
  }
  uint32_t gq[UNROLL][8], gr[UNROLL][8];     // raw loaded words; converted after ALL loads are in flight
  bool isa[8];
#pragma unroll
  for (int k = 0; k < 8; ++k) isa[k] = sa[k] != nullptr;
#pragma unroll
  for (int u = 0; u < UNROLL; ++u) {
    const long long v = 2 * (p0 + (long long)u * PPB);
#pragma unroll
    for (int k = 0; k < 8; ++k) {
      // two PREDICATED loads and a select, no branches: with nested ifs every load sat in its own basic block and a
      // thread had one load in flight at a time (2.25 ms against 0.41 ms for the fp32 kernel on the same batch)
      // Both sources land in the SAME two registers (disjoint predicates): a separate 8-byte destination for the
      // fp32 source doubled the registers held by loads in flight, and the compiler then funnelled the bf16 loads
      // through one register, i.e. serialised them (1.7 ms).
      const bool ina = sa[k] != nullptr && v < V, inb = sb[k] != nullptr && v < V;
      uint32_t r0 = 0u, r1 = 0u;
      if (ina) r0 = __ldg(reinterpret_cast<const uint32_t*>(sa[k] + v));
      if (inb) {
        r0 = __ldg(reinterpret_cast<const uint32_t*>(sb[k] + v));
        r1 = __ldg(reinterpret_cast<const uint32_t*>(sb[k] + v + 1));
      }
      gq[u][k] = r0; gr[u][k] = r1;
    }
  }
#pragma unroll
  for (int u = 0; u < UNROLL; ++u) {
    const long long v = 2 * (p0 + (long long)u * PPB);
    if (v >= V) continue;
    size_t row0, row1;
    if (S2D) {
      const uint32_t v32 = (uint32_t)v;    // 32-bit index math, see pack_ncdhw_kernel
      const int w = (int)(v32 % (uint32_t)W);          // even
      const uint32_t t = v32 / (uint32_t)W;
      const int h = (int)(t % (uint32_t)H), d = (int)(t / (uint32_t)H);
      const size_t par = (size_t)n * 8 + ((d & 1) * 4 + (h & 1) * 2);
      const size_t inner = ((size_t)(d >> 1) * (H >> 1) + (h >> 1)) * (W >> 1) + (w >> 1);
      const size_t sub = (size_t)(D >> 1) * (H >> 1) * (W >> 1);
      row0 = par * sub + inner;            // parity (.., .., 0)
      row1 = (par + 1) * sub + inner;      // parity (.., .., 1): the odd neighbour lands at the same sub-volume offset
    } else {
      row0 = (size_t)n * V + v;
      row1 = row0 + 1;
    }
    float g0[8], g1[8];
#pragma unroll
    for (int k = 0; k < 8; ++k) {
      g0[k] = __uint_as_float(isa[k] ? gq[u][k] << 16 : gq[u][k]);
      g1[k] = __uint_as_float(isa[k] ? gq[u][k] & 0xFFFF0000u : gr[u][k]);
    }
    st_stream(reinterpret_cast<bf16x8*>(dst + row0 * CP) + oct, pack8(g0));
    st_stream(reinterpret_cast<bf16x8*>(dst + row1 * CP) + oct, pack8(g1));
  }
}

// NDHWC bf16 -> the parity-planar space-to-depth layout [N][(pd,ph,pw)][D/2][H/2][W/2][Cp] of the same tensor (a
// permuting copy): what a stride-2 4x4x4 conv reads with plain, unstrided TMA boxes (UB_CONV_K4S2P1_S2D). The
// PatchGAN body d2 .. d5 (ref: model.py:74-82) converts its input this way instead of loading 8 parity tiles with
// element stride 2 (6.4 x L2 -> SM over-fetch on d2); the copy of a layer input costs a few tens of microseconds.
// thread = (destination voxel, channel octet): whole 16-byte vectors on both sides. grid = (blocks, N).
__global__ void __launch_bounds__(256)
to_s2d_kernel(const __nv_bfloat16* __restrict__ src, __nv_bfloat16* __restrict__ dst, int Cp, int D, int H, int W,
              uint32_t per_sample /* voxels * Cp/8 of one sample */) {
  const uint32_t j = blockIdx.x * 256u + threadIdx.x;
  if (j >= per_sample) return;
  const int n = blockIdx.y;
  const uint32_t c8 = (uint32_t)Cp >> 3;
  uint32_t r = j / c8;                      // destination row inside the sample: ((par * D2 + d2) * H2 + h2) * W2 + w2
  const uint32_t oct = j - r * c8;
  const uint32_t W2 = W >> 1, H2 = H >> 1, D2 = D >> 1;
  const uint32_t w2 = r % W2; r /= W2;
  const uint32_t h2 = r % H2; r /= H2;
  const uint32_t d2 = r % D2;
  const uint32_t par = r / D2;
  const uint32_t d = 2 * d2 + (par >> 2), h = 2 * h2 + ((par >> 1) & 1), w = 2 * w2 + (par & 1);
  const size_t srow = (((size_t)n * D + d) * H + h) * W + w;
  const bf16x8 v = ld_stream(reinterpret_cast<const bf16x8*>(src) + srow * c8 + oct);
  st_stream(reinterpret_cast<bf16x8*>(dst) + (size_t)n * per_sample + j, v);
}

// Patch gather (sliding-window inference): sample n of the output batch is the d x h x w sub-volume of an
// NCDHW fp32 tensor that starts at element offset G.offset[n]; element (c, z, y, x) of it lives at
// + c * stride_c + z * stride_d + y * stride_h + x. Replaces torchio's GridSampler patch extraction
// (ref: data_module.py:168-183, model.py:315-321) with index arithmetic inside the layout pack.
constexpr int kMaxPatchBatch = 64;
struct PatchGeom {
  long long offset[kMaxPatchBatch];
  long long stride_c, stride_d, stride_h;
  int d, h, w;
};
template <int CP, int UNROLL>
__global__ void __launch_bounds__(256)
pack_patches_kernel(const float* __restrict__ a, int ca, __nv_bfloat16* __restrict__ dst, PatchGeom G) {
  constexpr int OCT = CP / 8;
  constexpr int VPB = 256 / OCT;
  const int n = blockIdx.y;
  const int oct = threadIdx.x % OCT;
  const uint32_t V = (uint32_t)G.d * G.h * G.w;
  const uint32_t v0 = blockIdx.x * (VPB * UNROLL) + threadIdx.x / OCT;
  const float* base = a + G.offset[n];
  float g[UNROLL][8];
#pragma unroll
  for (int u = 0; u < UNROLL; ++u) {
    const uint32_t v = v0 + u * VPB;
    const uint32_t x = v % G.w, t = v / G.w;
    const uint32_t y = t % G.h, z = t / G.h;
    const float* p = base + (size_t)z * G.stride_d + (size_t)y * G.stride_h + x;
#pragma unroll
    for (int k = 0; k < 8; ++k) {
      const int c = oct * 8 + k;
      g[u][k] = (c < ca && v < V) ? __ldg(p + (size_t)c * G.stride_c) : 0.f;
    }
  }
#pragma unroll
  for (int u = 0; u < UNROLL; ++u) {
    const uint32_t v = v0 + u * VPB;
    if (v >= V) continue;
    reinterpret_cast<bf16x8*>(dst + ((size_t)n * V + v) * CP)[oct] = pack8(g[u]);
  }
}

// Patch scatter: channels [c_begin, c_begin + c) of sample `sample` of an NDHWC bf16 batch -> a d x h x w
// region of an NCDHW fp32 volume (same addressing as PatchGeom, one region: offset[0]). Later patches
// overwrite earlier ones when launched in sampler order: torchio GridAggregator.add_batch with
// overlap 0 (ref: model.py:322).
__global__ void unpack_patch_kernel(const __nv_bfloat16* __restrict__ src, float* __restrict__ dst, int cp, int c_begin,
                                    int c, int sample, PatchGeom G) {
  const uint32_t V = (uint32_t)G.d * G.h * G.w;
  const uint32_t v = blockIdx.x * blockDim.x + threadIdx.x;
  if (v >= V) return;
  const uint32_t x = v % G.w, t = v / G.w;
  const uint32_t y = t % G.h, z = t / G.h;
  const __nv_bfloat16* s = src + ((size_t)sample * V + v) * cp + c_begin;
  float* d = dst + G.offset[0] + (size_t)z * G.stride_d + (size_t)y * G.stride_h + x;
  for (int k = 0; k < c; ++k) d[(size_t)k * G.stride_c] = __bfloat162float(s[k]);
}

// Same for an NCDHW fp32 patch (c, d, h, w contiguous), e.g. the output of the fused generator head.
__global__ void paste_patch_kernel(const float* __restrict__ src, float* __restrict__ dst, int c, PatchGeom G) {
  const uint32_t V = (uint32_t)G.d * G.h * G.w;
  const uint32_t v = blockIdx.x * blockDim.x + threadIdx.x;
  if (v >= V) return;
  const uint32_t x = v % G.w, t = v / G.w;
  const uint32_t y = t % G.h, z = t / G.h;
  float* d = dst + G.offset[0] + (size_t)z * G.stride_d + (size_t)y * G.stride_h + x;
  for (int k = 0; k < c; ++k) d[(size_t)k * G.stride_c] = __ldcs(src + (size_t)k * V + v);
}

// Overlapping sliding-window aggregation (torchio 0.19.6 GridAggregator.add_batch): up to kMaxPatchBatch NCDHW fp32
// patches [n][c][pd][ph][pw], in sampler order, into an NCDHW fp32 volume. One thread per voxel of the batch's
// bounding box (x fastest) tests the patches' boxes in order:
//   kBlendCrop     the last patch whose box (its crop box) holds the voxel is assigned: "the later patch wins";
//   kBlendAverage  out += p and weight += 1 for every covering patch;
//   kBlendHann     w = (wz * wy) * wx from the window vectors, out += p * w and weight += w.
// The accumulating modes keep the voxel's numerator and weight in registers across the batch and load / store them
// once, so each voxel sees its additions in sampler order, across launches too. __fmul_rn / __fadd_rn keep nvcc
// from contracting num + p * w into an FMA: the sums are the ones torch computes, bit for bit.
enum BlendMode { kBlendCrop = 0, kBlendAverage = 1, kBlendHann = 2 };
constexpr int kMaxBlendChannels = 8;
struct BlendGeom {
  int org[kMaxPatchBatch][3];             // patch origin (z, y, x) in the volume
  int box[kMaxPatchBatch][6];             // volume region the patch writes: z0, y0, x0, z1, y1, x1 (half-open)
  int n, c, pd, ph, pw;
  int b0[3], bh, bw;                      // bounding box of the batch's boxes: origin and its two inner extents
  int H, W;                               // volume [c][D][H][W] and weight [D][H][W], both contiguous
  long long V;                            // D * H * W
};
template <int MODE>
__global__ void __launch_bounds__(256)
blend_patches_kernel(const float* __restrict__ src, float* __restrict__ out, float* __restrict__ weight,
                     const float* __restrict__ window /* wz[pd], wy[ph], wx[pw] */, const __grid_constant__ BlendGeom G,
                     uint32_t voxels) {
  const uint32_t v = blockIdx.x * 256u + threadIdx.x;
  if (v >= voxels) return;
  const uint32_t t = v / (uint32_t)G.bw;
  const int x = G.b0[2] + (int)(v - t * (uint32_t)G.bw);
  const int y = G.b0[1] + (int)(t % (uint32_t)G.bh);
  const int z = G.b0[0] + (int)(t / (uint32_t)G.bh);
  const size_t PV = (size_t)G.pd * G.ph * G.pw;
  const size_t vox = ((size_t)z * G.H + y) * G.W + x;
  float* o = out + vox;
  auto local = [&](int j) {                // element (0, lz, ly, lx) of patch j
    return ((size_t)j * G.c * G.pd + (z - G.org[j][0])) * G.ph * G.pw + (size_t)(y - G.org[j][1]) * G.pw + (x - G.org[j][2]);
  };
  auto covers = [&](int j) {
    return z >= G.box[j][0] && y >= G.box[j][1] && x >= G.box[j][2] && z < G.box[j][3] && y < G.box[j][4] && x < G.box[j][5];
  };
  if (MODE == kBlendCrop) {
    int last = -1;
    for (int j = 0; j < G.n; ++j)
      if (covers(j)) last = j;
    if (last < 0) return;
    const float* s = src + local(last);
    for (int k = 0; k < G.c; ++k) o[(size_t)k * G.V] = __ldcs(s + (size_t)k * PV);
    return;
  }
  float num[kMaxBlendChannels];
  float den = 0.f;
  bool any = false;
  for (int j = 0; j < G.n; ++j) {
    if (!covers(j)) continue;
    if (!any) {
      any = true;
      den = weight[vox];
#pragma unroll
      for (int k = 0; k < kMaxBlendChannels; ++k)
        if (k < G.c) num[k] = o[(size_t)k * G.V];
    }
    const float* s = src + local(j);
    float w = 1.f;
    if (MODE == kBlendHann)
      w = __fmul_rn(__fmul_rn(window[z - G.org[j][0]], window[G.pd + (y - G.org[j][1])]),
                    window[G.pd + G.ph + (x - G.org[j][2])]);
#pragma unroll
    for (int k = 0; k < kMaxBlendChannels; ++k) {
      if (k >= G.c) break;
      const float p = __ldcs(s + (size_t)k * PV);
      num[k] = __fadd_rn(num[k], MODE == kBlendHann ? __fmul_rn(p, w) : p);
    }
    den = __fadd_rn(den, w);
  }
  if (!any) return;
  weight[vox] = den;
#pragma unroll
  for (int k = 0; k < kMaxBlendChannels; ++k)
    if (k < G.c) o[(size_t)k * G.V] = num[k];
}

// out / weight after the last batch of an accumulating blend: the true_divide of GridAggregator.get_output_tensor.
__global__ void __launch_bounds__(256)
blend_finish_kernel(float* __restrict__ out, const float* __restrict__ weight, int c, uint32_t voxels) {
  const uint32_t v = blockIdx.x * 256u + threadIdx.x;
  if (v >= voxels) return;
  const float w = weight[v];
  for (int k = 0; k < c; ++k) out[(size_t)k * voxels + v] = __fdiv_rn(out[(size_t)k * voxels + v], w);
}

// channels [c_begin, c_begin + c) of an NDHWC bf16 tensor -> NCDHW fp32
__global__ void unpack_ncdhw_kernel(const __nv_bfloat16* __restrict__ src, float* __restrict__ dst, int cp,
                                    int c_begin, int c, long long V, long long total) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total) return;
  const long long n = i / V, v = i - n * V;
  const __nv_bfloat16* s = src + (size_t)i * cp + c_begin;
  float* d = dst + (size_t)n * c * V + v;
  for (int k = 0; k < c; ++k) d[(size_t)k * V] = __bfloat162float(s[k]);
}

// ------------------------------------------------------------------------------------------------
// statistics: reduce the conv epilogue's per-tile partials to scale / shift (and saved mean, rstd)
// ------------------------------------------------------------------------------------------------
// mode 0: InstanceNorm (per sample, per channel; biased variance)       ref: monai ADN "N"
// mode 1: BatchNorm, training (per channel over N and voxels; updates running stats with
//         momentum and the unbiased variance)                           ref: model.py:53-54
// mode 2: BatchNorm, eval (running statistics; partials unused)
// grid = (Cp/32, N) for InstanceNorm, (Cp/32, 1) for the BatchNorm modes (one reduction over all
// samples, results broadcast to every n); block = (32, 32)
__global__ void stats_finalize_kernel(const float* __restrict__ partial, int tiles_per_sample, int Nb, int Cp, int C,
                                      double count_per_sample, const float* __restrict__ gamma,
                                      const float* __restrict__ beta, float eps, int mode, float momentum,
                                      float* __restrict__ running_mean, float* __restrict__ running_var,
                                      float* __restrict__ scale, float* __restrict__ shift,
                                      float* __restrict__ mean_out, float* __restrict__ rstd_out) {
  __shared__ double sh_s[32][32], sh_q[32][32];
  const int c = blockIdx.x * 32 + threadIdx.x;
  const int n = blockIdx.y;
  double s = 0.0, q = 0.0;
  if (mode != 2) {
    const int t0 = mode == 0 ? n * tiles_per_sample : 0;
    const int t1 = mode == 0 ? t0 + tiles_per_sample : Nb * tiles_per_sample;
    // four independent accumulation chains per thread keep enough loads in flight
    float fs[4] = {0.f, 0.f, 0.f, 0.f}, fq[4] = {0.f, 0.f, 0.f, 0.f};
    int t = t0 + threadIdx.y;
    for (; t + 96 < t1; t += 128) {
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        fs[u] = partial[((size_t)(t + 32 * u) * 2 + 0) * Cp + c];
        fq[u] = partial[((size_t)(t + 32 * u) * 2 + 1) * Cp + c];
      }
      s += ((double)fs[0] + (double)fs[1]) + ((double)fs[2] + (double)fs[3]);
      q += ((double)fq[0] + (double)fq[1]) + ((double)fq[2] + (double)fq[3]);
    }
    for (; t < t1; t += 32) {
      s += (double)partial[((size_t)t * 2 + 0) * Cp + c];
      q += (double)partial[((size_t)t * 2 + 1) * Cp + c];
    }
  }
  sh_s[threadIdx.y][threadIdx.x] = s;
  sh_q[threadIdx.y][threadIdx.x] = q;
  __syncthreads();
  if (threadIdx.y != 0) return;
  for (int k = 1; k < 32; ++k) { s += sh_s[k][threadIdx.x]; q += sh_q[k][threadIdx.x]; }
  double mean, var;
  if (mode == 2) {
    mean = c < C ? (double)running_mean[c] : 0.0;
    var = c < C ? (double)running_var[c] : 1.0;
  } else {
    const double cnt = mode == 0 ? count_per_sample : count_per_sample * Nb;
    mean = s / cnt;
    var = q / cnt - mean * mean;
    if (var < 0.0) var = 0.0;
    if (mode == 1 && n == 0 && c < C && running_mean != nullptr) {
      const double unbiased = cnt > 1.0 ? var * cnt / (cnt - 1.0) : var;
      running_mean[c] = (float)((1.0 - momentum) * running_mean[c] + momentum * mean);
      running_var[c] = (float)((1.0 - momentum) * running_var[c] + momentum * unbiased);
    }
  }
  const double rstd = 1.0 / sqrt(var + (double)eps);
  const float g = c < C ? gamma[c] : 0.f, b = c < C ? beta[c] : 0.f;
  const int n_lo = mode == 0 ? n : 0, n_hi = mode == 0 ? n + 1 : Nb;
  for (int nn = n_lo; nn < n_hi; ++nn) {
    const size_t o = (size_t)nn * Cp + c;
    scale[o] = (float)(g * rstd);
    shift[o] = (float)(b - mean * g * rstd);
    mean_out[o] = (float)mean;
    rstd_out[o] = (float)rstd;
  }
}

// BatchNorm (training) statistics over MANY tile partials (the full-resolution input head: 32 768 records) in two
// stages, so the reduction is not one thread block reading 8 MB. Stage 1, grid = (Cp/32, N), block = (32, 32): the
// fp64 sums of sample n go, as raw bits, into the four per-(n, c) output slots (scale | shift hold sum, mean | rstd
// hold sumsq) -- scratch that stage 2 overwrites. Stage 2, grid = (Cp/32), block = 32: channel c adds its N pairs in
// order and writes the final values to every row.
__global__ void bn_stats_stage1_kernel(const float* __restrict__ partial, int tiles_per_sample, int Cp,
                                       float* __restrict__ scale, float* __restrict__ shift,
                                       float* __restrict__ mean_out, float* __restrict__ rstd_out) {
  __shared__ double sh_s[32][32], sh_q[32][32];
  const int c = blockIdx.x * 32 + threadIdx.x;
  const int n = blockIdx.y;
  const int t0 = n * tiles_per_sample, t1 = t0 + tiles_per_sample;
  double s = 0.0, q = 0.0;
  float fs[4], fq[4];
  int t = t0 + threadIdx.y;
  for (; t + 96 < t1; t += 128) {
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      fs[u] = partial[((size_t)(t + 32 * u) * 2 + 0) * Cp + c];
      fq[u] = partial[((size_t)(t + 32 * u) * 2 + 1) * Cp + c];
    }
    s += ((double)fs[0] + (double)fs[1]) + ((double)fs[2] + (double)fs[3]);
    q += ((double)fq[0] + (double)fq[1]) + ((double)fq[2] + (double)fq[3]);
  }
  for (; t < t1; t += 32) {
    s += (double)partial[((size_t)t * 2 + 0) * Cp + c];
    q += (double)partial[((size_t)t * 2 + 1) * Cp + c];
  }
  sh_s[threadIdx.y][threadIdx.x] = s;
  sh_q[threadIdx.y][threadIdx.x] = q;
  __syncthreads();
  if (threadIdx.y != 0) return;
  for (int k = 1; k < 32; ++k) { s += sh_s[k][threadIdx.x]; q += sh_q[k][threadIdx.x]; }
  const size_t o = (size_t)n * Cp + c;
  const unsigned long long sb = (unsigned long long)__double_as_longlong(s), qb = (unsigned long long)__double_as_longlong(q);
  scale[o] = __uint_as_float((uint32_t)sb); shift[o] = __uint_as_float((uint32_t)(sb >> 32));
  mean_out[o] = __uint_as_float((uint32_t)qb); rstd_out[o] = __uint_as_float((uint32_t)(qb >> 32));
}
__global__ void bn_stats_stage2_kernel(int Nb, int Cp, int C, double count_per_sample, const float* __restrict__ gamma,
                                       const float* __restrict__ beta, float eps, float momentum,
                                       float* __restrict__ running_mean, float* __restrict__ running_var,
                                       float* __restrict__ scale, float* __restrict__ shift,
                                       float* __restrict__ mean_out, float* __restrict__ rstd_out) {
  const int c = blockIdx.x * 32 + threadIdx.x;
  double s = 0.0, q = 0.0;
  for (int n = 0; n < Nb; ++n) {
    const size_t o = (size_t)n * Cp + c;
    const unsigned long long sb = (unsigned long long)__float_as_uint(scale[o]) | ((unsigned long long)__float_as_uint(shift[o]) << 32);
    const unsigned long long qb = (unsigned long long)__float_as_uint(mean_out[o]) | ((unsigned long long)__float_as_uint(rstd_out[o]) << 32);
    s += __longlong_as_double((long long)sb);
    q += __longlong_as_double((long long)qb);
  }
  const double cnt = count_per_sample * Nb;
  const double mean = s / cnt;
  double var = q / cnt - mean * mean;
  if (var < 0.0) var = 0.0;
  if (c < C && running_mean != nullptr) {
    const double unbiased = cnt > 1.0 ? var * cnt / (cnt - 1.0) : var;
    running_mean[c] = (float)((1.0 - momentum) * running_mean[c] + momentum * mean);
    running_var[c] = (float)((1.0 - momentum) * running_var[c] + momentum * unbiased);
  }
  const double rstd = 1.0 / sqrt(var + (double)eps);
  const float g = c < C ? gamma[c] : 0.f, b = c < C ? beta[c] : 0.f;
  for (int n = 0; n < Nb; ++n) {
    const size_t o = (size_t)n * Cp + c;
    scale[o] = (float)(g * rstd);
    shift[o] = (float)(b - mean * g * rstd);
    mean_out[o] = (float)mean;
    rstd_out[o] = (float)rstd;
  }
}

// ------------------------------------------------------------------------------------------------
// forward: a = LeakyReLU(Dropout(y * scale + shift)); optional fused MaxPool3d(2)
// ------------------------------------------------------------------------------------------------
// grid = (ceil(vps / (256 * UNROLL)), N), vps = vectors (8 channels) per sample. FIXED: Cp/8 divides
// 256, so a thread keeps the same channel octet for all its vectors and the per-channel scale / shift
// live in registers. No 64-bit divisions on the path.
// a (bf16) and / or a16 (the fp16 operand copy of the same values) are written; either may be nullptr.
template <int UNROLL, bool FIXED>
__global__ void __launch_bounds__(256)
norm_act_fwd_kernel(const __nv_bfloat16* __restrict__ y /* fp16 bits */, __nv_bfloat16* __restrict__ a,
                    __nv_bfloat16* __restrict__ a16 /* fp16 bits */, NormActArgs A, int Cp, uint32_t vps) {
  const int n = blockIdx.y;
  const uint32_t c8 = (uint32_t)Cp >> 3;
  const size_t base = (size_t)n * vps;
  const bf16x8* yv = reinterpret_cast<const bf16x8*>(y) + base;
  bf16x8* av = reinterpret_cast<bf16x8*>(a) + base;
  bf16x8* av16 = reinterpret_cast<bf16x8*>(a16) + base;
  const uint32_t i0 = blockIdx.x * (256u * UNROLL) + threadIdx.x;
  DeferredOctet K;
  if (FIXED) K.load(A, n, Cp, (int)(threadIdx.x % c8) * 8);
  bf16x8 in[UNROLL];
#pragma unroll
  for (int u = 0; u < UNROLL; ++u) {
    const uint32_t idx = i0 + u * 256u;
    if (idx < vps) in[u] = ld_stream(yv + idx);
  }
#pragma unroll
  for (int u = 0; u < UNROLL; ++u) {
    const uint32_t idx = i0 + u * 256u;
    if (idx >= vps) continue;
    if (!FIXED) K.load(A, n, Cp, (int)(idx % c8) * 8);
    bf16x8 h;
    const bf16x8 o = K.apply(in[u], (unsigned long long)(base + idx) * 8ull, a16 != nullptr ? &h : nullptr);
    if (a != nullptr) st_stream(av + idx, o);
    if (a16 != nullptr) st_stream(av16 + idx, h);
  }
}

// thread = (pooled voxel, 8 channels): writes the 8 activated voxels (unless a == nullptr: the activations stay
// deferred and only the pooled tensor is materialised) and their max
__global__ void norm_act_pool_fwd_kernel(const __nv_bfloat16* __restrict__ y /* fp16 bits */, __nv_bfloat16* __restrict__ a,
                                         __nv_bfloat16* __restrict__ a16 /* fp16 bits, may be nullptr */,
                                         __nv_bfloat16* __restrict__ pooled, NormActArgs A, int Cp, int Nb, int D,
                                         int H, int W, uint32_t per_sample /* pooled voxels * Cp/8 of one sample */) {
  // grid = (blocks, N): 32-bit index math inside a sample
  const uint32_t j0 = blockIdx.x * blockDim.x + threadIdx.x;
  if (j0 >= per_sample) return;
  const int n = blockIdx.y;
  const long long i = (long long)n * per_sample + j0;
  const uint32_t c8 = (uint32_t)Cp >> 3;
  uint32_t pv = j0 / c8;
  const int c0 = (int)(j0 - pv * c8) * 8;
  const uint32_t Wp = W >> 1, Hp = H >> 1;
  const int wx = (int)(pv % Wp); pv /= Wp;
  const int hy = (int)(pv % Hp);
  const int dz = (int)(pv / Hp);
  DeferredOctet K;
  K.load(A, n, Cp, c0);
  float m[8];
#pragma unroll
  for (int k = 0; k < 8; ++k) m[k] = -INFINITY;
  bf16x8 raw[8];
  size_t e[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    const int d = 2 * dz + (j >> 2), h = 2 * hy + ((j >> 1) & 1), w = 2 * wx + (j & 1);
    const size_t vox = (((size_t)n * D + d) * H + h) * W + w;
    e[j] = vox * c8 + (c0 >> 3);
    raw[j] = ld_stream(reinterpret_cast<const bf16x8*>(y) + e[j]);
  }
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    bf16x8 h;
    const bf16x8 pk = K.apply(raw[j], (unsigned long long)e[j] * 8ull, a16 != nullptr ? &h : nullptr);
    if (a != nullptr) st_stream(reinterpret_cast<bf16x8*>(a) + e[j], pk);
    if (a16 != nullptr) st_stream(reinterpret_cast<bf16x8*>(a16) + e[j], h);
    float xr[8];
    unpack8(pk, xr);  // max over the stored (rounded) values
#pragma unroll
    for (int k = 0; k < 8; ++k) m[k] = xr[k] > m[k] ? xr[k] : m[k];
  }
  st_stream(reinterpret_cast<bf16x8*>(pooled) + i, pack8(m));
}

// ------------------------------------------------------------------------------------------------
// backward of (norm -> dropout -> LeakyReLU)
//   dz1 = dA * lrelu'(a) * keep / (1-p)          (sign(a) == sign of the pre-activation, slope > 0)
//   reduce: S1[n,c] = sum dz1, S2[n,c] = sum dz1 * xhat,   xhat = (y - mean) * rstd
//   apply : dy = g*rstd * (dz1 - c1 - xhat * c2),  c1 = S1/cnt, c2 = S2/cnt   (c1 = c2 = 0 in eval-BN / no-norm)
// ------------------------------------------------------------------------------------------------
struct NormBwdArgs {
  const float* mean;    // [N][Cp] (nullptr: no norm)
  const float* rstd;    // [N][Cp]
  const float* gscale;  // [N][Cp] gamma * rstd
  const float* c1;      // [N][Cp]
  const float* c2;      // [N][Cp]
  const float* fshift;  // [N][Cp] forward shift (beta - mean * gscale); non-null: the LeakyReLU branch is taken
                        // from sign(y * gscale + fshift) -- the forward's own fma -- and `a` is not read
  float slope, drop_p;
  uint32_t drop_seed, drop_thresh;
};

__device__ __forceinline__ void dz1_8(const bf16x8& da8, const bf16x8& a8, const NormBwdArgs& B,
                                      unsigned long long e0, float (&dz)[8]) {
  float da[8], av[8];
  bf16x8 dm = da8;
  float inv = 1.f;
  if (B.drop_p > 0.f) {
    uint32_t mw[4];
    dropout_maskw(e0, B.drop_seed, B.drop_thresh, mw);
    apply_maskw(dm, mw);
    inv = 1.f / (1.f - B.drop_p);
  }
  const float sinv = B.slope * inv;
  unpack8(dm, da);
  unpack8(a8, av);
#pragma unroll
  for (int i = 0; i < 8; ++i) dz[i] = da[i] * (av[i] > 0.f ? inv : sinv);
}

// Same with the activation sign recomputed from the raw conv output y (no read of `a`): sc / sh are the FOLDED
// forward constants (scale * inv, shift * inv -- fold_inv), i.e. the very fma whose sign the forward took.
__device__ __forceinline__ void dz1_from_y8(const bf16x8& da8, const float (&yy)[8], const float (&sc)[8],
                                            const float (&sh)[8], const NormBwdArgs& B, unsigned long long e0,
                                            float (&dz)[8]) {
  float da[8];
  bf16x8 dm = da8;
  float inv = 1.f;
  if (B.drop_p > 0.f) {
    uint32_t mw[4];
    dropout_maskw(e0, B.drop_seed, B.drop_thresh, mw);
    apply_maskw(dm, mw);
    inv = 1.f / (1.f - B.drop_p);
  }
  const float sinv = B.slope * inv;
  unpack8(dm, da);
#pragma unroll
  for (int i = 0; i < 8; ++i) dz[i] = da[i] * (fmaf(yy[i], sc[i], sh[i]) > 0.f ? inv : sinv);
}

// grid = (blocks_per_sample, N); each block strides over the vectors of one sample; partial sums are
// written per block: part[(n * blocks_per_sample + b)][2][Cp]. Cp/8 must divide blockDim.x (256), so a
// thread keeps one channel octet; two vectors per thread are in flight per iteration.
__global__ void __launch_bounds__(512)
norm_act_bwd_reduce_kernel(const __nv_bfloat16* __restrict__ dA, const __nv_bfloat16* __restrict__ a,
                           const __nv_bfloat16* __restrict__ y, NormBwdArgs B, int Cp, uint32_t vps,
                           float* __restrict__ part) {
  extern __shared__ float sh[];  // [2][blockDim.x][8]
  const uint32_t c8 = (uint32_t)Cp >> 3;
  const int n = blockIdx.y;
  const int lanes_v = blockDim.x / c8;
  const int cidx = threadIdx.x % c8;
  const int c0 = cidx * 8;
  const size_t base = (size_t)n * vps;
  const bf16x8* dAv = reinterpret_cast<const bf16x8*>(dA) + base;
  const bf16x8* av = reinterpret_cast<const bf16x8*>(a) + base;
  const bf16x8* yv = reinterpret_cast<const bf16x8*>(y) + base;
  float rstd[8], moff[8];   // xhat = y * rstd + moff
  float sc[8], sh_[8];
  const bool from_y = B.fshift != nullptr;
  const float finv = B.drop_p > 0.f ? 1.f / (1.f - B.drop_p) : 1.f;
#pragma unroll
  for (int k = 0; k < 8; ++k) {
    const float m = B.mean ? B.mean[(size_t)n * Cp + c0 + k] : 0.f;
    rstd[k] = B.rstd ? B.rstd[(size_t)n * Cp + c0 + k] : 0.f;
    moff[k] = -m * rstd[k];
    sc[k] = from_y ? fold_inv(B.gscale[(size_t)n * Cp + c0 + k], finv) : 0.f;
    sh_[k] = from_y ? fold_inv(B.fshift[(size_t)n * Cp + c0 + k], finv) : 0.f;
  }
  float s1[8], s2[8];
#pragma unroll
  for (int k = 0; k < 8; ++k) { s1[k] = 0.f; s2[k] = 0.f; }
  const uint32_t stride = gridDim.x * blockDim.x;
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < vps; i += 4 * stride) {
    bf16x8 d_[4], y_[4], a_[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const uint32_t idx = i + u * stride;
      if (idx < vps) {
        d_[u] = ld_stream(dAv + idx);
        y_[u] = ld_stream(yv + idx);
        if (!from_y) a_[u] = av[idx];
      }
    }
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const uint32_t idx = i + u * stride;
      if (idx >= vps) continue;
      float dz[8], yy[8];
      unpack8h(y_[u], yy);
      if (from_y) dz1_from_y8(d_[u], yy, sc, sh_, B, (unsigned long long)(base + idx) * 8ull, dz);
      else dz1_8(d_[u], a_[u], B, (unsigned long long)(base + idx) * 8ull, dz);
#pragma unroll
      for (int k = 0; k < 8; ++k) {
        s1[k] += dz[k];
        s2[k] = fmaf(dz[k], fmaf(yy[k], rstd[k], moff[k]), s2[k]);
      }
    }
  }
  float* sh1 = sh;
  float* sh2 = sh + blockDim.x * 8;
#pragma unroll
  for (int k = 0; k < 8; ++k) { sh1[threadIdx.x * 8 + k] = s1[k]; sh2[threadIdx.x * 8 + k] = s2[k]; }
  __syncthreads();
  // threads [0, Cp): channel c sums over the voxel lanes
  if (threadIdx.x < Cp) {
    const int c = threadIdx.x;
    float t1 = 0.f, t2 = 0.f;
    for (int l = 0; l < lanes_v; ++l) {
      t1 += sh1[(l * c8 + (c >> 3)) * 8 + (c & 7)];
      t2 += sh2[(l * c8 + (c >> 3)) * 8 + (c & 7)];
    }
    float* p = part + ((size_t)(n * gridDim.x + blockIdx.x) * 2) * Cp;
    p[c] = t1;
    p[Cp + c] = t2;
  }
}

// Reduce block partials -> c1, c2 per (n,c) and accumulate dgamma / dbeta (/ bias grad in eval-BN).
// mode as in stats_finalize. grid = (Cp/32), block = (32 channels, 32 lanes over the partial records): coalesced
// 128-byte rows, four loads in flight per thread, ONE block barrier per sample (the lane sums of sample n go to
// shared-memory buffer n & 1, which row 0 folds while the other rows already load sample n + 1). Fixed summation
// order: deterministic. This kernel sits on the critical path of every norm backward (~31 launches per step).
__global__ void __launch_bounds__(1024)
norm_bwd_finalize_kernel(const float* __restrict__ part, int blocks_per_sample, int Nb, int Cp, int C,
                         double count_per_sample, int mode, const float* __restrict__ xscale, float* __restrict__ c1,
                         float* __restrict__ c2, float* __restrict__ dgamma, float* __restrict__ dbeta,
                         float* __restrict__ dbias) {
  __shared__ double sh1[2][32][33], sh2[2][32][33];
  const int c = blockIdx.x * 32 + threadIdx.x;
  const int lane = threadIdx.y;
  double tot1 = 0.0, tot2 = 0.0;
  for (int n = 0; n < Nb; ++n) {
    const float* p0 = part + ((size_t)n * blocks_per_sample * 2) * Cp + c;
    double s1 = 0.0, s2 = 0.0;
    int b = lane;
    for (; b + 96 < blocks_per_sample; b += 128) {
      float f1[4], f2[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        f1[u] = p0[(size_t)(b + 32 * u) * 2 * Cp];
        f2[u] = p0[(size_t)(b + 32 * u) * 2 * Cp + Cp];
      }
      s1 += ((double)f1[0] + (double)f1[1]) + ((double)f1[2] + (double)f1[3]);
      s2 += ((double)f2[0] + (double)f2[1]) + ((double)f2[2] + (double)f2[3]);
    }
    for (; b < blocks_per_sample; b += 32) {
      s1 += (double)p0[(size_t)b * 2 * Cp];
      s2 += (double)p0[(size_t)b * 2 * Cp + Cp];
    }
    sh1[n & 1][lane][threadIdx.x] = s1;
    sh2[n & 1][lane][threadIdx.x] = s2;
    __syncthreads();
    if (lane == 0) {
      for (int k = 1; k < 32; ++k) { s1 += sh1[n & 1][k][threadIdx.x]; s2 += sh2[n & 1][k][threadIdx.x]; }
      tot1 += s1;
      tot2 += s2;
      if (mode == 0) {
        c1[(size_t)n * Cp + c] = (float)(s1 / count_per_sample);
        c2[(size_t)n * Cp + c] = (float)(s2 / count_per_sample);
      }
    }
  }
  if (lane != 0) return;
  if (mode != 0) {
    const double cnt = count_per_sample * Nb;
    for (int n = 0; n < Nb; ++n) {
      c1[(size_t)n * Cp + c] = mode == 1 ? (float)(tot1 / cnt) : 0.f;
      c2[(size_t)n * Cp + c] = mode == 1 ? (float)(tot2 / cnt) : 0.f;
    }
  }
  if (c < C) {
    if (dgamma) dgamma[c] = (float)tot2;
    if (dbeta) dbeta[c] = (float)tot1;
    // conv bias feeding a batch-statistics norm has an analytically zero gradient; with running
    // statistics (eval BatchNorm) it is gamma * rstd * S1.
    if (dbias) dbias[c] = mode == 2 ? (float)(tot1 * (double)xscale[c]) : 0.f;
  }
}

// dy = g*rstd * (dz1 - c1 - xhat * c2) = ka * dz1 + kc * y + kb with per-(n,c) constants held in
// registers (Cp/8 divides 256: fixed channel octet per thread). grid = (ceil(vps / (256*UNROLL)), N).
template <int UNROLL>
__global__ void __launch_bounds__(256, 2)
norm_act_bwd_apply_kernel(const __nv_bfloat16* __restrict__ dA, const __nv_bfloat16* __restrict__ a,
                          const __nv_bfloat16* __restrict__ y, __nv_bfloat16* __restrict__ dy, NormBwdArgs B, int Cp,
                          uint32_t vps) {
  const int n = blockIdx.y;
  const uint32_t c8 = (uint32_t)Cp >> 3;
  const size_t base = (size_t)n * vps;
  const bf16x8* dAv = reinterpret_cast<const bf16x8*>(dA) + base;
  const bf16x8* av = reinterpret_cast<const bf16x8*>(a) + base;
  const bf16x8* yv = reinterpret_cast<const bf16x8*>(y) + base;
  bf16x8* dyv = reinterpret_cast<bf16x8*>(dy) + base;
  const bool has_norm = B.mean != nullptr;
  const bool from_y = B.fshift != nullptr;
  float ka[8], kb[8], kc[8], sc_f[8], sh_f[8];   // sc_f / sh_f: the forward's folded affine constants (sign test)
  if (has_norm) {
    const size_t o = (size_t)n * Cp + (threadIdx.x % c8) * 8;
    const float finv = B.drop_p > 0.f ? 1.f / (1.f - B.drop_p) : 1.f;
#pragma unroll
    for (int k = 0; k < 8; ++k) {
      const float g = B.gscale[o + k], r = B.rstd[o + k], m = B.mean[o + k];
      ka[k] = g;
      kc[k] = -g * r * B.c2[o + k];
      kb[k] = -g * B.c1[o + k] - kc[k] * m;
      sc_f[k] = fold_inv(g, finv);
      sh_f[k] = from_y ? fold_inv(B.fshift[o + k], finv) : 0.f;
    }
  }
  const uint32_t i0 = blockIdx.x * (256u * UNROLL) + threadIdx.x;
  bf16x8 d_[UNROLL], a_[UNROLL], y_[UNROLL];
#pragma unroll
  for (int u = 0; u < UNROLL; ++u) {
    const uint32_t idx = i0 + u * 256u;
    if (idx < vps) {
      d_[u] = ld_stream(dAv + idx);
      if (!from_y) a_[u] = ld_stream(av + idx);
      if (has_norm) y_[u] = ld_stream(yv + idx);
    }
  }
#pragma unroll
  for (int u = 0; u < UNROLL; ++u) {
    const uint32_t idx = i0 + u * 256u;
    if (idx >= vps) continue;
    float dz[8], yy[8];
    if (has_norm) unpack8h(y_[u], yy);
    if (from_y) dz1_from_y8(d_[u], yy, sc_f, sh_f, B, (unsigned long long)(base + idx) * 8ull, dz);
    else dz1_8(d_[u], a_[u], B, (unsigned long long)(base + idx) * 8ull, dz);
    if (has_norm) {
#pragma unroll
      for (int k = 0; k < 8; ++k) dz[k] = fmaf(ka[k], dz[k], fmaf(kc[k], yy[k], kb[k]));
    }
    st_stream(dyv + idx, pack8(dz));
  }
}

// The same apply pass for the case every normed block of the networks takes (statistics present, activation sign
// recomputed from y), written for the INSTRUCTION roof: ncu showed the generic kernel above issue-bound, not
// HBM-bound (profiles/r02b_nab_apply_ncu_summary.txt: 219 warp instructions per 16-byte vector, 48 scalar constant
// loads + ~100 ALU instructions of per-thread prologue amortised over only 4 vectors, DRAM at 4.3 of 6.5 TB/s).
// Here the block derives the five per-channel constants ONCE into shared memory (thread = channel), every thread
// reads its octet's 40 floats as ten 16-byte shared loads and then streams kApplyVPT vectors in rounds of four loads
// in flight; dropout is a template parameter (no uniform branches in the loop), the tail test is one compare per
// round for whole blocks. Arithmetic and rounding are those of the generic kernel (same expressions).
constexpr int kApplyVPT = 8;   // 16-byte vectors per thread
template <bool DROP>
__global__ void __launch_bounds__(256, 2)
norm_act_bwd_apply_y_kernel(const __nv_bfloat16* __restrict__ dA, const __nv_bfloat16* __restrict__ y,
                            __nv_bfloat16* __restrict__ dy, NormBwdArgs B, int Cp, uint32_t vps) {
  __shared__ __align__(16) float ks[5][512];   // ka | kb | kc | sign-test scale | sign-test shift
  const int n = blockIdx.y;
  const float finv = DROP ? 1.f / (1.f - B.drop_p) : 1.f;
  for (int c = threadIdx.x; c < Cp; c += 256) {
    const size_t o = (size_t)n * Cp + c;
    const float g = B.gscale[o], r = B.rstd[o], m = B.mean[o];
    const float kc = -g * r * B.c2[o];
    ks[0][c] = g;
    ks[1][c] = -g * B.c1[o] - kc * m;
    ks[2][c] = kc;
    ks[3][c] = fold_inv(g, finv);
    ks[4][c] = fold_inv(B.fshift[o], finv);
  }
  __syncthreads();
  const uint32_t c8 = (uint32_t)Cp >> 3;
  const int c0 = (int)(threadIdx.x % c8) * 8;
  float ka[8], kb[8], kc[8], sc[8], sh[8];
#pragma unroll
  for (int h = 0; h < 2; ++h) {
    const float4 a4 = *reinterpret_cast<const float4*>(&ks[0][c0 + 4 * h]);
    const float4 b4 = *reinterpret_cast<const float4*>(&ks[1][c0 + 4 * h]);
    const float4 c4 = *reinterpret_cast<const float4*>(&ks[2][c0 + 4 * h]);
    const float4 s4 = *reinterpret_cast<const float4*>(&ks[3][c0 + 4 * h]);
    const float4 t4 = *reinterpret_cast<const float4*>(&ks[4][c0 + 4 * h]);
    ka[4 * h] = a4.x; ka[4 * h + 1] = a4.y; ka[4 * h + 2] = a4.z; ka[4 * h + 3] = a4.w;
    kb[4 * h] = b4.x; kb[4 * h + 1] = b4.y; kb[4 * h + 2] = b4.z; kb[4 * h + 3] = b4.w;
    kc[4 * h] = c4.x; kc[4 * h + 1] = c4.y; kc[4 * h + 2] = c4.z; kc[4 * h + 3] = c4.w;
    sc[4 * h] = s4.x; sc[4 * h + 1] = s4.y; sc[4 * h + 2] = s4.z; sc[4 * h + 3] = s4.w;
    sh[4 * h] = t4.x; sh[4 * h + 1] = t4.y; sh[4 * h + 2] = t4.z; sh[4 * h + 3] = t4.w;
  }
  const size_t base = (size_t)n * vps;
  const bf16x8* dAv = reinterpret_cast<const bf16x8*>(dA) + base;
  const bf16x8* yv = reinterpret_cast<const bf16x8*>(y) + base;
  bf16x8* dyv = reinterpret_cast<bf16x8*>(dy) + base;
  const float sinv = B.slope * finv;
  const uint32_t blk0 = blockIdx.x * (256u * kApplyVPT);
  const bool whole = blk0 + 256u * kApplyVPT <= vps;
#pragma unroll 1
  for (int rnd = 0; rnd < kApplyVPT / 4; ++rnd) {
    const uint32_t i0 = blk0 + rnd * 1024u + threadIdx.x;
    bf16x8 d_[4], y_[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const uint32_t idx = i0 + u * 256u;
      if (whole || idx < vps) {
        d_[u] = ld_stream(dAv + idx);
        y_[u] = ld_stream(yv + idx);
      }
    }
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const uint32_t idx = i0 + u * 256u;
      if (!whole && idx >= vps) continue;
      if (DROP) {
        uint32_t mw[4];
        dropout_maskw((unsigned long long)(base + idx) * 8ull, B.drop_seed, B.drop_thresh, mw);
        apply_maskw(d_[u], mw);
      }
      float da[8], yy[8], o[8];
      unpack8(d_[u], da);
      unpack8h(y_[u], yy);
#pragma unroll
      for (int k = 0; k < 8; ++k) {
        const float dz = da[k] * (fmaf(yy[k], sc[k], sh[k]) > 0.f ? finv : sinv);
        o[k] = fmaf(ka[k], dz, fmaf(kc[k], yy[k], kb[k]));
      }
      st_stream(dyv + idx, pack8(o));
    }
  }
}

// ------------------------------------------------------------------------------------------------
// MaxPool3d(2) backward: route dP to the first maximum of each window (d,h,w scan order, as torch)
// thread = (pooled voxel, 8 channels). accumulate != 0: dA += routed grad (skip-path grad already there)
// ------------------------------------------------------------------------------------------------
// DEFERRED: `a` points at the block's raw conv output y (fp16) and A describes its deferred activation; the
// activated values are recomputed with deferred_act8 (bit-identical to what the pooling forward compared).
template <bool DEFERRED>
__global__ void maxpool_bwd_kernel(const __nv_bfloat16* __restrict__ a, const __nv_bfloat16* __restrict__ dP,
                                   __nv_bfloat16* __restrict__ dA, int accumulate, int Cp, int Nb, int D, int H, int W,
                                   uint32_t per_sample /* pooled voxels * Cp/8 of one sample */, NormActArgs A) {
  // grid = (blocks, N): 32-bit index math inside a sample
  const uint32_t j0 = blockIdx.x * blockDim.x + threadIdx.x;
  if (j0 >= per_sample) return;
  const int n = blockIdx.y;
  const long long i = (long long)n * per_sample + j0;
  const uint32_t c8 = (uint32_t)Cp >> 3;
  uint32_t pv = j0 / c8;
  const int cidx = (int)(j0 - pv * c8);
  const uint32_t Wp = W >> 1, Hp = H >> 1;
  const int wx = (int)(pv % Wp); pv /= Wp;
  const int hy = (int)(pv % Hp);
  const int dz = (int)(pv / Hp);
  DeferredOctet K;
  if (DEFERRED) K.load(A, n, Cp, cidx * 8);
  float g[8];
  unpack8(ld_stream(reinterpret_cast<const bf16x8*>(dP) + i), g);
  float best[8];
  int arg[8];
#pragma unroll
  for (int k = 0; k < 8; ++k) { best[k] = -INFINITY; arg[k] = 0; }
  size_t e[8];
  bf16x8 raw[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    const int d = 2 * dz + (j >> 2), h = 2 * hy + ((j >> 1) & 1), w = 2 * wx + (j & 1);
    e[j] = ((((size_t)n * D + d) * H + h) * W + w) * c8 + cidx;
    raw[j] = ld_stream(reinterpret_cast<const bf16x8*>(a) + e[j]);
  }
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    float x[8];
    unpack8(DEFERRED ? K.apply(raw[j], (unsigned long long)e[j] * 8ull) : raw[j], x);
#pragma unroll
    for (int k = 0; k < 8; ++k)
      if (x[k] > best[k]) { best[k] = x[k]; arg[k] = j; }
  }
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    float o[8];
    if (accumulate) unpack8(ld_stream(reinterpret_cast<const bf16x8*>(dA) + e[j]), o);
#pragma unroll
    for (int k = 0; k < 8; ++k) o[k] = (accumulate ? o[k] : 0.f) + (arg[k] == j ? g[k] : 0.f);
    st_stream(reinterpret_cast<bf16x8*>(dA) + e[j], pack8(o));
  }
}

// The same routing for a block whose dA is COMPLETE after this pass (skip gradient + routed pool gradient), fused with
// that block's norm-backward reduction: the kernel already holds the block's raw output y (the activations it
// compares are recomputed from it, bit-identical to the materialised tensor), so it also accumulates
//   S1[n,c] = sum dz,  S2[n,c] = sum dz * xhat,   dz = bf16(dA) * lrelu'(y * sc + sh) * keep / (1 - p)
// into per-block records part[(n * gridDim.x + blockIdx.x)][2][Cp] (the format ub_norm_act_bwd takes as
// ext_partial), and the separate reduction pass over dA and y (4 B / element) is not run for the encoder blocks.
// Each block walks `iters` groups of 256 thread items so that a sample yields a few hundred records at most.
// blockDim.x = 256 and Cp / 8 divides 256: a thread keeps one channel octet.
__global__ void __launch_bounds__(256, 2)
maxpool_bwd_sums_kernel(const __nv_bfloat16* __restrict__ y, const __nv_bfloat16* __restrict__ dP,
                        __nv_bfloat16* __restrict__ dA, int accumulate, int Cp, int D, int H, int W,
                        uint32_t per_sample, int iters, NormActArgs A, const float* __restrict__ mean,
                        const float* __restrict__ rstd, float* __restrict__ part) {
  extern __shared__ float sh[];  // [2][256][8]
  const int n = blockIdx.y;
  const uint32_t c8 = (uint32_t)Cp >> 3;
  const int cidx = (int)(threadIdx.x % c8);
  const uint32_t Wp = W >> 1, Hp = H >> 1;
  DeferredOctet K;
  K.load(A, n, Cp, cidx * 8);
  const float inv = K.has_drop ? 1.f / (1.f - A.drop_p) : 1.f;
  const float sinv = A.slope * inv;
  // 32-bit vector offsets inside the sample (vectors per sample < 2^31): window voxel j = (jd, jh, jw)
  const uint32_t vps = (uint32_t)D * H * W * c8;
  const uint32_t off_w = c8, off_h = (uint32_t)W * c8, off_d = (uint32_t)H * W * c8;
  const bf16x8* ys = reinterpret_cast<const bf16x8*>(y) + (size_t)n * vps;
  bf16x8* dAs = reinterpret_cast<bf16x8*>(dA) + (size_t)n * vps;
  const bf16x8* dPs = reinterpret_cast<const bf16x8*>(dP) + (size_t)n * per_sample;
  const unsigned long long ebase = (unsigned long long)n * vps * 8ull;   // element index of the sample's first channel
  float s1[8], s2[8];
#pragma unroll
  for (int k = 0; k < 8; ++k) { s1[k] = 0.f; s2[k] = 0.f; }
#pragma unroll 1
  for (int it = 0; it < iters; ++it) {
    const uint32_t j0 = (blockIdx.x * (uint32_t)iters + it) * 256u + threadIdx.x;
    if (j0 >= per_sample) break;
    uint32_t pv = j0 / c8;
    const uint32_t wx = pv % Wp; pv /= Wp;
    const uint32_t hy = pv % Hp;
    const uint32_t dz_ = pv / Hp;
    const uint32_t e00 = ((2 * dz_ * H + 2 * hy) * W + 2 * wx) * c8 + cidx;     // window voxel (0, 0, 0)
    uint32_t arg = 0;          // 3 bits per channel: index of the first maximum of the window
    {
      // y is read through L1 (default caching): the second phase below re-reads the same 8 rows a few hundred
      // cycles later instead of holding them in 32 registers (the kernel was register-bound at one block per SM)
      bf16x8 raw[8];
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const uint4 t = __ldg(reinterpret_cast<const uint4*>(ys + e00 + (j >> 2) * off_d + ((j >> 1) & 1) * off_h + (j & 1) * off_w));
        *reinterpret_cast<uint4*>(&raw[j]) = t;
      }
      float best[8];
#pragma unroll
      for (int k = 0; k < 8; ++k) best[k] = -INFINITY;
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const uint32_t ej = e00 + (j >> 2) * off_d + ((j >> 1) & 1) * off_h + (j & 1) * off_w;
        float x[8];
        unpack8(K.apply(raw[j], ebase + (unsigned long long)ej * 8ull), x);
#pragma unroll
        for (int k = 0; k < 8; ++k)
          if (x[k] > best[k]) { best[k] = x[k]; arg = (arg & ~(7u << (3 * k))) | ((uint32_t)j << (3 * k)); }
      }
    }
    float g[8];
    unpack8(ld_stream(dPs + j0), g);
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const uint32_t ej = e00 + (j >> 2) * off_d + ((j >> 1) & 1) * off_h + (j & 1) * off_w;
      float o[8];
      if (accumulate) unpack8(ld_stream(dAs + ej), o);
#pragma unroll
      for (int k = 0; k < 8; ++k) o[k] = (accumulate ? o[k] : 0.f) + (((arg >> (3 * k)) & 7u) == (uint32_t)j ? g[k] : 0.f);
      bf16x8 pk = pack8(o);
      st_stream(dAs + ej, pk);
      // reduction terms from the ROUNDED gradient (what the apply pass reads back) and the forward's own fma
      if (K.has_drop) {
        uint32_t mw[4];
        dropout_maskw(ebase + (unsigned long long)ej * 8ull, K.seed, K.thresh, mw);
        apply_maskw(pk, mw);
      }
      float da[8], yy[8];
      unpack8(pk, da);
      bf16x8 yraw;
      *reinterpret_cast<uint4*>(&yraw) = __ldg(reinterpret_cast<const uint4*>(ys + ej));
      unpack8h(yraw, yy);
#pragma unroll
      for (int k = 0; k < 8; ++k) {
        const float dz = da[k] * (fmaf(yy[k], K.sc[k], K.sh[k]) > 0.f ? inv : sinv);
        s1[k] += dz;
        s2[k] = fmaf(dz, yy[k], s2[k]);
      }
    }
  }
  // S2 = sum dz * xhat = rstd * sum dz*y - mean*rstd * sum dz
  float* sh1 = sh;
  float* sh2 = sh + 256 * 8;
#pragma unroll
  for (int k = 0; k < 8; ++k) {
    const float r = rstd[(size_t)n * Cp + cidx * 8 + k], m = mean[(size_t)n * Cp + cidx * 8 + k];
    sh1[threadIdx.x * 8 + k] = s1[k];
    sh2[threadIdx.x * 8 + k] = fmaf(r, s2[k], -m * r * s1[k]);
  }
  __syncthreads();
  const int lanes_v = 256 / (int)c8;
  for (int c = threadIdx.x; c < Cp; c += 256) {
    float t1 = 0.f, t2 = 0.f;
    for (int l = 0; l < lanes_v; ++l) {
      t1 += sh1[(l * c8 + (c >> 3)) * 8 + (c & 7)];
      t2 += sh2[(l * c8 + (c >> 3)) * 8 + (c & 7)];
    }
    float* p = part + ((size_t)(n * gridDim.x + blockIdx.x) * 2) * Cp;
    p[c] = t1;
    p[Cp + c] = t2;
  }
}

// ------------------------------------------------------------------------------------------------
// column sums of a bf16 [rows][Cp] matrix -> fp32 [C] (bias gradients of convs without a norm)
// grid = nblocks; block = 256; part[nblocks][Cp]; second launch with rows=nblocks reduces partials
// ------------------------------------------------------------------------------------------------
__global__ void colsum_bf16_kernel(const __nv_bfloat16* __restrict__ x, long long rows, int Cp,
                                   float* __restrict__ part) {
  extern __shared__ float sh[];
  const int c8 = Cp >> 3;
  const int lanes_v = blockDim.x / c8;
  const int cidx = threadIdx.x % c8, vlane = threadIdx.x / c8;
  float s[8];
#pragma unroll
  for (int k = 0; k < 8; ++k) s[k] = 0.f;
  if (vlane < lanes_v)
    for (long long r = (long long)blockIdx.x * lanes_v + vlane; r < rows; r += (long long)gridDim.x * lanes_v) {
      float v[8];
      unpack8(ld_stream(reinterpret_cast<const bf16x8*>(x) + (size_t)r * c8 + cidx), v);
#pragma unroll
      for (int k = 0; k < 8; ++k) s[k] += v[k];
    }
#pragma unroll
  for (int k = 0; k < 8; ++k) sh[threadIdx.x * 8 + k] = vlane < lanes_v ? s[k] : 0.f;
  __syncthreads();
  if (threadIdx.x < Cp) {
    const int c = threadIdx.x;
    float t = 0.f;
    for (int l = 0; l < lanes_v; ++l) t += sh[(l * c8 + (c >> 3)) * 8 + (c & 7)];
    part[(size_t)blockIdx.x * Cp + c] = t;
  }
}
// grid = ceil(C / 8), block = (32 lanes over the block partials, 8 channels): one warp per channel, shuffle tree
__global__ void colsum_finish_kernel(const float* __restrict__ part, int nblocks, int Cp, int C,
                                     float* __restrict__ out) {
  const int c = blockIdx.x * blockDim.y + threadIdx.y;
  if (c >= C) return;
  double t = 0.0;
  for (int b = threadIdx.x; b < nblocks; b += 32) t += (double)part[(size_t)b * Cp + c];
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) t += __shfl_xor_sync(0xffffffffu, t, o);
  if (threadIdx.x == 0) out[c] = (float)t;
}

// ------------------------------------------------------------------------------------------------
// weights: torch fp32 layout -> packed bf16 [block][rows_pad][cols_pad] (K-major rows), and back
// ------------------------------------------------------------------------------------------------
struct WeightPackArgs {
  int nblocks, rows, cols, rows_pad, cols_pad;
  long long stride_row, stride_col;  // element strides in the fp32 source for (row, col)
  int src_tap_stride;                // element stride of the source tap index
  int split_pad, split_real;         // concat: padded channel p >= split_pad maps to real p - split_pad + split_real
  int split_on_rows;                 // the concatenated (input-channel) axis is rows (dgrad) or cols (fwd)
  int rows_fold, fold_tap_stride;    // rows_fold > 0: row = fold * rows_fold + r, source tap += fold * fold_tap_stride
  int f16_cols;                      // columns [0, f16_cols) are written as IEEE fp16 instead of bf16 (the K range of
                                     // a source whose activations the consumer evaluates as an fp16 operand)
  int tapmap[64];                    // packed block -> source tap index
};
// padded concat index -> real channel index, or -1 for a pad slot
__device__ __forceinline__ int concat_real_index(int p, int split_pad, int split_real, int n_real) {
  if (split_pad == 0) return p < n_real ? p : -1;
  if (p < split_pad) return p < split_real ? p : -1;
  const int r = p - split_pad + split_real;
  return r < n_real ? r : -1;
}
__device__ __forceinline__ void pack_weight_element(const float* __restrict__ w, __nv_bfloat16* __restrict__ out,
                                                    const WeightPackArgs& A, long long i) {
  const int col = (int)(i % A.cols_pad);
  int row = (int)((i / A.cols_pad) % A.rows_pad);
  const int blk = (int)(i / ((long long)A.cols_pad * A.rows_pad));
  int tap = A.tapmap[blk];
  if (A.rows_fold > 0) {
    tap += (row / A.rows_fold) * A.fold_tap_stride;
    row = row % A.rows_fold;
  }
  const int rr = A.split_on_rows ? concat_real_index(row, A.split_pad, A.split_real, A.rows) : (row < A.rows ? row : -1);
  const int cc = A.split_on_rows ? (col < A.cols ? col : -1) : concat_real_index(col, A.split_pad, A.split_real, A.cols);
  float v = 0.f;
  if (rr >= 0 && cc >= 0)
    v = w[(size_t)rr * A.stride_row + (size_t)cc * A.stride_col + (size_t)tap * A.src_tap_stride];
  if (col < A.f16_cols) reinterpret_cast<__half*>(out)[i] = __float2half_rn(v);
  else out[i] = __float2bfloat16_rn(v);
}
__global__ void pack_weights_kernel(const float* __restrict__ w, __nv_bfloat16* __restrict__ out, WeightPackArgs A) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const long long total = (long long)A.nblocks * A.rows_pad * A.cols_pad;
  if (i >= total) return;
  pack_weight_element(w, out, A, i);
}

// All the weights of a network in ONE launch (a forward / backward pass re-packs its bf16 operand copies from the
// live fp32 Parameters every time it runs: ~25 us for the generator's 22.6 M weights, and no cache that an
// out-of-band write to parameter memory could leave stale). The table is a __grid_constant__ kernel argument.
constexpr int kPackMaxTensors = 32;
struct WeightPackBatch {
  WeightPackArgs a[kPackMaxTensors];
  const float* w[kPackMaxTensors];
  __nv_bfloat16* out[kPackMaxTensors];
  int block_begin[kPackMaxTensors + 1];
  int count;
};
// thread = one (packed row, packed column) pair, looping over the packed tap blocks: the taps of one (co, ci) pair
// are contiguous in the torch layout (<= 256 bytes), so a warp reads whole cache lines once and every block's
// write is a contiguous run of columns (the per-element kernel above gathers with a 108-byte stride instead).
__global__ void __launch_bounds__(256) pack_weights_multi_kernel(const __grid_constant__ WeightPackBatch B) {
  __shared__ int s_t;
  if (threadIdx.x == 0) {
    int t = 0;
    while (t + 1 < B.count && (int)blockIdx.x >= B.block_begin[t + 1]) ++t;
    s_t = t;
  }
  __syncthreads();
  const int t = s_t;
  const WeightPackArgs& A = B.a[t];
  const float* __restrict__ w = B.w[t];
  __nv_bfloat16* __restrict__ out = B.out[t];
  const long long plane = (long long)A.rows_pad * A.cols_pad;
  const long long j = (long long)((int)blockIdx.x - B.block_begin[t]) * 256 + threadIdx.x;
  if (j >= plane) return;
  const int col = (int)(j % A.cols_pad);
  int row = (int)(j / A.cols_pad);
  int fold_tap = 0;
  if (A.rows_fold > 0) {
    fold_tap = (row / A.rows_fold) * A.fold_tap_stride;
    row = row % A.rows_fold;
  }
  const int rr = A.split_on_rows ? concat_real_index(row, A.split_pad, A.split_real, A.rows) : (row < A.rows ? row : -1);
  const int cc = A.split_on_rows ? (col < A.cols ? col : -1) : concat_real_index(col, A.split_pad, A.split_real, A.cols);
  const bool real = rr >= 0 && cc >= 0;
  const float* src = w + (real ? (size_t)rr * A.stride_row + (size_t)cc * A.stride_col : 0);
  const bool f16 = col < A.f16_cols;
  // the taps of a thread are independent loads from one or two cache lines: keep several in flight (the serial
  // loop was latency-bound: 64 us for the generator's 135 MB of traffic)
  int blk = 0;
  for (; blk + 4 <= A.nblocks; blk += 4) {
    float v[4];
#pragma unroll
    for (int q = 0; q < 4; ++q)
      v[q] = real ? __ldg(src + (size_t)(A.tapmap[blk + q] + fold_tap) * A.src_tap_stride) : 0.f;
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const long long i = (blk + q) * plane + j;
      if (f16) reinterpret_cast<__half*>(out)[i] = __float2half_rn(v[q]);
      else out[i] = __float2bfloat16_rn(v[q]);
    }
  }
  for (; blk < A.nblocks; ++blk) {
    const float v = real ? __ldg(src + (size_t)(A.tapmap[blk] + fold_tap) * A.src_tap_stride) : 0.f;
    const long long i = blk * plane + j;
    if (f16) reinterpret_cast<__half*>(out)[i] = __float2half_rn(v);
    else out[i] = __float2bfloat16_rn(v);
  }
}

// split-K reduction of wgrad partials [nsplit][ntap][ci_total][co_total] -> torch layout fp32 grad
struct WgradReduceArgs {
  int nsplit, ntap, ci_total, co_total, ci, co;
  long long stride_ci, stride_co;    // element strides in the destination for (ci, co)
  int dst_tap_stride;
  int split_pad, split_real;         // concat mapping of the padded ci index (see WeightPackArgs)
  int tapmap[64];                    // partial tap index -> destination tap index (-1: skip)
};
__global__ void wgrad_reduce_kernel(const float* __restrict__ part, float* __restrict__ grad, WgradReduceArgs A) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const long long per_split = (long long)A.ntap * A.ci_total * A.co_total;
  if (i >= per_split) return;
  const int co = (int)(i % A.co_total);
  const int ci = (int)((i / A.co_total) % A.ci_total);
  const int tap = (int)(i / ((long long)A.co_total * A.ci_total));
  const int cir = concat_real_index(ci, A.split_pad, A.split_real, A.ci);
  if (co >= A.co || cir < 0 || A.tapmap[tap] < 0) return;
  float s = 0.f;
  for (int k = 0; k < A.nsplit; ++k) s += part[(size_t)k * per_split + i];
  grad[(size_t)cir * A.stride_ci + (size_t)co * A.stride_co + (size_t)A.tapmap[tap] * A.dst_tap_stride] = s;
}
// Tiled variant for the LARGE outputs (>= 512 blocks of one padded input-channel row x 64 output channels): a block
// sums the splits reading 256-byte runs of the partial records, transposes (co, tap) through shared memory and writes
// runs of `taps` contiguous floats of the torch layout -- the kernel above scatters single floats 108 bytes
// ([co][ci][27]) or more apart, 32 sectors per warp store. Measured per launch (profiles/r02i_reduce_pack_ab.txt):
// 512 x 256 x 4^3 89 -> 51 us, 512 x 512 x 3^3 88 -> 45 us, 256 x 512 x 3^3 38 -> 27 us; with fewer blocks the
// scatter kernel's 27x finer grid wins (64 -> 64 x 3^3, 37 splits: 10 us against 43 us) and keeps the job.
constexpr int kRedTileCols = 64;
__global__ void __launch_bounds__(256) wgrad_reduce_tiled_kernel(const float* __restrict__ part, float* __restrict__ grad,
                                                                 WgradReduceArgs A, int dst_ntaps) {
  __shared__ float tile[kRedTileCols * 65];
  const int ctiles = (A.co_total + kRedTileCols - 1) / kRedTileCols;
  const int ci = (int)blockIdx.x / ctiles, co0 = ((int)blockIdx.x % ctiles) * kRedTileCols;
  const int cir = concat_real_index(ci, A.split_pad, A.split_real, A.ci);
  if (cir < 0) return;
  const int TP = dst_ntaps | 1;
  const long long per_split = (long long)A.ntap * A.ci_total * A.co_total;
  for (int idx = threadIdx.x; idx < kRedTileCols * dst_ntaps; idx += 256) tile[(idx / dst_ntaps) * TP + idx % dst_ntaps] = 0.f;
  __syncthreads();
  for (int idx = threadIdx.x; idx < A.ntap * kRedTileCols; idx += 256) {
    const int c = idx & (kRedTileCols - 1), tap = idx / kRedTileCols;
    const int dt = A.tapmap[tap];
    if (dt < 0 || co0 + c >= A.co_total) continue;
    const float* p = part + ((size_t)tap * A.ci_total + ci) * A.co_total + co0 + c;
    float s = 0.f;
    for (int k = 0; k < A.nsplit; ++k) s += __ldg(p + (size_t)k * per_split);
    tile[c * TP + dt] = s;
  }
  __syncthreads();
  for (int idx = threadIdx.x; idx < kRedTileCols * dst_ntaps; idx += 256) {
    const int c = idx / dst_ntaps, t = idx - c * dst_ntaps;
    const int co = co0 + c;
    if (co >= A.co) continue;
    grad[(size_t)cir * A.stride_ci + (size_t)co * A.stride_co + (size_t)t * A.dst_tap_stride] = tile[c * TP + t];
  }
}
// Same reduction for SMALL outputs with many splits (the 32-channel layers: 27.6 k outputs x 148 splits): eight lanes
// share one output and stride over the splits, so the serial chain is 8x shorter; shuffle tree, fixed order.
__global__ void wgrad_reduce_wide_kernel(const float* __restrict__ part, float* __restrict__ grad, WgradReduceArgs A) {
  const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const long long per_split = (long long)A.ntap * A.ci_total * A.co_total;
  const long long i = t >> 3;
  const int sub = (int)(t & 7);
  float s = 0.f;
  if (i < per_split)
    for (int k = sub; k < A.nsplit; k += 8) s += part[(size_t)k * per_split + i];
#pragma unroll
  for (int o = 4; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  if (i >= per_split || sub != 0) return;
  const int co = (int)(i % A.co_total);
  const int ci = (int)((i / A.co_total) % A.ci_total);
  const int tap = (int)(i / ((long long)A.co_total * A.ci_total));
  const int cir = concat_real_index(ci, A.split_pad, A.split_real, A.ci);
  if (co >= A.co || cir < 0 || A.tapmap[tap] < 0) return;
  grad[(size_t)cir * A.stride_ci + (size_t)co * A.stride_co + (size_t)A.tapmap[tap] * A.dst_tap_stride] = s;
}

// ------------------------------------------------------------------------------------------------
// losses (fp32 NCDHW tensors at the module boundary)
// ------------------------------------------------------------------------------------------------
// L1: loss = mean |a - b|  (ref: model.py:126,136).  Block partials + last-block finish.
__global__ void l1_fwd_kernel(const float* __restrict__ a, const float* __restrict__ b, long long n,
                              double* __restrict__ part, unsigned int* __restrict__ ticket, float* __restrict__ loss) {
  __shared__ double sh[32];
  double s = 0.0;
  const long long n4 = n >> 2;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (long long)gridDim.x * blockDim.x) {
    const float4 x = __ldg(reinterpret_cast<const float4*>(a) + i), y = __ldg(reinterpret_cast<const float4*>(b) + i);
    s += (double)(fabsf(x.x - y.x) + fabsf(x.y - y.y) + fabsf(x.z - y.z) + fabsf(x.w - y.w));
  }
  if (blockIdx.x == 0 && threadIdx.x == 0)
    for (long long i = n4 * 4; i < n; ++i) s += (double)fabsf(a[i] - b[i]);
  for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = s;
  __syncthreads();
  if (threadIdx.x == 0) {
    double t = 0.0;
    for (int i = 0; i < (int)(blockDim.x >> 5); ++i) t += sh[i];
    part[blockIdx.x] = t;
    __threadfence();
    const unsigned int k = atomicAdd(ticket, 1u);
    if (k == gridDim.x - 1) {
      double tot = 0.0;
      for (unsigned int j = 0; j < gridDim.x; ++j) tot += ((volatile double*)part)[j];
      *loss = (float)(tot / (double)n);
      *ticket = 0u;
    }
  }
}
// d a = sign(a - b) * g / n ; g is a device scalar (upstream gradient)
__global__ void l1_bwd_kernel(const float* __restrict__ a, const float* __restrict__ b, const float* __restrict__ g,
                              long long n, float* __restrict__ da) {
  const float gs = __ldg(g) / (float)n;
  const long long n4 = n >> 2;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (long long)gridDim.x * blockDim.x) {
    const float4 x = __ldg(reinterpret_cast<const float4*>(a) + i), y = __ldg(reinterpret_cast<const float4*>(b) + i);
    float4 o;
    o.x = x.x > y.x ? gs : (x.x < y.x ? -gs : 0.f);
    o.y = x.y > y.y ? gs : (x.y < y.y ? -gs : 0.f);
    o.z = x.z > y.z ? gs : (x.z < y.z ? -gs : 0.f);
    o.w = x.w > y.w ? gs : (x.w < y.w ? -gs : 0.f);
    reinterpret_cast<float4*>(da)[i] = o;
  }
  if (blockIdx.x == 0 && threadIdx.x == 0)
    for (long long i = n4 * 4; i < n; ++i) da[i] = a[i] > b[i] ? gs : (a[i] < b[i] ? -gs : 0.f);
}

// BCE with logits against a constant target t in {0,1} (ref: model.py:155,175,191-192):
// loss = mean(max(x,0) - x t + log1p(exp(-|x|))); unit gradient (sigmoid(x) - t) / n is emitted in the
// same pass. One block (the PatchGAN logit map is tiny).
__global__ void bce_logits_kernel(const float* __restrict__ x, const float* __restrict__ target_ptr, float target_const,
                                  int n, float* __restrict__ loss, float* __restrict__ dx_unit) {
  __shared__ double sh[32];
  double s = 0.0;
  for (int i = threadIdx.x; i < n; i += blockDim.x) {
    const float v = x[i];
    const float target = target_ptr ? target_ptr[i] : target_const;
    s += (double)(fmaxf(v, 0.f) - v * target + log1pf(expf(-fabsf(v))));
    if (dx_unit) dx_unit[i] = (1.f / (1.f + expf(-v)) - target) / (float)n;
  }
  for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = s;
  __syncthreads();
  if (threadIdx.x == 0) {
    double t = 0.0;
    for (int i = 0; i < (int)(blockDim.x >> 5); ++i) t += sh[i];
    *loss = (float)(t / n);
  }
}

// y[i] = x[i] * (*g)   (scale a unit gradient by a device scalar)
__global__ void scale_by_scalar_kernel(const float* __restrict__ x, const float* __restrict__ g, long long n,
                                       float* __restrict__ y) {
  const float gs = __ldg(g);
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
    y[i] = x[i] * gs;
}

// ------------------------------------------------------------------------------------------------
// evaluation: per-voxel relative error + masked, probseg-weighted ROI means
//   ref: eval.py:154-166 (do_calc_diff_maps) and eval.py:217-258 (do_calc_error_avg)
// Volumes are channel-last [X][Y][Z][C] as nibabel stores them (np.moveaxis(0,-1), model.py:344-346).
//   angular == 0: diff = |p - t| / t          (division by zero gives inf / nan exactly as numpy)
//   angular == 1: d = (p - t) mod 360 (python sign convention), diff = d < 180 ? d : 360 - d
// Reduction: e = |diff|; e = mask > 0 ? e : 0; e = (e == inf) ? 0 : e (NaN kept);
//            sums[r][c] += probseg[v][r] * e;  norms[r] += probseg[v][r]
// ------------------------------------------------------------------------------------------------
__global__ void relerr_kernel(const float* __restrict__ pred, const float* __restrict__ tgt,
                              const unsigned char* __restrict__ mask, const float* __restrict__ probseg, int C, int R,
                              long long nvox, int angular, float* __restrict__ diff, double* __restrict__ sums,
                              double* __restrict__ norms) {
  // per-thread accumulators for up to 3 ROIs x 8 channels
  double acc[3][8];
  double nrm[3];
#pragma unroll
  for (int r = 0; r < 3; ++r) {
    nrm[r] = 0.0;
#pragma unroll
    for (int c = 0; c < 8; ++c) acc[r][c] = 0.0;
  }
  for (long long v = (long long)blockIdx.x * blockDim.x + threadIdx.x; v < nvox; v += (long long)gridDim.x * blockDim.x) {
    float ps[3] = {0.f, 0.f, 0.f};
    if (probseg)
      for (int r = 0; r < R; ++r) { ps[r] = probseg[(size_t)v * R + r]; nrm[r] += (double)ps[r]; }
    const bool in_mask = mask ? mask[v] > 0 : true;
    for (int c = 0; c < C; ++c) {
      const float p = pred[(size_t)v * C + c], t = tgt[(size_t)v * C + c];
      float d;
      if (!angular) {
        d = fabsf(p - t) / t;
      } else {
        float m = fmodf(p - t, 360.f);
        if (m < 0.f) m += 360.f;
        d = m < 180.f ? m : 360.f - m;
      }
      if (diff) diff[(size_t)v * C + c] = d;
      float e = fabsf(d);
      e = in_mask ? e : 0.f;
      e = isinf(e) ? 0.f : e;
      if (probseg)
        for (int r = 0; r < R; ++r) acc[r][c] += (double)ps[r] * (double)e;
    }
  }
  if (!probseg) return;
  // warp reduce then one atomic per warp per entry (3*8+3 doubles)
  for (int r = 0; r < R; ++r) {
    double t = nrm[r];
    for (int o = 16; o > 0; o >>= 1) t += __shfl_xor_sync(0xffffffffu, t, o);
    if ((threadIdx.x & 31) == 0) atomicAdd(norms + r, t);
    for (int c = 0; c < C; ++c) {
      double s = acc[r][c];
      for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
      if ((threadIdx.x & 31) == 0) atomicAdd(sums + r * C + c, s);
    }
  }
}

// ------------------------------------------------------------------------------------------------
// Output head of the generator: 1x1x1 conv to <= 8 channels fused with the layout change
//   ref: monai BasicUNet.final_conv (nn.Conv3d(32, 6, 1)), ref:model.py:22-28; output NCDHW fp32.
// The tensor-core path would write a 32-channel padded bf16 tensor and unpack it (192 B/voxel of traffic
// for 24 B of result); this is a matvec of 6 x 32 per voxel, done on the CUDA cores at HBM speed.
// thread = (voxel, octet of input channels): 16-byte coalesced loads, partial dot products over the 8
// channels, two xor-shuffles across the 4 octet lanes, lane `oct` stores outputs oct and oct + 4.
// ------------------------------------------------------------------------------------------------
constexpr int kC1MaxCo = 8;
struct Conv1x1Weights {
  float w[kC1MaxCo][32];   // [co][ci], zero padded
  float b[kC1MaxCo];
};

// DEFERRED: u is the raw conv output y (fp16) of the last block and A its deferred activation.
template <int CO, bool DEFERRED>
__global__ void __launch_bounds__(256)
conv1x1_to_ncdhw_kernel(const __nv_bfloat16* __restrict__ u, float* __restrict__ out, const Conv1x1Weights* __restrict__ Wg,
                        uint32_t V, NormActArgs A) {
  // grid = (blocks, N): each block strides over the voxels of one sample; weights live in registers
  const int n = blockIdx.y;
  const int oct = threadIdx.x & 3;
  float wr[CO][8], br[CO];
#pragma unroll
  for (int c = 0; c < CO; ++c) {
    br[c] = Wg->b[c];
#pragma unroll
    for (int k = 0; k < 8; ++k) wr[c][k] = Wg->w[c][oct * 8 + k];
  }
  const bf16x8* up = reinterpret_cast<const bf16x8*>(u + (size_t)n * V * 32);
  float* op = out + (size_t)n * CO * V;
  DeferredOctet K;
  if (DEFERRED) K.load(A, n, 32, oct * 8);
  constexpr int UNR = 4;             // independent 16-byte loads in flight per thread
  const uint32_t vstep = gridDim.x * (64 * UNR);
  // all lanes of a warp run the same number of iterations (the shuffles below need the full warp)
  for (uint32_t vb = blockIdx.x * (64 * UNR); vb < V; vb += vstep) {
    bf16x8 raw[UNR];
#pragma unroll
    for (int q = 0; q < UNR; ++q) {
      const uint32_t v = vb + q * 64 + (threadIdx.x >> 2);
      if (v < V) raw[q] = ld_stream(up + (size_t)v * 4 + oct);
    }
#pragma unroll
    for (int q = 0; q < UNR; ++q) {
      const uint32_t v = vb + q * 64 + (threadIdx.x >> 2);
      const bool ok = v < V;
      float x[8];
      unpack8(DEFERRED ? K.apply(raw[q], ((unsigned long long)n * V + v) * 32ull + oct * 8) : raw[q], x);
      float mine0 = 0.f, mine1 = 0.f;   // outputs oct and oct + 4
#pragma unroll
      for (int c = 0; c < CO; ++c) {
        float a = 0.f;
#pragma unroll
        for (int k = 0; k < 8; ++k) a = fmaf(ok ? x[k] : 0.f, wr[c][k], a);
        a += __shfl_xor_sync(0xffffffffu, a, 1);
        a += __shfl_xor_sync(0xffffffffu, a, 2);
        if ((c & 3) == oct) { if (c < 4) mine0 = a + br[c]; else mine1 = a + br[c]; }
      }
      if (ok) {
        if (oct < CO) __stcs(op + (size_t)oct * V + v, mine0);
        if (oct + 4 < CO) __stcs(op + (size_t)(oct + 4) * V + v, mine1);
      }
    }
  }
}

// Backward of the above in one pass over dout (NCDHW fp32) and u (NDHWC bf16, 32 channels):
//   du[v][ci] = sum_co dout[co][v] * W[co][ci]          (bf16, may be skipped)
//   dW[co][ci] = sum_v dout[co][v] * u[v][ci],  db[co] = sum_v dout[co][v]     (per-block partials)
// thread = (voxel, octet of ci); grid = (blocks, N); part: [blocks * N][kC1MaxCo][33] floats (column 32 =
// bias gradient).
template <int CO, bool DEFERRED>
__global__ void __launch_bounds__(256, 2)
conv1x1_from_ncdhw_bwd_kernel(const float* __restrict__ dout, const __nv_bfloat16* __restrict__ u,
                              __nv_bfloat16* __restrict__ du, const Conv1x1Weights* __restrict__ Wg, uint32_t V,
                              int want_w, float* __restrict__ part, NormActArgs A) {
  __shared__ float red[8][CO][33];
  const int n = blockIdx.y;
  const int oct = threadIdx.x & 3;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  float wr[CO][8];
#pragma unroll
  for (int c = 0; c < CO; ++c)
#pragma unroll
    for (int k = 0; k < 8; ++k) wr[c][k] = Wg->w[c][oct * 8 + k];
  float gw[CO][8], gb[CO];
#pragma unroll
  for (int c = 0; c < CO; ++c) {
    gb[c] = 0.f;
#pragma unroll
    for (int k = 0; k < 8; ++k) gw[c][k] = 0.f;
  }
  const float* gp = dout + (size_t)n * CO * V;
  const bf16x8* up = reinterpret_cast<const bf16x8*>(u) + (size_t)n * V * 4;
  bf16x8* dup = reinterpret_cast<bf16x8*>(du) + (size_t)n * V * 4;
  DeferredOctet K;
  if (DEFERRED) K.load(A, n, 32, oct * 8);
  constexpr int UNR = 2;
  const uint32_t vstep = gridDim.x * (64 * UNR);
  for (uint32_t vb = blockIdx.x * (64 * UNR) + (threadIdx.x >> 2); vb < V; vb += vstep) {
    float g[UNR][CO];
    bf16x8 ux[UNR];
#pragma unroll
    for (int q = 0; q < UNR; ++q) {
      const uint32_t v = vb + q * 64;
      if (v < V) {
#pragma unroll
        for (int c = 0; c < CO; ++c) g[q][c] = __ldcs(gp + (size_t)c * V + v);
        if (want_w) ux[q] = ld_stream(up + (size_t)v * 4 + oct);
      }
    }
#pragma unroll
    for (int q = 0; q < UNR; ++q) {
      const uint32_t v = vb + q * 64;
      if (v >= V) continue;
      if (du != nullptr) {
        float o[8];
#pragma unroll
        for (int k = 0; k < 8; ++k) {
          float a = 0.f;
#pragma unroll
          for (int c = 0; c < CO; ++c) a = fmaf(g[q][c], wr[c][k], a);
          o[k] = a;
        }
        st_stream(dup + (size_t)v * 4 + oct, pack8(o));
      }
      if (want_w) {
        float x[8];
        unpack8(DEFERRED ? K.apply(ux[q], ((unsigned long long)n * V + v) * 32ull + oct * 8) : ux[q], x);
#pragma unroll
        for (int c = 0; c < CO; ++c) {
          gb[c] += g[q][c];
#pragma unroll
          for (int k = 0; k < 8; ++k) gw[c][k] = fmaf(g[q][c], x[k], gw[c][k]);
        }
      }
    }
  }
  if (!want_w) return;
  // reduce over the 8 voxel lanes that share an octet (xor 4, 8, 16), then over the 8 warps through smem
#pragma unroll
  for (int c = 0; c < CO; ++c) {
#pragma unroll
    for (int k = 0; k < 8; ++k) {
      float a = gw[c][k];
      a += __shfl_xor_sync(0xffffffffu, a, 4);
      a += __shfl_xor_sync(0xffffffffu, a, 8);
      a += __shfl_xor_sync(0xffffffffu, a, 16);
      gw[c][k] = a;
    }
    float bsum = gb[c];
    bsum += __shfl_xor_sync(0xffffffffu, bsum, 4);
    bsum += __shfl_xor_sync(0xffffffffu, bsum, 8);
    bsum += __shfl_xor_sync(0xffffffffu, bsum, 16);
    gb[c] = bsum;
  }
  if (lane < 4) {
#pragma unroll
    for (int c = 0; c < CO; ++c) {
#pragma unroll
      for (int k = 0; k < 8; ++k) red[warp][c][lane * 8 + k] = gw[c][k];
      if (lane == 0) red[warp][c][32] = gb[c];   // every octet lane saw the same dout values
    }
  }
  __syncthreads();
  float* pb = part + (size_t)(blockIdx.y * gridDim.x + blockIdx.x) * kC1MaxCo * 33;
  for (int i = threadIdx.x; i < CO * 33; i += blockDim.x) {
    float a = 0.f;
#pragma unroll
    for (int wq = 0; wq < 8; ++wq) a += red[wq][i / 33][i % 33];
    pb[i] = a;
  }
}
// sums the block partials in fp64: dw [co][ci], db [co]. block = (32 lanes over the partials, 4 outputs)
__global__ void conv1x1_bwd_finish_kernel(const float* __restrict__ part, int nblocks, int co, int ci, float* __restrict__ dw,
                                          float* __restrict__ db) {
  const int i = blockIdx.x * blockDim.y + threadIdx.y;
  if (i >= kC1MaxCo * 33) return;
  const int c = i / 33, k = i % 33;
  if (c >= co) return;
  double a = 0.0;
  for (int b = threadIdx.x; b < nblocks; b += 32) a += (double)part[(size_t)b * kC1MaxCo * 33 + i];
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) a += __shfl_xor_sync(0xffffffffu, a, o);
  if (threadIdx.x != 0) return;
  if (k == 32) { if (db) db[c] = (float)a; }
  else if (k < ci && dw) dw[c * ci + k] = (float)a;
}

// ------------------------------------------------------------------------------------------------
// evaluation: DTI scalar maps from the 6 unique tensor components (dxx, dxy, dxz, dyy, dyz, dzz)
//   ref: eval.py:73-116 (do_calc_scalar_maps: np.linalg.eigh per voxel in a Python triple loop)
// One thread per voxel, fp64 cyclic Jacobi on the symmetric 3x3 (converged to machine precision in
// <= 8 sweeps), eigenvalues ascending as LAPACK returns them:
//   AD = l3, RD = (l1 + l2) / 2, MD = mean, FA = sqrt(1.5) * |l - MD| / |l|   (0/0 -> NaN as numpy)
//   azimuth = atan2(v_y, v_x), inclination = acos(v_z / |v|) in degrees, RGB = FA * |v|,  v = principal axis.
// The SIGN of an eigenvector is implementation-defined in LAPACK; here v is oriented with v_z >= 0
// (then v_y >= 0, then v_x >= 0 on ties), so inclination lies in [0, 90].
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ void jacobi_rotate(double (&A)[3][3], double (&V)[3][3], int p, int q) {
  if (A[p][q] == 0.0) return;
  const double theta = (A[q][q] - A[p][p]) / (2.0 * A[p][q]);
  const double t = (theta >= 0.0 ? 1.0 : -1.0) / (fabs(theta) + sqrt(theta * theta + 1.0));
  const double c = 1.0 / sqrt(t * t + 1.0), s_ = t * c;
  const double app = A[p][p], aqq = A[q][q], apq = A[p][q];
  A[p][p] = app - t * apq;
  A[q][q] = aqq + t * apq;
  A[p][q] = A[q][p] = 0.0;
  const int r = 3 - p - q;
  const double arp = A[r][p], arq = A[r][q];
  A[r][p] = A[p][r] = c * arp - s_ * arq;
  A[r][q] = A[q][r] = s_ * arp + c * arq;
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    const double vkp = V[k][p], vkq = V[k][q];
    V[k][p] = c * vkp - s_ * vkq;
    V[k][q] = s_ * vkp + c * vkq;
  }
}

__global__ void dti_scalar_maps_kernel(const float* __restrict__ t6, long long nvox, float* __restrict__ fa,
                                       float* __restrict__ md, float* __restrict__ ad, float* __restrict__ rd,
                                       float* __restrict__ azimuth, float* __restrict__ inclination,
                                       float* __restrict__ rgb) {
  const long long v = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (v >= nvox) return;
  const float* t = t6 + v * 6;
  double A[3][3], V[3][3] = {{1, 0, 0}, {0, 1, 0}, {0, 0, 1}};
  A[0][0] = t[0]; A[0][1] = A[1][0] = t[1]; A[0][2] = A[2][0] = t[2];
  A[1][1] = t[3]; A[1][2] = A[2][1] = t[4]; A[2][2] = t[5];
  for (int sweep = 0; sweep < 8; ++sweep) {
    const double off = fabs(A[0][1]) + fabs(A[0][2]) + fabs(A[1][2]);
    if (off == 0.0) break;
    jacobi_rotate(A, V, 0, 1);
    jacobi_rotate(A, V, 0, 2);
    jacobi_rotate(A, V, 1, 2);
  }
  double l[3] = {A[0][0], A[1][1], A[2][2]};
  int idx[3] = {0, 1, 2};
  // ascending, stable
  if (l[idx[1]] < l[idx[0]]) { const int s_ = idx[0]; idx[0] = idx[1]; idx[1] = s_; }
  if (l[idx[2]] < l[idx[1]]) { const int s_ = idx[1]; idx[1] = idx[2]; idx[2] = s_; }
  if (l[idx[1]] < l[idx[0]]) { const int s_ = idx[0]; idx[0] = idx[1]; idx[1] = s_; }
  const double l1 = l[idx[0]], l2 = l[idx[1]], l3 = l[idx[2]];
  double vx = V[0][idx[2]], vy = V[1][idx[2]], vz = V[2][idx[2]];
  if (vz < 0.0 || (vz == 0.0 && (vy < 0.0 || (vy == 0.0 && vx < 0.0)))) { vx = -vx; vy = -vy; vz = -vz; }
  const double mean = (l1 + l2 + l3) / 3.0;
  const double var = sqrt((l1 - mean) * (l1 - mean) + (l2 - mean) * (l2 - mean) + (l3 - mean) * (l3 - mean));
  const double nrm = sqrt(l1 * l1 + l2 * l2 + l3 * l3);
  const double f = sqrt(1.5) * var / nrm;
  const double r = sqrt(vx * vx + vy * vy + vz * vz);
  const double kDeg = 57.29577951308232087680;
  if (fa) fa[v] = (float)f;
  if (md) md[v] = (float)mean;
  if (ad) ad[v] = (float)l3;
  if (rd) rd[v] = (float)((l1 + l2) * 0.5);
  if (azimuth) azimuth[v] = (float)(kDeg * atan2(vy, vx));
  if (inclination) {
    double cz = vz / r;
    cz = cz > 1.0 ? 1.0 : cz;
    inclination[v] = (float)(kDeg * acos(cz));
  }
  if (rgb) {
    rgb[v * 3 + 0] = (float)(f * fabs(vx));
    rgb[v * 3 + 1] = (float)(f * fabs(vy));
    rgb[v * 3 + 2] = (float)(f * fabs(vz));
  }
}

}  // namespace ub
