// libubssfp.so -- host planners + C ABI (include/ub_api.h) over the sm_100a kernels.
// No torch types cross this boundary; no CPU fallback exists: an unsupported request is an error.
#include <cstdio>
#include <cstdarg>
#include <cstring>
#include <cstdlib>
#include <mutex>
#include <atomic>
#include "../../include/ub_api.h"
#include "igemm_fwd.cuh"
#include "igemm_wgrad.cuh"
#include "igemm_march.cuh"
#include "wgrad_march.cuh"
#include "pointwise.cuh"
#include "head_mma.cuh"
#include "optim_io.cuh"
#include "fp32_path.cuh"

using namespace ub;

// --------------------------------------------------------------------------------------------------
// errors
// --------------------------------------------------------------------------------------------------
static thread_local char g_err[512] = "";
static int fail(int code, const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
  return code;
}
#define UB_CUDA(x)                                                                         \
  do {                                                                                     \
    cudaError_t e_ = (x);                                                                  \
    if (e_ != cudaSuccess) return fail(-3, "%s failed: %s", #x, cudaGetErrorString(e_));   \
  } while (0)
static std::atomic<long long> g_launches{0};
#define UB_LAUNCH_CHECK()                                                                  \
  do {                                                                                     \
    g_launches.fetch_add(1, std::memory_order_relaxed);                                    \
    cudaError_t e_ = cudaGetLastError();                                                   \
    if (e_ != cudaSuccess) return fail(-3, "kernel launch failed: %s", cudaGetErrorString(e_)); \
  } while (0)

// Switches to a reference path (read on every call: tests and tools flip them inside one process)
static bool env_flag(const char* name) {
  const char* v = getenv(name);
  return v && atoi(v) != 0;
}

extern "C" int ub_version(void) { return 100; }
extern "C" const char* ub_last_error(void) { return g_err; }
extern "C" long long ub_launch_count(void) { return g_launches.load(std::memory_order_relaxed); }

// --------------------------------------------------------------------------------------------------
// tensor maps
// --------------------------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static EncodeTiledFn g_encode = nullptr;
static std::once_flag g_encode_once;
static int ensure_encode() {
  std::call_once(g_encode_once, [] {
    cudaDriverEntryPointQueryResult q;
    void* fn = nullptr;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &q) == cudaSuccess)
      g_encode = (EncodeTiledFn)fn;
  });
  if (!g_encode) return fail(-3, "cuTensorMapEncodeTiled unavailable (no CUDA driver / no GPU)");
  // cuTensorMapEncodeTiled is a DRIVER call: it needs a context current on the calling thread. A host thread that
  // has not issued a runtime call yet (a user's worker thread) has none: bind the primary context once per thread.
  static thread_local bool ctx_bound = false;
  if (!ctx_bound) {
    cudaError_t e = cudaFree(0);
    if (e != cudaSuccess) return fail(-3, "no CUDA context on this thread: %s", cudaGetErrorString(e));
    ctx_bound = true;
  }
  return 0;
}
static CUtensorMapSwizzle swz_for_bytes(int b) {
  return b == 128 ? CU_TENSOR_MAP_SWIZZLE_128B : b == 64 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_32B;
}
// NDHWC bf16 activation: dims (C, W, H, D, N); box (box_c, bw*es, bh*es, 1, 1); element stride es on w,h
static int make_act_map(CUtensorMap* m, const void* ptr, int cp, int W, int H, int D, int N, int box_c, int bw,
                        int bh, int es, int bd = 1) {
  cuuint64_t gd[5] = {(cuuint64_t)cp, (cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)D, (cuuint64_t)N};
  cuuint64_t gs[4] = {(cuuint64_t)cp * 2, (cuuint64_t)W * cp * 2, (cuuint64_t)H * W * cp * 2,
                      (cuuint64_t)D * H * W * cp * 2};
  cuuint32_t bx[5] = {(cuuint32_t)box_c, (cuuint32_t)(bw * es), (cuuint32_t)(bh * es), (cuuint32_t)(bd > 1 ? bd * es : 1), 1};
  cuuint32_t st[5] = {1, (cuuint32_t)es, (cuuint32_t)es, (cuuint32_t)(bd > 1 ? es : 1), 1};
  CUresult r = g_encode(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 5, const_cast<void*>(ptr), gd, gs, bx, st,
                        CU_TENSOR_MAP_INTERLEAVE_NONE, swz_for_bytes(box_c * 2), CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                        CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  return r == CUDA_SUCCESS ? 0 : fail(-3, "cuTensorMapEncodeTiled(act) failed: %d", (int)r);
}
// packed weights [rows][K] bf16: dims (K, rows); box (kc, nt)
static int make_w_map(CUtensorMap* m, const void* ptr, long long K, long long rows, int kc, int nt) {
  cuuint64_t gd[2] = {(cuuint64_t)K, (cuuint64_t)rows};
  cuuint64_t gs[1] = {(cuuint64_t)K * 2};
  cuuint32_t bx[2] = {(cuuint32_t)kc, (cuuint32_t)nt};
  cuuint32_t st[2] = {1, 1};
  CUresult r = g_encode(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(ptr), gd, gs, bx, st,
                        CU_TENSOR_MAP_INTERLEAVE_NONE, swz_for_bytes(kc * 2), CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                        CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  return r == CUDA_SUCCESS ? 0 : fail(-3, "cuTensorMapEncodeTiled(weights) failed: %d", (int)r);
}

// --------------------------------------------------------------------------------------------------
// descriptor helpers
// --------------------------------------------------------------------------------------------------
static inline bool is_k4(int kind) { return kind == UB_CONV_K4S2P1 || kind == UB_CONV_K4S2P1_S2D; }
static int check_desc(const ub_conv_desc* d) {
  if (!d) return fail(-1, "null conv desc");
  if (d->kind < 0 || d->kind > 4) return fail(-1, "bad conv kind %d", d->kind);
  if (d->n <= 0 || d->d <= 0 || d->h <= 0 || d->w <= 0) return fail(-1, "bad conv dims");
  if (d->c0p <= 0 || d->c0p % 32 || d->c1p % 32 || d->cop <= 0 || d->cop % 32)
    return fail(-1, "padded channel counts must be positive multiples of 32 (c0p=%d c1p=%d cop=%d)", d->c0p, d->c1p,
                d->cop);
  if (d->c0 > d->c0p || d->c1 > d->c1p || d->co > d->cop) return fail(-1, "real channels exceed padded channels");
  if (is_k4(d->kind) && ((d->d | d->h | d->w) & 1)) return fail(-1, "k4s2p1 needs even input dims");
  if (d->kind == UB_CONV_K4S2P1_S2D && d->c1p) return fail(-1, "the space-to-depth stem takes one source");
  if (d->kind == UB_DECONV_K2S2 && d->c1p) return fail(-1, "transposed conv takes one source");
  if (d->cop > 128 && d->cop % 128) return fail(-1, "cop > 128 must be a multiple of 128");
  return 0;
}
static int ntaps_of(int kind) { return kind == UB_CONV_K3S1P1 ? 27 : kind == UB_CONV_K1 ? 1 : is_k4(kind) ? 64 : 8; }
static void out_dims(const ub_conv_desc* d, int* od, int* oh, int* ow) {
  if (is_k4(d->kind)) { *od = d->d / 2; *oh = d->h / 2; *ow = d->w / 2; }
  else if (d->kind == UB_DECONV_K2S2) { *od = d->d * 2; *oh = d->h * 2; *ow = d->w * 2; }
  else { *od = d->d; *oh = d->h; *ow = d->w; }
}
static inline int align_up(int x, int a) { return (x + a - 1) / a * a; }
static inline int cdiv(int a, int b) { return (a + b - 1) / b; }
static int next_pow2_cols(int c) { int p = 32; while (p < c) p <<= 1; return p; }

// The marching-plane kernel (igemm_march.cuh) serves the 3x3x3 convs whose GEMM N is 32:
//   forward with cop == 32 (K = c0p + c1p <= 96), dgrad with a single 32-channel source (K = cop <= 96).
static bool use_march(const ub_conv_desc* d, int dir) {
  if (d->kind != UB_CONV_K3S1P1) return false;
  if (dir == 0) return d->cop == 32 && d->c0p + d->c1p <= 96;
  return d->c1p == 0 && d->c0p == 32 && d->cop <= 96;
}

// Depth-tap folding in the generic kernel (igemm_fwd.cuh, kd_fold): 3x3x3 layers whose GEMM N is a
// single tile (<= 128 columns) and that are not served by the marching kernel. Returns the fold
// factor (depth taps per UMMA, N = factor * nt <= 256) or 0.
static int use_kd_fold(const ub_conv_desc* d, int dir) {
  if (d->kind != UB_CONV_K3S1P1 || use_march(d, dir)) return 0;
  const int nt = dir == 0 ? d->cop : d->c0p + d->c1p;
  if (nt > 128) return 0;
  const int f = 256 / nt;
  return f > 3 ? 3 : f;
}

extern "C" long long ub_packed_weight_elems(const ub_conv_desc* d, int dir) {
  if (check_desc(d)) return -1;
  const long long cin = d->c0p + d->c1p;
  (void)dir;
  return (long long)ntaps_of(d->kind) * d->cop * cin;
}

extern "C" int ub_conv_deferred_src0_ok(const ub_conv_desc* d);
// dir: bit 0 = direction (0 forward, 1 dgrad); UB_PACK_F16_SRC0: the K columns of source 0 are packed as fp16
// (forward packs of convs whose source 0 is a deferred activation evaluated as an fp16 operand)
static int build_pack_args(const ub_conv_desc* d, int dir_flags, WeightPackArgs* out) {
  const int dir = dir_flags & 1;
  if (dir_flags & ~(1 | UB_PACK_F16_SRC0)) return fail(-1, "bad weight pack direction / flags %d", dir_flags);
  if ((dir_flags & UB_PACK_F16_SRC0) && (dir != 0 || ub_conv_deferred_src0_ok(d) != 1))
    return fail(-2, "UB_PACK_F16_SRC0 applies to the forward pack of a conv that accepts a deferred source 0");
  const int nt = ntaps_of(d->kind);
  const int ci = d->c0 + d->c1;
  WeightPackArgs& A = *out;
  memset(&A, 0, sizeof(A));
  A.nblocks = nt;
  const bool deconv = d->kind == UB_DECONV_K2S2;
  // source strides of (co, ci, tap)
  const long long s_co = deconv ? nt : (long long)ci * nt;
  const long long s_ci = deconv ? (long long)d->co * nt : nt;
  if (dir == 0) {  // rows = co, cols = ci
    A.rows = d->co; A.rows_pad = d->cop; A.cols = ci; A.cols_pad = d->c0p + d->c1p;
    A.stride_row = s_co; A.stride_col = s_ci;
    for (int t = 0; t < nt; ++t) A.tapmap[t] = t;
  } else {         // rows = ci, cols = co ; 3x3x3 dgrad correlates with the flipped filter
    A.rows = ci; A.rows_pad = d->c0p + d->c1p; A.cols = d->co; A.cols_pad = d->cop;
    A.stride_row = s_ci; A.stride_col = s_co;
    for (int t = 0; t < nt; ++t) A.tapmap[t] = d->kind == UB_CONV_K3S1P1 ? nt - 1 - t : t;
  }
  A.src_tap_stride = 1;
  if (use_march(d, dir)) {
    // [kh*3+kw][kd*32 + n][K]: the depth taps are folded into the GEMM N dimension
    A.nblocks = 9;
    A.rows_fold = 32;
    A.rows_pad = 96;
    A.fold_tap_stride = dir == 0 ? 9 : -9;
    for (int t = 0; t < 9; ++t) A.tapmap[t] = dir == 0 ? t : 26 - t;
  }
  if (use_kd_fold(d, dir)) {
    // [kh*3+kw][(2 - kd) * rows_pad + n][K]
    A.nblocks = 9;
    A.rows_fold = A.rows_pad;
    A.rows_pad = 3 * A.rows_pad;
    A.fold_tap_stride = dir == 0 ? -9 : 9;
    for (int t = 0; t < 9; ++t) A.tapmap[t] = dir == 0 ? 18 + t : 8 - t;
  }
  // concat split: padded index -> real channel (source 1 starts at c0p in padded space, c0 in real space)
  A.split_pad = d->c1p ? d->c0p : 0;
  A.split_real = d->c1p ? d->c0 : 0;
  A.split_on_rows = dir == 1;
  A.f16_cols = (dir_flags & UB_PACK_F16_SRC0) ? d->c0p : 0;
  return 0;
}

extern "C" int ub_pack_conv_weights(const ub_conv_desc* d, int dir, const float* w, void* packed, void* stream) {
  if (int e = check_desc(d)) return e;
  if (!w || !packed) return fail(-1, "null weight pointer");
  WeightPackArgs A;
  if (int e = build_pack_args(d, dir, &A)) return e;
  const long long total = (long long)A.nblocks * A.rows_pad * A.cols_pad;
  pack_weights_kernel<<<(unsigned)((total + 255) / 256), 256, 0, (cudaStream_t)stream>>>(
      w, reinterpret_cast<__nv_bfloat16*>(packed), A);
  UB_LAUNCH_CHECK();
  return 0;
}

extern "C" int ub_pack_conv_weights_multi(const ub_weight_pack_item* items, int count, void* stream) {
  if (count < 0 || (count > 0 && !items)) return fail(-1, "bad arguments to ub_pack_conv_weights_multi");
  static WeightPackBatch B;            // 11 KB table: built under a lock, copied into the launch by value
  static std::mutex mu;
  std::lock_guard<std::mutex> lock(mu);
  int i = 0;
  while (i < count) {
    B.count = 0;
    B.block_begin[0] = 0;
    while (i < count && B.count < kPackMaxTensors) {
      const ub_weight_pack_item& it = items[i++];
      if (int e = check_desc(&it.desc)) return e;
      if (!it.w || !it.packed) return fail(-1, "ub_pack_conv_weights_multi: item %d has a null pointer", i - 1);
      const int k = B.count++;
      if (int e = build_pack_args(&it.desc, it.dir, &B.a[k])) return e;
      B.w[k] = it.w;
      B.out[k] = reinterpret_cast<__nv_bfloat16*>(it.packed);
      const long long plane = (long long)B.a[k].rows_pad * B.a[k].cols_pad;      // one thread per (row, column)
      B.block_begin[k + 1] = B.block_begin[k] + (int)((plane + 255) / 256);
    }
    if (B.count == 0) break;
    pack_weights_multi_kernel<<<(unsigned)B.block_begin[B.count], 256, 0, (cudaStream_t)stream>>>(B);
    UB_LAUNCH_CHECK();
  }
  return 0;
}

// --------------------------------------------------------------------------------------------------
// igemm launch plumbing
// --------------------------------------------------------------------------------------------------
static const int kSmemBudget = 220 * 1024;

struct IgemmPlan {
  IgemmParams P;
  dim3 grid;
  int smem;
};

// Per-device state: the SM count and the "large dynamic shared memory" opt-in of every kernel are properties of
// the CURRENT device (one process may drive several GPUs), so both are cached per device ordinal.
static const int kMaxDevices = 64;
static int current_device() {
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= kMaxDevices) dev = 0;
  return dev;
}
static int sm_count() {
  static std::atomic<int> n[kMaxDevices];
  const int dev = current_device();
  int v = n[dev].load(std::memory_order_relaxed);
  if (v == 0) {
    if (cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || v <= 0) v = 148;
    n[dev].store(v, std::memory_order_relaxed);
  }
  return v;
}
// cudaFuncAttributeMaxDynamicSharedMemorySize of `fn` on the current device, once per (kernel, device)
struct SmemOptIn {
  std::atomic<unsigned long long> done{0};
};
static int opt_in_smem(SmemOptIn& st, const void* fn, const char* what) {
  const int dev = current_device();
  if (st.done.load(std::memory_order_acquire) & (1ull << dev)) return 0;
  cudaError_t e = cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
  if (e != cudaSuccess) return fail(-3, "cudaFuncSetAttribute(%s): %s", what, cudaGetErrorString(e));
  st.done.fetch_or(1ull << dev, std::memory_order_release);
  return 0;
}

// K chunks of the generic kernel are kIgemmKc = 32 channels. 64-channel chunks (128-byte rows, half the TMA rows) were
// measured on the transposed convs (profiles/r02j_kc64_ab.txt): 64 -> 64 forward 0.496 -> 0.507 ms (bound by its 2.1 GB
// of output stores, not by the loads), 128 -> 64 0.083 -> 0.078, dgrads equal or slower (one-plane tiles); removed.

// Planes per activation TMA box of the generic kernel: all the planes of a tile in ONE box (the producer thread's
// issue rate bounds the launches with little MMA work per box). One box per plane for every shape was measured
// (profiles/r02i_producer_ab.txt) and removed; it remains for the shapes rejected here.
static int plane_box(const IgemmParams& P) {
  if (P.n_in_planes <= 1 || P.n_in_planes * P.in_stride > 256) return 1;
  // several A tiles per stage: every tile's box must start on a 128-byte boundary
  if (P.n_atiles > 1 && (P.n_in_planes * P.bh * P.bw * kIgemmKc * 2) % 128 != 0) return 1;
  return P.n_in_planes;
}

// Fill the smem plan / grid once the geometry fields of P are set. nt_max = widest N tile.
// The kernel is persistent with one CTA per SM: the whole shared memory goes to the TMA rings.
static int finish_plan(IgemmPlan* pl, int nt_max) {
  IgemmParams& P = pl->P;
  const int pitch = kIgemmKc * 2;
  P.box_planes = plane_box(P);
  // a multi-plane box writes its planes back to back; the swizzle is a function of the absolute shared-memory address
  // (tools/probe_umma.cu), so a plane may start at any multiple of 128 bytes
  P.plane_stride = P.box_planes > 1 ? P.bh * P.bw * pitch : align_up(P.bh * P.bw * pitch, 1024);
  P.a_stage_bytes = align_up(P.n_atiles * P.n_in_planes * P.plane_stride, 1024);
  P.b_stage_bytes = align_up((P.kd_fold ? P.fold_nd : 1) * nt_max * pitch, 1024);
  const int misc = 8 * 80 + 64 + kFwdRedFloats * 4 + 1024;
  // A stages: two (the next chunk / next tile loads while this one is multiplied) when they fit.
  // B ring: as deep as the remaining budget allows (<= 16): a weight tile is consumed in td*2 MMAs,
  // far faster than one TMA round trip, so the ring must cover ~2k cycles of latency.
  // Layers with few taps per K chunk (the space-to-depth stem: 4) consume an A stage faster than one TMA
  // round trip: give them up to four stages.
  P.nsa = P.ntaps * P.td <= 32 ? 4 : 2;
  while (P.nsa > 1 && P.nsa * P.a_stage_bytes + 4 * P.b_stage_bytes + misc > kSmemBudget) --P.nsa;
  P.nsb = (kSmemBudget - P.nsa * P.a_stage_bytes - misc) / P.b_stage_bytes;
  if (P.nsb > 16) P.nsb = 16;
  if (P.nsb < 2) return fail(-2, "igemm smem plan: no room for the weight ring");
  pl->smem = P.nsa * P.a_stage_bytes + P.nsb * P.b_stage_bytes + misc;
  if (pl->smem > 227 * 1024) return fail(-2, "igemm smem plan too large: %d bytes", pl->smem);
  if (pl->smem < 120 * 1024) pl->smem = 120 * 1024;   // never two CTAs on one SM (persistent: one per SM)
  const int set_cols = P.td * align_up(nt_max, 32);
  if (set_cols > 512) return fail(-2, "igemm TMEM plan too large: %d columns", set_cols);
  // Two accumulator sets: the epilogue of a tile overlaps the next tile's MMAs. Four sets were measured on the
  // narrow-tile launches (1x1x1 head, stem forward / dgrad, d2: <= 128 columns per set) and changed nothing
  // (profiles/r02g_nacc.txt; removed) -- those launches are bound by the epilogue's per-tile instruction count
  // (statistics transpose) or the MMA thread's issue rate, not by the hand-off depth.
  P.nacc = 512 / set_cols;
  if (P.nacc > kMaxAccSets) P.nacc = kMaxAccSets;
  if (P.nacc < 1) P.nacc = 1;
  P.tmem_cols = next_pow2_cols(P.nacc * set_cols);
  P.tiles_w = cdiv(P.Wo, 8);
  P.tiles_h = cdiv(P.Ho, 16);
  P.tiles_d = cdiv(P.Do, P.td);
  P.total_tiles = P.Nb * P.tiles_d * P.tiles_h * P.tiles_w;
  int gx = sm_count() / P.n_ntiles;
  if (gx < 1) gx = 1;
  if (gx > P.total_tiles) gx = P.total_tiles;
  pl->grid = dim3((unsigned)gx, (unsigned)P.n_ntiles, 1);
  return 0;
}

static int launch_igemm(const IgemmPlan& pl, cudaStream_t st) {
  // Instantiations by statistics: with them (forward convs in front of a norm: 64 accumulator registers per epilogue
  // thread) and without. Measured (profiles/r02g_epi16.txt): dropping the statistics code alone takes the transposed
  // conv 64 -> 64 from 0.568 to 0.503 ms and the stem dgrad from 0.69 to 0.64 ms (120 instead of 168 registers);
  // sixteen epilogue warps add little there (0.486) and cost elsewhere (32 -> 96-column dgrad 2.39 -> 2.47 ms, stem
  // dgrad 0.70): measured, removed.
  // Two issuing warps that split the PLANES of a tile (kMma = 2, independent accumulators). Measured per shape
  // (profiles/r02j_fwd_mma_planes.txt): the four-plane tiles with three depth taps per UMMA -- the 64-channel 3x3x3
  // layers -- gain 6-9 % (64 -> 64 @64^3 forward 0.365 -> 0.341 ms, dgrad 0.357 -> 0.325, 64+64 -> 64 0.679 -> 0.640,
  // 32 -> 64 0.210 -> 0.195); two-plane tiles (128 channels, the 96-column dgrad) do not move, the stem, the transposed
  // convs, the 1x1x1 head and the 8^3 level lose 2-20 %. So: that schedule only (the other choices measured, removed).
  const int stats = pl.P.stats != nullptr ? 1 : 0;
  const int mma2 = pl.P.kd_fold == 3 && pl.P.fold_nd == 3 && pl.P.td == 4 ? 1 : 0;
  typedef void (*IgemmFn)(const IgemmParams);
  static const IgemmFn fns[2][2] = {{igemm_fwd_kernel<false, 1>, igemm_fwd_kernel<false, 2>},
                                    {igemm_fwd_kernel<true, 1>, igemm_fwd_kernel<true, 2>}};
  static SmemOptIn opt[2][2];
  const IgemmFn fn = fns[stats][mma2];
  if (int e = opt_in_smem(opt[stats][mma2], (const void*)fn, "igemm_fwd")) return e;
  fn<<<pl.grid, (kFwdEpiWarps + 3 + mma2) * 32, pl.smem, st>>>(pl.P);
  UB_LAUNCH_CHECK();
  return 0;
}

// Map the output columns onto N tiles of <= 128. Two destinations (dgrad of a skip-concat conv:
// columns [0,n0p) -> dst0, [n0p, n0p+n1p) -> dst1) share one tile when they fit in 128 columns.
static void make_ntiles(IgemmParams& P, int n0p, void* dst0, int n1p, void* dst1) {
  P.n_ntiles = 0;
  if (n1p && n0p + n1p <= 128) {
    IgemmNTile& T = P.ntile[P.n_ntiles++];
    T.n0 = 0; T.nt = n0p + n1p; T.out = dst0; T.out_cpitch = n0p; T.out_coff = 0;
    T.split = n0p; T.out2 = dst1; T.out2_cpitch = n1p;
    return;
  }
  for (int s = 0; s < 2; ++s) {
    const int np = s ? n1p : n0p;
    void* dst = s ? dst1 : dst0;
    for (int c = 0; c < np; c += 128) {
      IgemmNTile& T = P.ntile[P.n_ntiles++];
      T.n0 = (s ? n0p : 0) + c;
      T.nt = np - c < 128 ? np - c : 128;
      T.out = dst;
      T.out_cpitch = np;
      T.out_coff = c;
      T.split = T.nt; T.out2 = dst; T.out2_cpitch = np;
    }
  }
}

static void march_geometry(int n, int D, int H, int W, int* tiles_w, int* tiles_h, int* nseg, int* seg_len) {
  *tiles_w = cdiv(W, 8);
  *tiles_h = cdiv(H, 16);
  const int columns = n * *tiles_h * *tiles_w;
  int ns = cdiv(4 * sm_count(), columns);
  const int max_seg = D / 8 > 1 ? D / 8 : 1;
  if (ns > max_seg) ns = max_seg;
  if (ns < 1) ns = 1;
  *seg_len = cdiv(D, ns);
  *nseg = cdiv(D, *seg_len);
}

// 15-bit keep threshold round(p * 32768), replicated into both 16-bit lanes (pointwise.cuh: dropout_maskw)
static uint32_t drop_thresh(float p) {
  uint32_t t = (uint32_t)(p * 32768.0f + 0.5f);
  if (t > 32767u) t = 32767u;
  return t * 0x00010001u;
}

static int fill_deferred(NormActArgs* A, const ub_deferred_act* tf) {
  if (!tf->scale || !tf->shift) return fail(-1, "ub_deferred_act needs scale and shift");
  if (tf->drop_p < 0.f || tf->drop_p >= 1.f) return fail(-1, "dropout p out of range");
  A->scale = tf->scale; A->shift = tf->shift; A->slope = tf->slope; A->drop_p = tf->drop_p;
  A->drop_seed = tf->drop_seed; A->drop_thresh = drop_thresh(tf->drop_p);
  return 0;
}

static int launch_march(const void* src0, int c0p, const void* src1, int c1p, int n, int D, int H, int W,
                        const void* w_packed, const float* bias, int bias_n, void* out, float* stats,
                        const ub_norm_bwd_fuse* fuse, const ub_deferred_act* tf, int src0_f16, cudaStream_t st) {
  MarchParams P;
  memset(&P, 0, sizeof(P));
  P.src0_f16 = src0_f16 ? 1 : 0;
  if (tf) {
    if (fuse) return fail(-1, "a deferred source and the norm-backward fusion are exclusive");
    if (c0p != 32) return fail(-2, "a deferred activation source must have 32 padded channels (got %d)", c0p);
    if (int e = fill_deferred(&P.tf, tf)) return e;
    P.tf_f16 = tf->f16_operand ? 1 : 0;
  }
  if (fuse) {
    if (!fuse->y || !fuse->scale || !fuse->shift || !fuse->mean || !fuse->rstd || !fuse->partial)
      return fail(-1, "incomplete ub_norm_bwd_fuse");
    if (fuse->drop_p < 0.f || fuse->drop_p >= 1.f) return fail(-1, "dropout p out of range");
    P.nb_y = fuse->y; P.nb_scale = fuse->scale; P.nb_shift = fuse->shift; P.nb_mean = fuse->mean; P.nb_rstd = fuse->rstd;
    P.nb_slope = fuse->slope; P.nb_drop_p = fuse->drop_p; P.nb_drop_seed = fuse->drop_seed;
    P.nb_drop_thresh = drop_thresh(fuse->drop_p);
    stats = fuse->partial;
  }
  P.n_chunks_src0 = c0p / 32;
  P.n_chunks_total = (c0p + c1p) / 32;
  P.Nb = n; P.D = D; P.H = H; P.W = W;
  march_geometry(n, D, H, W, &P.tiles_w, &P.tiles_h, &P.nseg, &P.seg_len);
  P.out = out; P.bias = bias; P.bias_n = bias_n; P.stats = stats;
  // CTA pairs (cta_group::2) whenever the w tiles pair up and a plane has >= 2 K chunks (a plane must be long enough to
  // amortise the cross-CTA barrier traffic: measured on B200 at 8x128^3, 1 K chunk 805 vs 1200 TFLOP/s single-CTA,
  // 2 chunks 1374 vs 1330, 3 chunks 1576 vs 1360)
  const bool pair = (P.tiles_w % 2 == 0) && P.n_chunks_total >= 2;
  const int wbytes = P.n_chunks_total * 9 * (pair ? kMarchWTileBytes / 2 : kMarchWTileBytes);
  const int misc = 8 * 48 + 64 + (kMarchEpiWarps * 2 * 32 + 32 + 128) * 4 + 64 + 1024;
  P.nsa = (220 * 1024 - wbytes - misc) / kMarchPlaneBytes;
  if (P.nsa > 8) P.nsa = 8;
  if (P.nsa < 2) return fail(-2, "march smem plan: no room for the plane ring");
  const int smem = wbytes + P.nsa * kMarchPlaneBytes + misc;
  if (int e = make_act_map(&P.tm_src[0], src0, c0p, W, H, D, n, 32, 10, 18, 1)) return e;
  if (c1p)
    if (int e = make_act_map(&P.tm_src[1], src1, c1p, W, H, D, n, 32, 10, 18, 1)) return e;
  if (int e = make_w_map(&P.tm_w, w_packed, c0p + c1p, 9 * 96, 32, pair ? 48 : 96)) return e;
  // instantiation: [fuse | tf][pair]
  typedef void (*MarchFn)(const MarchParams);
  static const MarchFn fns[3][2] = {
      {igemm_march_kernel<false, false, false>, igemm_march_kernel<false, true, false>},
      {igemm_march_kernel<true, false, false>, igemm_march_kernel<true, true, false>},
      {igemm_march_kernel<false, false, true>, igemm_march_kernel<false, true, true>}};
  static SmemOptIn opt[3][2];
  const int variant = fuse ? 1 : (tf ? 2 : 0);
  MarchFn fn = fns[variant][pair ? 1 : 0];
  if (int e = opt_in_smem(opt[variant][pair ? 1 : 0], (const void*)fn, "igemm_march")) return e;
  const unsigned grid = (unsigned)(n * P.tiles_h * P.tiles_w * P.nseg);
  const unsigned threads = tf ? kMarchThreadsTf : kMarchThreads2;
  if (pair) {
    // cluster of two CTAs along x: blocks (2k, 2k+1) take the w tiles (2j, 2j+1) of one column pair
    cudaLaunchConfig_t cfg;
    memset(&cfg, 0, sizeof(cfg));
    cfg.gridDim = dim3(grid, 1, 1);
    cfg.blockDim = dim3(threads, 1, 1);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = 2; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    cudaError_t le = cudaLaunchKernelEx(&cfg, fn, P);
    if (le != cudaSuccess) return fail(-3, "cluster launch of igemm_march failed: %s", cudaGetErrorString(le));
  } else {
    fn<<<grid, threads, smem, st>>>(P);
  }
  UB_LAUNCH_CHECK();
  return 0;
}

// per-axis decomposition of the k=4,s=2,p=1 filter index: input i = 2*o - 1 + k
//   k -> (parity of i, shift inside the parity tile whose origin offset is (parity ? -1 : 0))
static inline int k4_parity(int k) { return (k & 1) ? 0 : 1; }
static inline int k4_shift(int k) { return k >> 1; }

// Planes per tile of the generic 3x3x3 / 1x1x1 kernel. Four planes amortise the depth halo and the weight stream
// best, but with an N tile of nt columns they need 4 * nt TMEM columns per accumulator set: above 256 the
// accumulators cannot be double-buffered and the epilogue of every tile is exposed. Measured on B200 (8 x 128^3
// step shapes, profiles/r01w_td2.txt): two-plane tiles (double-buffered) win whenever the layer has ONE N tile --
// 128 -> 128 @32^3 forward 0.194 -> 0.153 ms, 128+128 -> 128 0.352 -> 0.290, the 32 -> 96-column dgrad of
// upcat_1.conv_0 2.50 -> 2.42 -- and lose with several N tiles, where every tile re-streams the weights of its N
// tile (256 -> 256 @16^3 0.103 -> 0.124), except at the 8^3 level, where they double the number of tiles of an
// underfilled grid (512 -> 512 @8^3 0.177 -> 0.120).
static int planes_per_tile(int depth, int nt_max, int n_ntiles) {
  int td = depth < 4 ? depth : 4;
  const int cols = (nt_max + 31) / 32 * 32;
  if (td == 4 && 2 * 4 * cols > 512 && 2 * 2 * cols <= 512 && (n_ntiles == 1 || depth <= 8)) td = 2;
  return td;
}

extern "C" int ub_conv_num_tiles(const ub_conv_desc* d) {
  if (check_desc(d)) return -1;
  int od, oh, ow;
  out_dims(d, &od, &oh, &ow);
  if (use_march(d, 0)) {
    int tw, th, ns, sl;
    march_geometry(d->n, d->d, d->h, d->w, &tw, &th, &ns, &sl);
    return d->n * th * tw * ns;
  }
  int td = 4;
  int Dt = od, Ht = oh, Wt = ow;
  if (d->kind == UB_CONV_K3S1P1 || d->kind == UB_CONV_K1)
    td = planes_per_tile(d->d, d->cop < 128 ? d->cop : 128, cdiv(d->cop, 128));
  if (d->kind == UB_CONV_K4S2P1) td = 1;
  if (d->kind == UB_DECONV_K2S2) { Dt = d->d; Ht = d->h; Wt = d->w; }
  if (td > Dt) td = Dt;
  return d->n * cdiv(Dt, td) * cdiv(Ht, 16) * cdiv(Wt, 8);
}

// A deferred source 0 is served where BOTH consumers of the activations -- the forward conv and its weight
// gradient -- run on the marching kernels: 3x3x3, 32 output channels, one 32-channel source 0, planes >= 16 x 8.
static bool use_wgrad_march(const ub_conv_desc* d);
extern "C" int ub_conv_deferred_src0_ok(const ub_conv_desc* d) {
  if (check_desc(d)) return -1;
  return (use_march(d, 0) && d->c0p == 32 && use_wgrad_march(d)) ? 1 : 0;
}

extern "C" int ub_conv_fwd(const ub_conv_desc* d, const void* src0, const void* src1, const void* w_packed,
                           const float* bias, int act, float slope, void* out, float* stats_partial,
                           const ub_deferred_act* src0_act, int src0_f16, void* stream) {
  if (int e = check_desc(d)) return e;
  if ((src0_act || src0_f16) && ub_conv_deferred_src0_ok(d) != 1)
    return fail(-2, "a deferred / fp16 source 0 is not supported for this convolution (ub_conv_deferred_src0_ok)");
  if (src0_act && src0_f16) return fail(-1, "src0_f16 describes a materialised fp16 tensor: exclusive with src0_act");
  if (int e = ensure_encode()) return e;
  if (!src0 || !w_packed || !out) return fail(-1, "null pointer in ub_conv_fwd");
  if (d->c1p && !src1) return fail(-1, "second source missing");
  cudaStream_t st = (cudaStream_t)stream;
  int od, oh, ow;
  out_dims(d, &od, &oh, &ow);
  const int ktot = d->c0p + d->c1p;
  const int ntaps = ntaps_of(d->kind);
  if (use_march(d, 0)) {
    if (act) return fail(-2, "fused activation is not available on the marching conv path");
    return launch_march(src0, d->c0p, src1, d->c1p, d->n, d->d, d->h, d->w, w_packed, bias, d->co, out,
                        stats_partial, nullptr, src0_act, src0_f16, st);
  }

  IgemmPlan pl;
  memset(&pl, 0, sizeof(pl));
  IgemmParams& P = pl.P;
  P.n_chunks_src0 = d->c0p / kIgemmKc;
  P.n_chunks_total = ktot / kIgemmKc;
  P.w_rows_per_block = d->cop;
  P.Nb = d->n;
  P.bias = bias;
  P.bias_n = d->co;
  P.act = act;
  P.act_slope = slope;
  P.stats = stats_partial;
  P.oD = od; P.oH = oh; P.oW = ow;
  P.out_s = 1;
  make_ntiles(P, d->cop, out, 0, nullptr);
  const int nt_max = d->cop < 128 ? d->cop : 128;
  P.kd_fold = use_kd_fold(d, 0);
  P.fold_nd = 3;
  P.fold_row_step = nt_max;
  P.b_block_rows = P.kd_fold ? 3 * d->cop : d->cop;
  if (int e = make_w_map(&P.tm_w, w_packed, ktot, (long long)ntaps * d->cop, kIgemmKc, nt_max)) return e;

  if (d->kind == UB_CONV_K3S1P1 || d->kind == UB_CONV_K1) {
    const int k = d->kind == UB_CONV_K3S1P1 ? 3 : 1;
    P.td = planes_per_tile(d->d, nt_max, P.n_ntiles);
    P.Do = od; P.Ho = oh; P.Wo = ow;
    P.n_atiles = 1; P.bw = 8 + k - 1; P.bh = 16 + k - 1; P.n_in_planes = P.td + k - 1; P.in_stride = 1;
    P.atile_off[0][0] = P.atile_off[0][1] = P.atile_off[0][2] = -(k / 2);
    P.ntaps = ntaps;
    int t = 0;
    for (int kd = 0; kd < k; ++kd)
      for (int kh = 0; kh < k; ++kh)
        for (int kw = 0; kw < k; ++kw, ++t)
          P.taps[t] = IgemmTap{0, (uint16_t)(kh * P.bw + kw), (uint16_t)kd, (uint16_t)t};
    if (P.kd_fold) P.ntaps = 9;   // taps 0..8 are (kd = 0, kh, kw): row offsets and weight blocks of the folded pack
    if (int e = make_act_map(&P.tm_src[0], src0, d->c0p, d->w, d->h, d->d, d->n, 32, P.bw, P.bh, 1, plane_box(P))) return e;
    if (d->c1p)
      if (int e = make_act_map(&P.tm_src[1], src1, d->c1p, d->w, d->h, d->d, d->n, 32, P.bw, P.bh, 1, plane_box(P))) return e;
    if (int e = finish_plan(&pl, nt_max)) return e;
    return launch_igemm(pl, st);
  }
  if (d->kind == UB_CONV_K4S2P1_S2D) {
    // source = space-to-depth tensor [n][d/2][h/2][w/2][(pd,ph,pw)][c0p]: chunk group = input parity,
    // per axis parity 0 pairs filter taps k = 1, 3 with q = o, o+1; parity 1 pairs k = 0, 2 with q = o-1, o
    P.td = od < 4 ? od : 4;
    P.Do = od; P.Ho = oh; P.Wo = ow;
    P.n_atiles = 1; P.bw = 9; P.bh = 17; P.n_in_planes = P.td + 1; P.in_stride = 1;
    P.chunks_per_group = d->c0p / 32;
    P.n_chunks_src0 = P.n_chunks_total = 8 * P.chunks_per_group;
    // single N tile of <= 128 columns: fold the two depth shifts of a parity group into one UMMA of
    // N = 2 * nt (input plane p of the tile feeds the output planes p-1 and p); the two depth-tap
    // blocks of a tile are 32 taps apart in the [tap][cop][cin] pack
    const bool fold = d->cop <= 128;
    P.kd_fold = fold ? 2 : 0;
    P.fold_nd = 2;
    P.fold_row_step = -32 * d->cop;
    P.ntaps = fold ? 4 : 8;
    for (int pd = 0; pd < 2; ++pd)
      for (int ph = 0; ph < 2; ++ph)
        for (int pw = 0; pw < 2; ++pw) {
          const int g = (pd * 2 + ph) * 2 + pw;
          P.atile_off[g][0] = pw ? -1 : 0;
          P.atile_off[g][1] = ph ? -1 : 0;
          P.atile_off[g][2] = pd ? -1 : 0;
          int t = 0;
          for (int sd = fold ? 1 : 0; sd < 2; ++sd)     // folded: the table entry names the sd = 1 tap (block j = 0)
            for (int sh = 0; sh < 2; ++sh)
              for (int sw = 0; sw < 2; ++sw, ++t) {
                const int kd = 2 * sd + (1 - pd), kh = 2 * sh + (1 - ph), kw = 2 * sw + (1 - pw);
                P.taps[g * P.ntaps + t] = IgemmTap{0, (uint16_t)(sh * P.bw + sw), (uint16_t)sd, (uint16_t)((kd * 4 + kh) * 4 + kw)};
              }
        }
    if (int e = make_act_map(&P.tm_src[0], src0, d->c0p, d->w / 2, d->h / 2, d->d / 2, d->n * 8, 32, P.bw, P.bh, 1, plane_box(P))) return e;
    if (int e = finish_plan(&pl, nt_max)) return e;
    return launch_igemm(pl, st);
  }
  if (d->kind == UB_CONV_K4S2P1) {
    P.td = 1;
    P.Do = od; P.Ho = oh; P.Wo = ow;
    P.n_atiles = 8; P.bw = 9; P.bh = 17; P.n_in_planes = 2; P.in_stride = 2;
    for (int pd = 0; pd < 2; ++pd)
      for (int ph = 0; ph < 2; ++ph)
        for (int pw = 0; pw < 2; ++pw) {
          const int at = (pd * 2 + ph) * 2 + pw;
          P.atile_off[at][0] = pw ? -1 : 0;
          P.atile_off[at][1] = ph ? -1 : 0;
          P.atile_off[at][2] = pd ? -1 : 0;
        }
    P.ntaps = 64;
    int t = 0;
    for (int kd = 0; kd < 4; ++kd)
      for (int kh = 0; kh < 4; ++kh)
        for (int kw = 0; kw < 4; ++kw, ++t) {
          const int at = (k4_parity(kd) * 2 + k4_parity(kh)) * 2 + k4_parity(kw);
          P.taps[t] = IgemmTap{(uint16_t)at, (uint16_t)(k4_shift(kh) * P.bw + k4_shift(kw)), (uint16_t)k4_shift(kd),
                               (uint16_t)t};
        }
    if (int e = make_act_map(&P.tm_src[0], src0, d->c0p, d->w, d->h, d->d, d->n, 32, P.bw, P.bh, 2, plane_box(P))) return e;
    if (d->c1p)
      if (int e = make_act_map(&P.tm_src[1], src1, d->c1p, d->w, d->h, d->d, d->n, 32, P.bw, P.bh, 2, plane_box(P))) return e;
    if (int e = finish_plan(&pl, nt_max)) return e;
    return launch_igemm(pl, st);
  }
  // UB_DECONV_K2S2 forward: one launch; the 8 output sub-positions are extra N tiles (blockIdx.y), each
  // with its own weight tap and scatter offset (stride 2)
  P.td = d->d < 4 ? d->d : 4;
  P.Do = d->d; P.Ho = d->h; P.Wo = d->w;
  P.n_atiles = 1; P.bw = 8; P.bh = 16; P.n_in_planes = P.td; P.in_stride = 1;
  P.ntaps = 1;
  P.out_s = 2;
  P.taps[0] = IgemmTap{0, 0, 0, 0};
  if (stats_partial) return fail(-1, "statistics are not produced by the transposed conv forward");
  if (d->cop == 64) {
    // 64 output channels: the sub-positions (pd, ph, 0) and (pd, ph, 1) share ONE N tile of 128 columns -- their
    // weight blocks are adjacent in the [sub-position][co][ci] pack and their voxels (2w, 2w+1) adjacent in the
    // output, so columns [64, 128) go to the same tensor one voxel further (the two-destination store of the
    // skip-concat dgrad). Four CTAs instead of eight read each input tile (the launch was bound by L2 traffic: 8 x
    // re-read of the input, profiles/r02b_deconv64_ncu_summary.txt), every UMMA is N = 128 and a lane pair writes
    // 256 contiguous bytes. Two planes per tile keep the 2 x 128-column accumulators double-buffered.
    P.td = d->d < 2 ? d->d : 2;
    P.n_in_planes = P.td;
    P.bias_wrap = 64;
    P.n_ntiles = 4;
    for (int sp2 = 0; sp2 < 4; ++sp2) {
      IgemmNTile& T = P.ntile[sp2];
      memset(&T, 0, sizeof(T));
      T.n0 = 0; T.nt = 128; T.out = out; T.out_cpitch = 64; T.out_coff = 0;
      T.split = 64; T.out2 = reinterpret_cast<__nv_bfloat16*>(out) + 64; T.out2_cpitch = 64;
      T.wblock_add = 2 * sp2;
      T.out_p[0] = 0; T.out_p[1] = sp2 & 1; T.out_p[2] = (sp2 >> 1) & 1;
    }
    if (int e = make_w_map(&P.tm_w, w_packed, ktot, (long long)ntaps * d->cop, kIgemmKc, 128)) return e;
    if (int e = make_act_map(&P.tm_src[0], src0, d->c0p, d->w, d->h, d->d, d->n, kIgemmKc, P.bw, P.bh, 1, plane_box(P))) return e;
    if (int e = finish_plan(&pl, 128)) return e;
    return launch_igemm(pl, st);
  }
  {
    const int base_tiles = P.n_ntiles;
    if (base_tiles * 8 > kMaxNTiles) return fail(-2, "transposed conv: too many output channels (%d)", d->cop);
    for (int sp = 1; sp < 8; ++sp)
      for (int i = 0; i < base_tiles; ++i) P.ntile[sp * base_tiles + i] = P.ntile[i];
    for (int sp = 0; sp < 8; ++sp)
      for (int i = 0; i < base_tiles; ++i) {
        IgemmNTile& T = P.ntile[sp * base_tiles + i];
        T.wblock_add = sp;
        T.out_p[0] = sp & 1; T.out_p[1] = (sp >> 1) & 1; T.out_p[2] = (sp >> 2) & 1;
      }
    P.n_ntiles = base_tiles * 8;
  }
  if (int e = make_act_map(&P.tm_src[0], src0, d->c0p, d->w, d->h, d->d, d->n, kIgemmKc, P.bw, P.bh, 1, plane_box(P))) return e;
  if (int e = finish_plan(&pl, nt_max)) return e;
  return launch_igemm(pl, st);
}

extern "C" int ub_conv_dgrad_fuse_records(const ub_conv_desc* d) {
  if (check_desc(d)) return -1;
  if (!use_march(d, 1)) return 0;
  int tw, th, ns, sl;
  march_geometry(d->n, d->d, d->h, d->w, &tw, &th, &ns, &sl);
  return d->n * th * tw * ns;
}

extern "C" int ub_conv_dgrad(const ub_conv_desc* d, const void* dy, const void* w_packed_dgrad, void* dsrc0,
                             void* dsrc1, void* stream) {
  return ub_conv_dgrad_fused(d, dy, w_packed_dgrad, dsrc0, dsrc1, nullptr, stream);
}

extern "C" int ub_conv_dgrad_fused(const ub_conv_desc* d, const void* dy, const void* w_packed_dgrad, void* dsrc0,
                                   void* dsrc1, const ub_norm_bwd_fuse* fuse, void* stream) {
  if (int e = check_desc(d)) return e;
  if (fuse && !use_march(d, 1)) return fail(-2, "fused norm-backward reduction is available on the marching dgrad path only");
  if (int e = ensure_encode()) return e;
  if (!dy || !w_packed_dgrad || !dsrc0) return fail(-1, "null pointer in ub_conv_dgrad");
  if (d->c1p && !dsrc1) return fail(-1, "second gradient destination missing");
  cudaStream_t st = (cudaStream_t)stream;
  int od, oh, ow;
  out_dims(d, &od, &oh, &ow);
  const int ntaps = ntaps_of(d->kind);
  const int ncols = d->c0p + d->c1p;
  if (use_march(d, 1))
    return launch_march(dy, d->cop, nullptr, 0, d->n, d->d, d->h, d->w, w_packed_dgrad, nullptr, 0, dsrc0, nullptr, fuse,
                        nullptr, 0, st);

  IgemmPlan pl;
  memset(&pl, 0, sizeof(pl));
  IgemmParams& P = pl.P;
  P.n_chunks_src0 = d->cop / kIgemmKc;
  P.n_chunks_total = d->cop / kIgemmKc;
  P.w_rows_per_block = ncols;
  P.Nb = d->n;
  P.oD = d->d; P.oH = d->h; P.oW = d->w;
  P.out_s = 1;
  make_ntiles(P, d->c0p, dsrc0, d->c1p, dsrc1);
  int nt_max = 0;
  for (int i = 0; i < P.n_ntiles; ++i) nt_max = P.ntile[i].nt > nt_max ? P.ntile[i].nt : nt_max;
  // N tiles may have different widths; the weight box uses the widest, narrower tiles read extra rows
  // of the following tap block / pad rows (never used by their MMA: idesc N = nt)
  P.kd_fold = use_kd_fold(d, 1);
  P.fold_nd = 3;
  P.fold_row_step = nt_max;
  P.b_block_rows = P.kd_fold ? 3 * ncols : ncols;
  if (int e = make_w_map(&P.tm_w, w_packed_dgrad, d->cop, (long long)ntaps * ncols, kIgemmKc, nt_max)) return e;
  bool uniform = true;
  for (int i = 0; i < P.n_ntiles; ++i) uniform = uniform && P.ntile[i].nt == nt_max;
  if (!uniform) return fail(-2, "dgrad N tiles of unequal width are not supported (c0p=%d c1p=%d)", d->c0p, d->c1p);

  if (d->kind == UB_CONV_K3S1P1 || d->kind == UB_CONV_K1) {
    const int k = d->kind == UB_CONV_K3S1P1 ? 3 : 1;
    P.td = planes_per_tile(d->d, nt_max, P.n_ntiles);
    P.Do = d->d; P.Ho = d->h; P.Wo = d->w;
    P.n_atiles = 1; P.bw = 8 + k - 1; P.bh = 16 + k - 1; P.n_in_planes = P.td + k - 1; P.in_stride = 1;
    P.atile_off[0][0] = P.atile_off[0][1] = P.atile_off[0][2] = -(k / 2);
    P.ntaps = ntaps;
    int t = 0;
    for (int kd = 0; kd < k; ++kd)
      for (int kh = 0; kh < k; ++kh)
        for (int kw = 0; kw < k; ++kw, ++t)
          P.taps[t] = IgemmTap{0, (uint16_t)(kh * P.bw + kw), (uint16_t)kd, (uint16_t)t};
    if (P.kd_fold) P.ntaps = 9;
    if (int e = make_act_map(&P.tm_src[0], dy, d->cop, ow, oh, od, d->n, 32, P.bw, P.bh, 1, plane_box(P))) return e;
    if (int e = finish_plan(&pl, nt_max)) return e;
    return launch_igemm(pl, st);
  }
  if (is_k4(d->kind)) {
    // 8 input parity classes; class p (per axis): p=0 -> taps (o=q-1,k=3),(o=q,k=1); p=1 -> (o=q,k=2),(o=q+1,k=0)
    P.td = od < 4 ? od : 4;
    P.Do = od; P.Ho = oh; P.Wo = ow;  // tile space = q grid (same size as dy)
    P.n_atiles = 1; P.bw = 9; P.bh = 17; P.n_in_planes = P.td + 1; P.in_stride = 1;
    // One N tile per class of <= 128 columns: fold the two depth shifts of a class into one UMMA of N = 2 * nt, as the
    // space-to-depth forward does (dy plane p of the halo feeds the output planes p-1 (sd = 1) and p (sd = 0) of the
    // class). With nt = 32 (stem, d2) the unfolded launches are bound by the MMA thread's instruction issue
    // (profiles/r02f_stem_fwd_ncu_summary.txt); folding halves the number of UMMAs. The sd = 0 tap block lies 32 taps
    // BEHIND the sd = 1 block in the [tap][cin][cop] pack (kd = 3 - 2 sd or 2 - 2 sd).
    const bool fold = P.n_ntiles == 1 && nt_max <= 128 && od >= 2;
    if (fold) {
      P.kd_fold = 2;
      P.fold_nd = 2;
      P.fold_row_step = 32 * ncols;
    }
    P.ntaps = fold ? 4 : 8;
    P.out_s = 2;
    if (int e = make_act_map(&P.tm_src[0], dy, d->cop, ow, oh, od, d->n, 32, P.bw, P.bh, 1, plane_box(P))) return e;
    // one launch: the 8 parity classes are extra N tiles (blockIdx.y), each with its own tap set,
    // tile origin and scatter offset
    const int base_tiles = P.n_ntiles;
    if (base_tiles * 8 > kMaxNTiles) return fail(-2, "stride-2 dgrad: too many input channels (%d)", ncols);
    for (int cls = 1; cls < 8; ++cls)
      for (int i = 0; i < base_tiles; ++i) P.ntile[cls * base_tiles + i] = P.ntile[i];
    P.n_ntiles = base_tiles * 8;
    for (int pd = 0; pd < 2; ++pd)
      for (int ph = 0; ph < 2; ++ph)
        for (int pw = 0; pw < 2; ++pw) {
          const int cls = (pd * 2 + ph) * 2 + pw;
          P.atile_off[cls][0] = pw ? 0 : -1;
          P.atile_off[cls][1] = ph ? 0 : -1;
          P.atile_off[cls][2] = pd ? 0 : -1;
          for (int i = 0; i < base_tiles; ++i) {
            IgemmNTile& T = P.ntile[cls * base_tiles + i];
            T.tapset = cls;
            T.out_p[0] = pw; T.out_p[1] = ph; T.out_p[2] = pd;
          }
          int t = 0;
          for (int sd = fold ? 1 : 0; sd < 2; ++sd)        // folded: the table entry names the sd = 1 tap (block j = 0)
            for (int sh = 0; sh < 2; ++sh)
              for (int sw = 0; sw < 2; ++sw, ++t) {
                // shift s of class p: p=0 -> k = 3 - 2 s ; p=1 -> k = 2 - 2 s
                const int kd = pd ? 2 - 2 * sd : 3 - 2 * sd;
                const int kh = ph ? 2 - 2 * sh : 3 - 2 * sh;
                const int kw = pw ? 2 - 2 * sw : 3 - 2 * sw;
                P.taps[cls * P.ntaps + t] = IgemmTap{0, (uint16_t)(sh * P.bw + sw), (uint16_t)sd, (uint16_t)((kd * 4 + kh) * 4 + kw)};
              }
        }
    if (int e = finish_plan(&pl, nt_max)) return e;
    return launch_igemm(pl, st);
  }
  // UB_DECONV_K2S2 dgrad: gather the 8 fine sub-positions (parity tiles of dy, element stride 2)
  // Two output planes per tile: the stage holds the 8 parity tiles of every plane (64 KB per plane and 32-channel
  // chunk), which leaves room for ONE stage (profiles/r02h_deconv_dgrad_ncu_summary.txt: 4 TB/s, tensor pipe 10 %,
  // nothing near a roof). One-plane tiles with two or three stages were measured SLOWER on every level (64 -> 64 @64^3
  // 0.61 -> 0.79 ms, profiles/r02i_wgrad_split_ab.txt; removed): the launch is bound by the number of element-strided
  // TMA boxes, not by exposed load latency.
  P.td = d->d < 2 ? d->d : 2;
  P.Do = d->d; P.Ho = d->h; P.Wo = d->w;
  P.n_atiles = 8; P.bw = 8; P.bh = 16; P.n_in_planes = P.td; P.in_stride = 2;
  P.ntaps = 8;
  for (int i = 0; i < 2; ++i)
    for (int j = 0; j < 2; ++j)
      for (int k = 0; k < 2; ++k) {
        const int at = (i * 2 + j) * 2 + k;
        P.atile_off[at][0] = k; P.atile_off[at][1] = j; P.atile_off[at][2] = i;
        P.taps[at] = IgemmTap{(uint16_t)at, 0, 0, (uint16_t)at};
      }
  if (int e = make_act_map(&P.tm_src[0], dy, d->cop, ow, oh, od, d->n, kIgemmKc, P.bw, P.bh, 2, plane_box(P))) return e;
  if (int e = finish_plan(&pl, nt_max)) return e;
  return launch_igemm(pl, st);
}

// --------------------------------------------------------------------------------------------------
// wgrad
// --------------------------------------------------------------------------------------------------
struct WgradPlan {
  WgradParams P;
  dim3 grid;
  int smem;
  int ntap_lin;
  int tapmap[64];
};

static int plan_wgrad(const ub_conv_desc* d, WgradPlan* pl) {
  WgradParams& P = pl->P;
  memset(pl, 0, sizeof(*pl));
  int od, oh, ow;
  out_dims(d, &od, &oh, &ow);
  P.n_chunks_src0 = d->c0p / 32;
  P.n_chunks_total = (d->c0p + d->c1p) / 32;
  P.ci_total = d->c0p + d->c1p;
  P.co_total = d->cop;
  P.nt = d->cop < 128 ? d->cop : 128;
  P.n_cotiles = d->cop / P.nt;
  P.ncb = P.nt < 64 ? P.nt : 64;
  P.Nb = d->n;
  P.x_stride = 1; P.dy_stride = 1;
  P.x_nmul = d->kind == UB_CONV_K4S2P1_S2D ? 8 : 1;
  for (int i = 0; i < 64; ++i) pl->tapmap[i] = -1;
  if (d->kind == UB_CONV_K3S1P1) {
    P.bw = 10; P.bh = 18; P.Dt = od; P.Ht = oh; P.Wt = ow;
    P.n_variants = 3; P.ngroups = 3; P.group_row_step = P.bw; P.natoms = 3;
    for (int kd = 0; kd < 3; ++kd) { P.x_off[kd][0] = -1; P.x_off[kd][1] = -1; P.x_off[kd][2] = kd - 1; }
    for (int t = 0; t < 27; ++t) pl->tapmap[t] = t;
  } else if (d->kind == UB_CONV_K1) {
    P.bw = 8; P.bh = 16; P.Dt = od; P.Ht = oh; P.Wt = ow;
    P.n_variants = 1; P.ngroups = 1; P.group_row_step = 0; P.natoms = 1;
    pl->tapmap[0] = 0;
  } else if (is_k4(d->kind)) {
    const bool s2d = d->kind == UB_CONV_K4S2P1_S2D;
    P.bw = 9; P.bh = 17; P.Dt = od; P.Ht = oh; P.Wt = ow;
    P.x_stride = s2d ? 1 : 2;
    P.n_variants = 16; P.ngroups = 2; P.group_row_step = P.bw; P.natoms = 2;
    for (int pd = 0; pd < 2; ++pd)
      for (int ph = 0; ph < 2; ++ph)
        for (int pw = 0; pw < 2; ++pw)
          for (int sd = 0; sd < 2; ++sd) {
            const int v = ((pd * 2 + ph) * 2 + pw) * 2 + sd;
            P.x_off[v][0] = pw ? -1 : 0;
            P.x_off[v][1] = ph ? -1 : 0;
            // plain source: parity tile with element stride 2 (depth in input planes);
            // space-to-depth source: q-space coordinates, parity selects the channel block
            P.x_off[v][2] = s2d ? sd + (pd ? -1 : 0) : 2 * sd + (pd ? -1 : 0);
            P.x_nadd[v] = s2d ? (pd * 2 + ph) * 2 + pw : 0;
            for (int sh = 0; sh < 2; ++sh)
              for (int sw = 0; sw < 2; ++sw) {
                const int kd = 2 * sd + (1 - pd), kh = 2 * sh + (1 - ph), kw = 2 * sw + (1 - pw);
                pl->tapmap[(v * 2 + sh) * 2 + sw] = (kd * 4 + kh) * 4 + kw;
              }
          }
  } else {  // deconv: X coarse (no halo), dy = fine grid at parity (i,j,k)
    P.bw = 8; P.bh = 16; P.Dt = d->d; P.Ht = d->h; P.Wt = d->w;
    P.dy_stride = 2;
    P.n_variants = 8; P.ngroups = 1; P.group_row_step = 0; P.natoms = 1;
    for (int i = 0; i < 2; ++i)
      for (int j = 0; j < 2; ++j)
        for (int k = 0; k < 2; ++k) {
          const int v = (i * 2 + j) * 2 + k;
          P.dy_off[v][0] = k; P.dy_off[v][1] = j; P.dy_off[v][2] = i;
          pl->tapmap[v] = v;
        }
  }
  pl->ntap_lin = P.n_variants * P.ngroups * P.natoms;
  P.tiles_w = cdiv(P.Wt, 8);
  P.tiles_h = cdiv(P.Ht, 16);
  P.x_stage_bytes = align_up(P.bh * P.bw * 64, 1024);
  P.dy_stage_bytes = 128 * P.nt * 2;
  if (d->kind == UB_DECONV_K2S2) {
    // chunks on the M atoms, sub-positions side by side in N (igemm_wgrad.cuh, "dc mode"); one CTA per (chunk,
    // sub-position) measured slower (profiles/r02i_dc_wgrad_ab.txt), removed
    P.chunk_atoms = P.n_chunks_total < 4 ? P.n_chunks_total : 4;
    P.var_boxes = 256 / P.nt >= 8 ? 8 : (256 / P.nt >= 4 ? 4 : (256 / P.nt >= 2 ? 2 : 1));
    P.x_stage_bytes = P.chunk_atoms * P.bh * P.bw * 64;      // 8 KB tiles, already 1024-aligned
    P.dy_stage_bytes = P.var_boxes * 128 * P.nt * 2;
  }
  const int stage = P.x_stage_bytes + P.dy_stage_bytes;
  P.nstages = (200 * 1024) / stage;
  if (P.nstages > 4) P.nstages = 4;
  if (P.nstages < 2) return fail(-2, "wgrad stage too large");
  pl->smem = P.nstages * stage + 8 * 16 + 64 + 1024;
  P.tmem_cols = next_pow2_cols(P.ngroups * align_up((P.chunk_atoms ? P.var_boxes : 1) * P.nt, 32));
  const long long total_tiles = (long long)P.Nb * P.Dt * P.tiles_h * P.tiles_w;
  const int items = P.chunk_atoms ? cdiv(P.n_chunks_total, P.chunk_atoms) * (P.n_variants / P.var_boxes) * P.n_cotiles
                                  : P.n_chunks_total * P.n_variants * P.n_cotiles;
  // Splits of the voxel range per (chunk, variant, co tile) item. The CTAs are not persistent, so the grid must fill
  // whole waves of the CTAs an SM can hold (shared memory and TMEM columns decide: one or two, three for the narrow
  // layers). The earlier rule, cdiv(2 * 148, items), put 304 CTAs on 296 slots for the 64 -> 64 transposed conv: a
  // second wave of 8 CTAs, SMs active 57 % of the launch (profiles/r02h_deconv_wgrad_ncu_summary.txt; measured against
  // this one in profiles/r02i_wgrad_split_ab.txt, removed). Now: the split count that minimises waves x tiles-per-split,
  // up to four waves' worth.
  int occ = (228 * 1024) / (pl->smem + 1024);
  if (occ > 512 / P.tmem_cols) occ = 512 / P.tmem_cols;
  if (occ > 4) occ = 4;
  if (occ < 1) occ = 1;
  const long long cap = (long long)occ * sm_count();
  long long nsplit = 1, best_cost = -1;
  const long long ns_max = cdiv(4 * cap, items) < total_tiles ? cdiv(4 * cap, items) : total_tiles;
  for (long long ns = 1; ns <= ns_max; ++ns) {
    // time ~ waves x (tiles per split + a fixed per-CTA cost: pipeline fill, TMEM read-out, partial record)
    const long long cost = cdiv(items * ns, cap) * (cdiv(total_tiles, ns) + 32);
    if (best_cost < 0 || cost < best_cost) { nsplit = ns; best_cost = cost; }
  }
  if (nsplit > total_tiles) nsplit = total_tiles;
  if (nsplit < 1) nsplit = 1;
  pl->grid = dim3((unsigned)nsplit, (unsigned)items, 1);
  return 0;
}

// The marching wgrad kernel works on (32 ci x 32 co) blocks; it serves the 3x3x3 layers whose planes
// fill the 16x8 voxel tile reasonably (the deep, tiny-plane layers stay on the generic kernel).
static bool use_wgrad_march(const ub_conv_desc* d) {
  if (d->kind == UB_CONV_K4S2P1_S2D)      // the stem: 2x2x2-tap conv per input parity on the half-resolution grid
    return d->h >= 32 && d->w >= 16 && (long long)d->c0p * d->cop <= 64 * 64;
  return d->kind == UB_CONV_K3S1P1 && d->h >= 16 && d->w >= 8 && (long long)(d->c0p + d->c1p) * d->cop <= 128 * 256;
}
static int wgrad_march_splits(const ub_conv_desc* d) {
  int cols = (d->c0p + d->c1p) / 32 * (d->cop / 32);
  if (d->kind == UB_CONV_K4S2P1_S2D) cols *= 8;
  int ns = sm_count() / cols;
  return ns < 1 ? 1 : ns;
}

// split-K reduction of the weight-gradient partial records into the torch layout: many splits of a small output ->
// the 8-lanes-per-output kernel; large outputs -> the tiled transpose (measured against one thread per output in
// profiles/r02i_reduce_pack_ab.txt); the rest -> one thread per output.
static void launch_wgrad_reduce(const float* partial, float* dw, const WgradReduceArgs& R, cudaStream_t st) {
  const long long per_split = (long long)R.ntap * R.ci_total * R.co_total;
  int dst_ntaps = 0;
  bool unit_taps = R.dst_tap_stride == 1;
  for (int i = 0; i < R.ntap && i < 64; ++i)
    if (R.tapmap[i] + 1 > dst_ntaps) dst_ntaps = R.tapmap[i] + 1;
  if (per_split <= 65536 && R.nsplit >= 32)
    wgrad_reduce_wide_kernel<<<(unsigned)((per_split * 8 + 255) / 256), 256, 0, st>>>(partial, dw, R);
  else if (!unit_taps || dst_ntaps < 1 || dst_ntaps > 64 || R.ntap > 64 ||
           R.ci_total * cdiv(R.co_total, kRedTileCols) < 512)
    wgrad_reduce_kernel<<<(unsigned)((per_split + 255) / 256), 256, 0, st>>>(partial, dw, R);
  else
    wgrad_reduce_tiled_kernel<<<(unsigned)(R.ci_total * cdiv(R.co_total, kRedTileCols)), 256, 0, st>>>(partial, dw, R, dst_ntaps);
}

// Which kernel serves (desc, dir): 0 = igemm_fwd_kernel (generic tap-table implicit GEMM), 1 = igemm_march_kernel,
// 2 = wgrad_march_kernel, 3 = igemm_wgrad_kernel. dir: 0 forward, 1 dgrad, 2 wgrad. Used by the profiler / bench.py
// to attribute time and FLOPs to kernel classes.
extern "C" int ub_conv_kernel_class(const ub_conv_desc* d, int dir) {
  if (check_desc(d)) return -1;
  if (dir == 2) return use_wgrad_march(d) ? 2 : 3;
  if (dir != 0 && dir != 1) return fail(-1, "dir must be 0 (forward), 1 (dgrad) or 2 (wgrad)");
  return use_march(d, dir) ? 1 : 0;
}

extern "C" long long ub_conv_wgrad_workspace_bytes(const ub_conv_desc* d) {
  if (check_desc(d)) return -1;
  if (use_wgrad_march(d)) return (long long)wgrad_march_splits(d) * ntaps_of(d->kind) * (d->c0p + d->c1p) * d->cop * 4;
  WgradPlan pl;
  if (plan_wgrad(d, &pl)) return -1;
  return (long long)pl.grid.x * pl.ntap_lin * pl.P.ci_total * pl.P.co_total * 4;
}

extern "C" int ub_conv_wgrad(const ub_conv_desc* d, const void* src0, const void* src1, const void* dy,
                             void* workspace, float* dw, const ub_deferred_act* src0_act, void* stream) {
  if (int e = check_desc(d)) return e;
  if (src0_act && ub_conv_deferred_src0_ok(d) != 1)
    return fail(-2, "a deferred source activation is not supported for this weight gradient (ub_conv_deferred_src0_ok)");
  if (src0_act && src0_act->f16_operand)
    return fail(-2, "the weight gradient pairs the activations with bf16 gradients: a deferred source must use the bf16 form");
  if (int e = ensure_encode()) return e;
  if (!src0 || !dy || !workspace || !dw) return fail(-1, "null pointer in ub_conv_wgrad");
  if (d->c1p && !src1) return fail(-1, "second source missing");
  cudaStream_t st = (cudaStream_t)stream;
  if (use_wgrad_march(d)) {
    const bool stem = d->kind == UB_CONV_K4S2P1_S2D;
    const int kt = stem ? 2 : 3;
    // the grid the reduction runs over: the dY grid (stem: half resolution)
    const int gd = stem ? d->d / 2 : d->d, gh = stem ? d->h / 2 : d->h, gw = stem ? d->w / 2 : d->w;
    const int ntap = ntaps_of(d->kind);
    WgradMarchParams M;
    memset(&M, 0, sizeof(M));
    M.n_chunks_src0 = d->c0p / 32;
    M.n_chunks_total = (d->c0p + d->c1p) / 32;
    M.Nb = d->n; M.D = gd; M.H = gh; M.W = gw;
    march_geometry(d->n, gd, gh, gw, &M.tiles_w, &M.tiles_h, &M.nseg, &M.seg_len);
    M.ci_total = d->c0p + d->c1p;
    M.co_total = d->cop;
    M.n_cotiles = d->cop / 32;
    M.ntaps = ntap;
    M.partial = reinterpret_cast<float*>(workspace);
    const int bw = 8 + kt - 1, bh = 16 + kt - 1;
    if (int e = make_act_map(&M.tm_x[0], src0, d->c0p, gw, gh, gd, stem ? d->n * 8 : d->n, 32, bw, bh, 1)) return e;
    if (d->c1p)
      if (int e = make_act_map(&M.tm_x[1], src1, d->c1p, gw, gh, gd, d->n, 32, bw, bh, 1)) return e;
    if (int e = make_act_map(&M.tm_dy, dy, d->cop, gw, gh, gd, d->n, 32, 8, 16, 1)) return e;
    if (src0_act)
      if (int e = fill_deferred(&M.tf, src0_act)) return e;
    typedef void (*WmFn)(const WgradMarchParams);
    static const WmFn wfns[3] = {wgrad_march_kernel<3, false>, wgrad_march_kernel<2, false>, wgrad_march_kernel<3, true>};
    static SmemOptIn wopt[3];
    const int wv = stem ? 1 : (src0_act ? 2 : 0);
    if (int e = opt_in_smem(wopt[wv], (const void*)wfns[wv], "wgrad_march")) return e;
    const int nsplit = wgrad_march_splits(d);
    const int smem = kWmXStages * kWmXBytes + (kWmYSlots + kt - 1) * kWmYBytes + 8 * 32 + 64 + 1024;
    const dim3 grid((unsigned)nsplit, (unsigned)(M.n_chunks_total * M.n_cotiles * (stem ? 8 : 1)));
    wfns[wv]<<<grid, kWgradMarchThreads, smem, st>>>(M);
    UB_LAUNCH_CHECK();
    WgradReduceArgs R;
    memset(&R, 0, sizeof(R));
    const int ci = d->c0 + d->c1;
    R.nsplit = nsplit; R.ntap = ntap; R.ci_total = M.ci_total; R.co_total = d->cop; R.ci = ci; R.co = d->co;
    R.stride_ci = ntap; R.stride_co = (long long)ci * ntap; R.dst_tap_stride = 1;
    R.split_pad = d->c1p ? d->c0p : 0;
    R.split_real = d->c1p ? d->c0 : 0;
    for (int i = 0; i < 64; ++i) R.tapmap[i] = i < ntap ? i : -1;
    launch_wgrad_reduce(M.partial, dw, R, st);
    UB_LAUNCH_CHECK();
    return 0;
  }
  WgradPlan pl;
  if (int e = plan_wgrad(d, &pl)) return e;
  WgradParams& P = pl.P;
  int od, oh, ow;
  out_dims(d, &od, &oh, &ow);
  P.partial = reinterpret_cast<float*>(workspace);
  if (d->kind == UB_CONV_K4S2P1_S2D) {
    if (int e = make_act_map(&P.tm_x[0], src0, d->c0p, d->w / 2, d->h / 2, d->d / 2, d->n * 8, 32, P.bw, P.bh, 1)) return e;
  } else {
    if (int e = make_act_map(&P.tm_x[0], src0, d->c0p, d->w, d->h, d->d, d->n, 32, P.bw, P.bh, P.x_stride)) return e;
  }
  if (d->c1p)
    if (int e = make_act_map(&P.tm_x[1], src1, d->c1p, d->w, d->h, d->d, d->n, 32, P.bw, P.bh, P.x_stride)) return e;
  if (int e = make_act_map(&P.tm_dy, dy, d->cop, ow, oh, od, d->n, P.ncb, 8, 16, P.dy_stride)) return e;
  static SmemOptIn gopt;
  if (int e = opt_in_smem(gopt, (const void*)igemm_wgrad_kernel, "igemm_wgrad")) return e;
  igemm_wgrad_kernel<<<pl.grid, kWgradThreads, pl.smem, st>>>(P);
  UB_LAUNCH_CHECK();

  // split-K reduce + conversion to the torch layout
  WgradReduceArgs R;
  memset(&R, 0, sizeof(R));
  const int ntaps = ntaps_of(d->kind);
  const int ci = d->c0 + d->c1;
  R.nsplit = (int)pl.grid.x; R.ntap = pl.ntap_lin; R.ci_total = P.ci_total; R.co_total = P.co_total;
  R.ci = ci; R.co = d->co;
  if (d->kind == UB_DECONV_K2S2) { R.stride_ci = (long long)d->co * ntaps; R.stride_co = ntaps; }
  else { R.stride_ci = ntaps; R.stride_co = (long long)ci * ntaps; }
  R.dst_tap_stride = 1;
  R.split_pad = d->c1p ? d->c0p : 0;
  R.split_real = d->c1p ? d->c0 : 0;
  for (int i = 0; i < 64; ++i) R.tapmap[i] = i < pl.ntap_lin ? pl.tapmap[i] : -1;
  launch_wgrad_reduce(P.partial, dw, R, st);
  UB_LAUNCH_CHECK();
  return 0;
}

// --------------------------------------------------------------------------------------------------
// layout
// --------------------------------------------------------------------------------------------------
template <bool S2D>
static int launch_pack(const void* a, int a_bf16, int ca, const float* b, int cb, int n, long long voxels, int d, int h, int w,
                       int cp, void* out, cudaStream_t st) {
  constexpr int UNROLL = 4;
  __nv_bfloat16* o = reinterpret_cast<__nv_bfloat16*>(out);
  // bf16 input: the two-voxels-per-thread kernel (needs an even voxel count; S2D always has even dims)
  const bool pairs = a_bf16 && (voxels % 2 == 0) && (!S2D || w % 2 == 0);
  const __nv_bfloat16* a16 = reinterpret_cast<const __nv_bfloat16*>(a);
  if (cp == 32) {
    if (pairs) {
      const dim3 grid((unsigned)((voxels / 2 + 64 * UNROLL - 1) / (64 * UNROLL)), n);
      pack_ncdhw_a16_kernel<32, S2D, UNROLL><<<grid, 256, 0, st>>>(a16, ca, b, cb, o, voxels, d, h, w);
    } else {
      const dim3 grid((unsigned)((voxels + 64 * UNROLL - 1) / (64 * UNROLL)), n);
      if (a_bf16) pack_ncdhw_kernel<32, S2D, UNROLL, true><<<grid, 256, 0, st>>>(a, ca, b, cb, o, voxels, d, h, w);
      else pack_ncdhw_kernel<32, S2D, UNROLL, false><<<grid, 256, 0, st>>>(a, ca, b, cb, o, voxels, d, h, w);
    }
  } else {
    if (pairs) {
      const dim3 grid((unsigned)((voxels / 2 + 32 * UNROLL - 1) / (32 * UNROLL)), n);
      pack_ncdhw_a16_kernel<64, S2D, UNROLL><<<grid, 256, 0, st>>>(a16, ca, b, cb, o, voxels, d, h, w);
    } else {
      const dim3 grid((unsigned)((voxels + 32 * UNROLL - 1) / (32 * UNROLL)), n);
      if (a_bf16) pack_ncdhw_kernel<64, S2D, UNROLL, true><<<grid, 256, 0, st>>>(a, ca, b, cb, o, voxels, d, h, w);
      else pack_ncdhw_kernel<64, S2D, UNROLL, false><<<grid, 256, 0, st>>>(a, ca, b, cb, o, voxels, d, h, w);
    }
  }
  UB_LAUNCH_CHECK();
  return 0;
}

extern "C" int ub_pack_ncdhw(const void* a, int a_bf16, int ca, const float* b, int cb, int n, long long voxels, int cp,
                             void* out, void* stream) {
  if (!a || !out || ca <= 0 || n <= 0 || n > 65535 || (cb > 0 && !b)) return fail(-1, "bad arguments to ub_pack_ncdhw");
  if (ca + cb > cp || cp % 32 || cp > 64) return fail(-1, "ub_pack_ncdhw supports cp in {32, 64}, got ca=%d cb=%d cp=%d", ca, cb, cp);
  return launch_pack<false>(a, a_bf16, ca, b, cb, n, voxels, 0, 0, 0, cp, out, (cudaStream_t)stream);
}

extern "C" int ub_pack_ncdhw_s2d(const void* a, int a_bf16, int ca, const float* b, int cb, int n, int d, int h, int w, int cp,
                                 void* out, void* stream) {
  if (!a || !out || ca <= 0 || n <= 0 || n > 65535 || (cb > 0 && !b)) return fail(-1, "bad arguments to ub_pack_ncdhw_s2d");
  if (ca + cb > cp || cp % 32 || cp > 64) return fail(-1, "ub_pack_ncdhw_s2d supports cp in {32, 64}, got ca=%d cb=%d cp=%d", ca, cb, cp);
  if (d <= 0 || h <= 0 || w <= 0 || ((d | h | w) & 1)) return fail(-1, "ub_pack_ncdhw_s2d needs even positive dims");
  if ((long long)d * h * w >= (1ll << 31)) return fail(-2, "ub_pack_ncdhw_s2d: sample too large");
  return launch_pack<true>(a, a_bf16, ca, b, cb, n, (long long)d * h * w, d, h, w, cp, out, (cudaStream_t)stream);
}

extern "C" int ub_to_s2d(const void* src, int n, int d, int h, int w, int cp, void* dst, void* stream) {
  if (!src || !dst || n <= 0 || n > 65535 || d <= 0 || h <= 0 || w <= 0 || ((d | h | w) & 1) || cp <= 0 || cp % 8)
    return fail(-1, "bad arguments to ub_to_s2d (even positive dims, cp a multiple of 8)");
  const long long per_sample = (long long)d * h * w * (cp / 8);
  if (per_sample >= (1ll << 31)) return fail(-2, "ub_to_s2d: sample too large");
  to_s2d_kernel<<<dim3((unsigned)((per_sample + 255) / 256), n), 256, 0, (cudaStream_t)stream>>>(
      reinterpret_cast<const __nv_bfloat16*>(src), reinterpret_cast<__nv_bfloat16*>(dst), cp, d, h, w, (uint32_t)per_sample);
  UB_LAUNCH_CHECK();
  return 0;
}

extern "C" int ub_pack_patches(const float* a, int ca, int n, const long long* offsets, int d, int h, int w,
                               long long stride_c, long long stride_d, long long stride_h, int cp, void* out,
                               void* stream) {
  if (!a || !out || !offsets || ca <= 0 || n <= 0 || d <= 0 || h <= 0 || w <= 0) return fail(-1, "bad arguments to ub_pack_patches");
  if (n > kMaxPatchBatch) return fail(-1, "ub_pack_patches: at most %d patches per call", kMaxPatchBatch);
  if (ca > cp || (cp != 32 && cp != 64)) return fail(-1, "ub_pack_patches supports cp in {32, 64}, got ca=%d cp=%d", ca, cp);
  PatchGeom G;
  memset(&G, 0, sizeof(G));
  for (int i = 0; i < n; ++i) G.offset[i] = offsets[i];
  G.stride_c = stride_c; G.stride_d = stride_d; G.stride_h = stride_h; G.d = d; G.h = h; G.w = w;
  const long long V = (long long)d * h * w;
  constexpr int UNROLL = 4;
  __nv_bfloat16* o = reinterpret_cast<__nv_bfloat16*>(out);
  cudaStream_t st = (cudaStream_t)stream;
  if (cp == 32) pack_patches_kernel<32, UNROLL><<<dim3((unsigned)((V + 64 * UNROLL - 1) / (64 * UNROLL)), n), 256, 0, st>>>(a, ca, o, G);
  else pack_patches_kernel<64, UNROLL><<<dim3((unsigned)((V + 32 * UNROLL - 1) / (32 * UNROLL)), n), 256, 0, st>>>(a, ca, o, G);
  UB_LAUNCH_CHECK();
  return 0;
}

extern "C" int ub_unpack_patch(const void* src, int cp, int c_begin, int c, int sample, int d, int h, int w, float* dst,
                               long long dst_offset, long long stride_c, long long stride_d, long long stride_h,
                               void* stream) {
  if (!src || !dst || c <= 0 || c_begin < 0 || c_begin + c > cp || cp % 8 || sample < 0 || d <= 0 || h <= 0 || w <= 0)
    return fail(-1, "bad arguments to ub_unpack_patch");
  PatchGeom G;
  memset(&G, 0, sizeof(G));
  G.offset[0] = dst_offset;
  G.stride_c = stride_c; G.stride_d = stride_d; G.stride_h = stride_h; G.d = d; G.h = h; G.w = w;
  const long long V = (long long)d * h * w;
  unpack_patch_kernel<<<(unsigned)((V + 127) / 128), 128, 0, (cudaStream_t)stream>>>(
      reinterpret_cast<const __nv_bfloat16*>(src), dst, cp, c_begin, c, sample, G);
  UB_LAUNCH_CHECK();
  return 0;
}

extern "C" int ub_paste_patch(const float* src, int c, int d, int h, int w, float* dst, long long dst_offset,
                              long long stride_c, long long stride_d, long long stride_h, void* stream) {
  if (!src || !dst || c <= 0 || d <= 0 || h <= 0 || w <= 0) return fail(-1, "bad arguments to ub_paste_patch");
  PatchGeom G;
  memset(&G, 0, sizeof(G));
  G.offset[0] = dst_offset;
  G.stride_c = stride_c; G.stride_d = stride_d; G.stride_h = stride_h; G.d = d; G.h = h; G.w = w;
  const long long V = (long long)d * h * w;
  paste_patch_kernel<<<(unsigned)((V + 255) / 256), 256, 0, (cudaStream_t)stream>>>(src, dst, c, G);
  UB_LAUNCH_CHECK();
  return 0;
}

extern "C" int ub_blend_patches(const float* src, int n, int c, int pd, int ph, int pw, const int* origins,
                                const int* boxes, int mode, const float* window, float* out, float* weight, int d,
                                int h, int w, void* stream) {
  if (!src || !out || !origins || n <= 0 || c <= 0 || pd <= 0 || ph <= 0 || pw <= 0 || d <= 0 || h <= 0 || w <= 0)
    return fail(-1, "bad arguments to ub_blend_patches");
  if (n > kMaxPatchBatch) return fail(-1, "ub_blend_patches: at most %d patches per call", kMaxPatchBatch);
  if (c > kMaxBlendChannels) return fail(-1, "ub_blend_patches: at most %d channels, got %d", kMaxBlendChannels, c);
  if (mode != kBlendCrop && mode != kBlendAverage && mode != kBlendHann) return fail(-1, "ub_blend_patches: unknown mode %d", mode);
  if (mode != kBlendCrop && !weight) return fail(-1, "ub_blend_patches: the accumulating modes need the weight volume");
  if (mode == kBlendHann && !window) return fail(-1, "ub_blend_patches: hann mode needs the window vectors");
  BlendGeom G;
  memset(&G, 0, sizeof(G));
  G.n = n; G.c = c; G.pd = pd; G.ph = ph; G.pw = pw; G.H = h; G.W = w; G.V = (long long)d * h * w;
  const int dims[3] = {d, h, w}, p[3] = {pd, ph, pw};
  int lo[3] = {d, h, w}, hi[3] = {0, 0, 0};
  for (int i = 0; i < n; ++i) {
    for (int a = 0; a < 3; ++a) {
      const int o = origins[3 * i + a];
      const int b0 = boxes ? boxes[6 * i + a] : o, b1 = boxes ? boxes[6 * i + 3 + a] : o + p[a];
      if (o < 0 || o + p[a] > dims[a] || b0 < o || b1 > o + p[a] || b0 >= b1)
        return fail(-1, "ub_blend_patches: patch %d (origin %d, box [%d, %d) on axis %d) leaves the patch or the volume", i, o, b0, b1, a);
      G.org[i][a] = o; G.box[i][a] = b0; G.box[i][3 + a] = b1;
      lo[a] = b0 < lo[a] ? b0 : lo[a];
      hi[a] = b1 > hi[a] ? b1 : hi[a];
    }
  }
  for (int a = 0; a < 3; ++a) G.b0[a] = lo[a];
  G.bh = hi[1] - lo[1]; G.bw = hi[2] - lo[2];
  const long long V = (long long)(hi[0] - lo[0]) * G.bh * G.bw;
  if (G.V >= (1ll << 31)) return fail(-2, "ub_blend_patches: volume too large");
  const dim3 grid((unsigned)((V + 255) / 256));
  cudaStream_t st = (cudaStream_t)stream;
  if (mode == kBlendCrop) blend_patches_kernel<kBlendCrop><<<grid, 256, 0, st>>>(src, out, weight, window, G, (uint32_t)V);
  else if (mode == kBlendAverage) blend_patches_kernel<kBlendAverage><<<grid, 256, 0, st>>>(src, out, weight, window, G, (uint32_t)V);
  else blend_patches_kernel<kBlendHann><<<grid, 256, 0, st>>>(src, out, weight, window, G, (uint32_t)V);
  UB_LAUNCH_CHECK();
  return 0;
}

extern "C" int ub_blend_finish(float* out, const float* weight, int c, long long voxels, void* stream) {
  if (!out || !weight || c <= 0 || voxels <= 0) return fail(-1, "bad arguments to ub_blend_finish");
  if (voxels >= (1ll << 31)) return fail(-2, "ub_blend_finish: volume too large");
  blend_finish_kernel<<<(unsigned)((voxels + 255) / 256), 256, 0, (cudaStream_t)stream>>>(out, weight, c, (uint32_t)voxels);
  UB_LAUNCH_CHECK();
  return 0;
}

extern "C" int ub_unpack_ncdhw(const void* src, int cp, int c_begin, int c, int n, long long voxels, float* out,
                               void* stream) {
  if (!src || !out || c <= 0 || c_begin < 0 || c_begin + c > cp || cp % 8) return fail(-1, "bad arguments to ub_unpack_ncdhw");
  const long long total = (long long)n * voxels;
  unpack_ncdhw_kernel<<<(unsigned)((total + 127) / 128), 128, 0, (cudaStream_t)stream>>>(
      reinterpret_cast<const __nv_bfloat16*>(src), out, cp, c_begin, c, voxels, total);
  UB_LAUNCH_CHECK();
  return 0;
}

// --------------------------------------------------------------------------------------------------
// norm / act
// --------------------------------------------------------------------------------------------------
extern "C" int ub_norm_finalize(const float* stats_partial, int tiles_per_sample, int n, int cp, int c,
                                double voxels_per_sample, const float* gamma, const float* beta, float eps, int mode,
                                float momentum, float* running_mean, float* running_var, float* scale, float* shift,
                                float* mean, float* rstd, void* stream) {
  if (mode < 0 || mode > 2) return fail(-1, "bad norm mode %d", mode);
  if ((mode != 2 && !stats_partial) || !gamma || !beta || !scale || !shift || !mean || !rstd || cp % 32)
    return fail(-1, "bad arguments to ub_norm_finalize");
  if (mode == 2 && (!running_mean || !running_var)) return fail(-1, "eval BatchNorm needs running statistics");
  if (mode == UB_NORM_BATCH_TRAIN && n > 1 && (long long)tiles_per_sample * n >= 2048) {
    // many tile partials (the full-resolution input head): per-sample sums first, then one small combine
    bn_stats_stage1_kernel<<<dim3(cp / 32, n), dim3(32, 32), 0, (cudaStream_t)stream>>>(stats_partial, tiles_per_sample, cp,
                                                                                      scale, shift, mean, rstd);
    UB_LAUNCH_CHECK();
    bn_stats_stage2_kernel<<<cp / 32, 32, 0, (cudaStream_t)stream>>>(n, cp, c, voxels_per_sample, gamma, beta, eps, momentum,
                                                                    running_mean, running_var, scale, shift, mean, rstd);
    UB_LAUNCH_CHECK();
    return 0;
  }
  stats_finalize_kernel<<<dim3(cp / 32, mode == UB_NORM_INSTANCE ? n : 1), dim3(32, 32), 0, (cudaStream_t)stream>>>(
      stats_partial, tiles_per_sample, n, cp, c, voxels_per_sample, gamma, beta, eps, mode, momentum, running_mean,
      running_var, scale, shift, mean, rstd);
  UB_LAUNCH_CHECK();
  return 0;
}

extern "C" int ub_norm_act_fwd(const void* y, const float* scale, const float* shift, float slope, float drop_p,
                               uint32_t drop_seed, int n, int d, int h, int w, int cp, void* a, void* a_f16, void* pooled,
                               void* stream) {
  if (!y || (!a && !a_f16 && !pooled) || cp % 8) return fail(-1, "bad arguments to ub_norm_act_fwd");
  if (drop_p < 0.f || drop_p >= 1.f) return fail(-1, "dropout p out of range");
  NormActArgs A{scale, shift, slope, drop_p, drop_seed, drop_thresh(drop_p)};
  const long long V = (long long)d * h * w;
  cudaStream_t st = (cudaStream_t)stream;
  if (!pooled) {
    const long long vps = V * (cp / 8);
    if (vps >= (1ll << 31) || n > 65535) return fail(-2, "ub_norm_act_fwd: sample too large");
    constexpr int UNROLL = 4;
    const dim3 grid((unsigned)((vps + 256 * UNROLL - 1) / (256 * UNROLL)), n);
    const __nv_bfloat16* yp = reinterpret_cast<const __nv_bfloat16*>(y);
    __nv_bfloat16* ap = reinterpret_cast<__nv_bfloat16*>(a);
    __nv_bfloat16* ap16 = reinterpret_cast<__nv_bfloat16*>(a_f16);
    if (256 % (cp / 8) == 0) norm_act_fwd_kernel<UNROLL, true><<<grid, 256, 0, st>>>(yp, ap, ap16, A, cp, (uint32_t)vps);
    else norm_act_fwd_kernel<UNROLL, false><<<grid, 256, 0, st>>>(yp, ap, ap16, A, cp, (uint32_t)vps);
  } else {
    if ((d | h | w) & 1) return fail(-1, "fused max-pool needs even dims");
    const long long per_sample = (V / 8) * (cp / 8);
    if (per_sample >= (1ll << 31) || n > 65535) return fail(-2, "ub_norm_act_fwd: sample too large");
    norm_act_pool_fwd_kernel<<<dim3((unsigned)((per_sample + 255) / 256), n), 256, 0, st>>>(
        reinterpret_cast<const __nv_bfloat16*>(y), reinterpret_cast<__nv_bfloat16*>(a),
        reinterpret_cast<__nv_bfloat16*>(a_f16), reinterpret_cast<__nv_bfloat16*>(pooled), A, cp, n, d, h, w,
        (uint32_t)per_sample);
  }
  UB_LAUNCH_CHECK();
  return 0;
}

// blocks per sample of the backward reduction: enough CTAs to fill the GPU whatever the batch size
static int bwd_blocks_per_sample(int n) {
  int b = (1184 + n - 1) / n;
  return b < 128 ? 128 : b;
}
extern "C" long long ub_norm_act_bwd_workspace_bytes(int n, int cp) {
  // block partials + c1 + c2
  return ((long long)n * bwd_blocks_per_sample(n) * 2 * cp + 2ll * n * cp) * 4;
}

extern "C" int ub_norm_act_bwd(const void* dA, const void* a, const void* y, int mode, const float* mean,
                               const float* rstd, const float* scale, const float* shift, float slope, float drop_p,
                               uint32_t drop_seed,
                               int n, long long voxels, int cp, int c, void* workspace, void* dy, float* dgamma,
                               float* dbeta, float* dbias, const float* ext_partial, int ext_records_per_sample,
                               void* stream) {
  if (!dA || !dy || cp % 8 || n <= 0 || n > 65535) return fail(-1, "bad arguments to ub_norm_act_bwd");
  if (!a && (mode == UB_NORM_NONE || !shift)) return fail(-1, "ub_norm_act_bwd needs the activations `a` or (y, scale, shift)");
  const int c8 = cp / 8;
  if (cp > 512 || 256 % c8) return fail(-2, "norm/activation backward supports cp in {8..512} with cp/8 dividing 256, got %d", cp);
  const long long vps = voxels * c8;
  if (vps >= (1ll << 31)) return fail(-2, "ub_norm_act_bwd: sample too large");
  cudaStream_t st = (cudaStream_t)stream;
  NormBwdArgs B;
  memset(&B, 0, sizeof(B));
  B.slope = slope; B.drop_p = drop_p; B.drop_seed = drop_seed; B.drop_thresh = drop_thresh(drop_p);
  if (mode != UB_NORM_NONE) {
    if (!y || !mean || !rstd || !scale || !workspace) return fail(-1, "norm backward needs y, mean, rstd, scale, workspace");
    const int bps_max = bwd_blocks_per_sample(n);
    float* part = reinterpret_cast<float*>(workspace);
    float* c1 = part + (size_t)n * bps_max * 2 * cp;
    float* c2 = c1 + (size_t)n * cp;
    B.mean = mean; B.rstd = rstd; B.gscale = scale; B.c1 = c1; B.c2 = c2;
    B.fshift = shift;   // non-null: LeakyReLU branch from sign(y * scale + shift), `a` is not read
    int threads = 256;
    if (threads < cp) threads = cp;
    long long bps = bps_max;
    if (bps * threads * 4 > vps) bps = (vps + 4ll * threads - 1) / (4ll * threads);
    if (bps < 1) bps = 1;
    const float* part_in = part;
    if (ext_partial) {
      // the reductions were accumulated by the producer of dA (ub_conv_dgrad_fused)
      if (ext_records_per_sample <= 0) return fail(-1, "ext_records_per_sample must be positive");
      part_in = ext_partial;
      bps = ext_records_per_sample;
    } else {
      norm_act_bwd_reduce_kernel<<<dim3((unsigned)bps, n), threads, 2 * threads * 8 * sizeof(float), st>>>(
          reinterpret_cast<const __nv_bfloat16*>(dA), reinterpret_cast<const __nv_bfloat16*>(a),
          reinterpret_cast<const __nv_bfloat16*>(y), B, cp, (uint32_t)vps, part);
      UB_LAUNCH_CHECK();
    }
    norm_bwd_finalize_kernel<<<cp / 32, dim3(32, 32), 0, st>>>(part_in, (int)bps, n, cp, c, (double)voxels, mode, scale, c1, c2,
                                                           dgamma, dbeta, dbias);
    UB_LAUNCH_CHECK();
  }
  if (mode != UB_NORM_NONE && shift != nullptr && !env_flag("UB_NAB_GENERIC")) {
    // statistics present, sign from y: the instruction-lean kernel
    const dim3 grid((unsigned)((vps + 256 * kApplyVPT - 1) / (256 * kApplyVPT)), n);
    if (drop_p > 0.f)
      norm_act_bwd_apply_y_kernel<true><<<grid, 256, 0, st>>>(reinterpret_cast<const __nv_bfloat16*>(dA),
                                                              reinterpret_cast<const __nv_bfloat16*>(y),
                                                              reinterpret_cast<__nv_bfloat16*>(dy), B, cp, (uint32_t)vps);
    else
      norm_act_bwd_apply_y_kernel<false><<<grid, 256, 0, st>>>(reinterpret_cast<const __nv_bfloat16*>(dA),
                                                               reinterpret_cast<const __nv_bfloat16*>(y),
                                                               reinterpret_cast<__nv_bfloat16*>(dy), B, cp, (uint32_t)vps);
    UB_LAUNCH_CHECK();
    return 0;
  }
  constexpr int UNROLL = 4;
  norm_act_bwd_apply_kernel<UNROLL><<<dim3((unsigned)((vps + 256 * UNROLL - 1) / (256 * UNROLL)), n), 256, 0, st>>>(
      reinterpret_cast<const __nv_bfloat16*>(dA), reinterpret_cast<const __nv_bfloat16*>(a),
      reinterpret_cast<const __nv_bfloat16*>(y), reinterpret_cast<__nv_bfloat16*>(dy), B, cp, (uint32_t)vps);
  UB_LAUNCH_CHECK();
  return 0;
}

extern "C" int ub_maxpool_bwd(const void* a, const void* dP, void* dA, int accumulate, int n, int d, int h, int w,
                              int cp, const ub_deferred_act* a_act, void* stream) {
  if (!a || !dP || !dA || cp % 8 || ((d | h | w) & 1)) return fail(-1, "bad arguments to ub_maxpool_bwd");
  NormActArgs A;
  memset(&A, 0, sizeof(A));
  if (a_act)
    if (int e = fill_deferred(&A, a_act)) return e;
  const long long per_sample = ((long long)d * h * w / 8) * (cp / 8);
  if (per_sample >= (1ll << 31) || n <= 0 || n > 65535) return fail(-2, "ub_maxpool_bwd: sample too large");
  const dim3 grid((unsigned)((per_sample + 255) / 256), n);
  if (a_act)
    maxpool_bwd_kernel<true><<<grid, 256, 0, (cudaStream_t)stream>>>(
        reinterpret_cast<const __nv_bfloat16*>(a), reinterpret_cast<const __nv_bfloat16*>(dP),
        reinterpret_cast<__nv_bfloat16*>(dA), accumulate, cp, n, d, h, w, (uint32_t)per_sample, A);
  else
    maxpool_bwd_kernel<false><<<grid, 256, 0, (cudaStream_t)stream>>>(
        reinterpret_cast<const __nv_bfloat16*>(a), reinterpret_cast<const __nv_bfloat16*>(dP),
        reinterpret_cast<__nv_bfloat16*>(dA), accumulate, cp, n, d, h, w, (uint32_t)per_sample, A);
  UB_LAUNCH_CHECK();
  return 0;
}

// ---- max-pool backward fused with the norm-backward reduction of the block it completes ----
static void maxpool_fuse_plan(int d, int h, int w, int cp, long long* per_sample, int* iters, int* blocks) {
  *per_sample = ((long long)d * h * w / 8) * (cp / 8);
  const long long nblk = (*per_sample + 255) / 256;
  long long it = (nblk + 295) / 296;       // a few hundred records per sample at most (the finalize walks them)
  if (it < 1) it = 1;
  *iters = (int)it;
  *blocks = (int)((nblk + it - 1) / it);
}
extern "C" int ub_maxpool_bwd_fuse_records(int n, int d, int h, int w, int cp) {
  if (n <= 0 || cp % 8 || cp > 512 || 256 % (cp / 8) || ((d | h | w) & 1)) return 0;
  long long ps; int it, nb;
  maxpool_fuse_plan(d, h, w, cp, &ps, &it, &nb);
  return n * nb;
}
extern "C" int ub_maxpool_bwd_fused(const void* dP, void* dA, int accumulate, int n, int d, int h, int w, int cp,
                                    const ub_norm_bwd_fuse* f, void* stream) {
  if (!dP || !dA || !f || !f->y || !f->scale || !f->shift || !f->mean || !f->rstd || !f->partial)
    return fail(-1, "bad arguments to ub_maxpool_bwd_fused");
  if (ub_maxpool_bwd_fuse_records(n, d, h, w, cp) <= 0 || n > 65535)
    return fail(-2, "ub_maxpool_bwd_fused: unsupported shape (cp/8 must divide 256, even sizes)");
  long long per_sample; int iters, blocks;
  maxpool_fuse_plan(d, h, w, cp, &per_sample, &iters, &blocks);
  if (per_sample >= (1ll << 31)) return fail(-2, "ub_maxpool_bwd_fused: sample too large");
  NormActArgs A;
  memset(&A, 0, sizeof(A));
  A.scale = f->scale; A.shift = f->shift; A.slope = f->slope; A.drop_p = f->drop_p; A.drop_seed = f->drop_seed;
  A.drop_thresh = drop_thresh(f->drop_p);
  maxpool_bwd_sums_kernel<<<dim3((unsigned)blocks, n), 256, 2 * 256 * 8 * sizeof(float), (cudaStream_t)stream>>>(
      reinterpret_cast<const __nv_bfloat16*>(f->y), reinterpret_cast<const __nv_bfloat16*>(dP),
      reinterpret_cast<__nv_bfloat16*>(dA), accumulate, cp, d, h, w, (uint32_t)per_sample, iters, A, f->mean, f->rstd,
      f->partial);
  UB_LAUNCH_CHECK();
  return 0;
}

static const int kColsumBlocks = 592;
extern "C" long long ub_colsum_workspace_bytes(int cp) { return (long long)kColsumBlocks * cp * 4; }
extern "C" int ub_colsum(const void* x, long long rows, int cp, int c, void* workspace, float* out, void* stream) {
  if (!x || !workspace || !out || cp % 8 || cp > 512) return fail(-1, "bad arguments to ub_colsum");
  cudaStream_t st = (cudaStream_t)stream;
  int threads = 256;
  if (threads < cp) threads = cp;
  colsum_bf16_kernel<<<kColsumBlocks, threads, threads * 8 * sizeof(float), st>>>(
      reinterpret_cast<const __nv_bfloat16*>(x), rows, cp, reinterpret_cast<float*>(workspace));
  UB_LAUNCH_CHECK();
  colsum_finish_kernel<<<(c + 7) / 8, dim3(32, 8), 0, st>>>(reinterpret_cast<const float*>(workspace), kColsumBlocks, cp, c, out);
  UB_LAUNCH_CHECK();
  return 0;
}

// --------------------------------------------------------------------------------------------------
// losses
// --------------------------------------------------------------------------------------------------
static const int kL1Blocks = 1184;
extern "C" long long ub_l1_workspace_bytes(void) { return (long long)kL1Blocks * 8 + 16; }
extern "C" int ub_l1_fwd(const float* a, const float* b, long long numel, void* workspace, float* loss, void* stream) {
  if (!a || !b || !workspace || !loss || numel <= 0) return fail(-1, "bad arguments to ub_l1_fwd");
  if (((uintptr_t)a | (uintptr_t)b) & 15) return fail(-1, "ub_l1_fwd needs 16-byte aligned inputs");
  double* part = reinterpret_cast<double*>(workspace);
  unsigned int* ticket = reinterpret_cast<unsigned int*>(part + kL1Blocks);  // must be zero on first use
  l1_fwd_kernel<<<kL1Blocks, 256, 0, (cudaStream_t)stream>>>(a, b, numel, part, ticket, loss);
  UB_LAUNCH_CHECK();
  return 0;
}
extern "C" int ub_l1_bwd(const float* a, const float* b, const float* grad_out, long long numel, float* da, void* stream) {
  if (!a || !b || !grad_out || !da || numel <= 0) return fail(-1, "bad arguments to ub_l1_bwd");
  if (((uintptr_t)a | (uintptr_t)b | (uintptr_t)da) & 15) return fail(-1, "ub_l1_bwd needs 16-byte aligned tensors");
  l1_bwd_kernel<<<kL1Blocks, 256, 0, (cudaStream_t)stream>>>(a, b, grad_out, numel, da);
  UB_LAUNCH_CHECK();
  return 0;
}
extern "C" int ub_bce_logits(const float* x, const float* target, float target_const, int numel, float* loss,
                             float* dx_unit, void* stream) {
  if (!x || !loss || numel <= 0) return fail(-1, "bad arguments to ub_bce_logits");
  bce_logits_kernel<<<1, 256, 0, (cudaStream_t)stream>>>(x, target, target_const, numel, loss, dx_unit);
  UB_LAUNCH_CHECK();
  return 0;
}
extern "C" int ub_scale(const float* x, const float* scalar, long long numel, float* y, void* stream) {
  if (!x || !scalar || !y || numel <= 0) return fail(-1, "bad arguments to ub_scale");
  long long blocks = (numel + 255) / 256;
  if (blocks > 2368) blocks = 2368;
  scale_by_scalar_kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(x, scalar, numel, y);
  UB_LAUNCH_CHECK();
  return 0;
}

// --------------------------------------------------------------------------------------------------
// evaluation
// --------------------------------------------------------------------------------------------------
extern "C" int ub_relerr_map_reduce(const float* pred, const float* target, const unsigned char* mask,
                                    const float* probseg, int c, int r, long long voxels, int angular, float* diff,
                                    double* sums, double* norms, void* stream) {
  if (!pred || !target || c <= 0 || c > 8 || r < 0 || r > 3 || voxels <= 0) return fail(-1, "bad arguments to ub_relerr_map_reduce");
  if (probseg && (!sums || !norms || r == 0)) return fail(-1, "ROI reduction needs sums, norms and r > 0");
  cudaStream_t st = (cudaStream_t)stream;
  if (probseg) {
    UB_CUDA(cudaMemsetAsync(sums, 0, sizeof(double) * r * c, st));
    UB_CUDA(cudaMemsetAsync(norms, 0, sizeof(double) * r, st));
  }
  long long blocks = (voxels + 255) / 256;
  if (blocks > 1184) blocks = 1184;
  relerr_kernel<<<(unsigned)blocks, 256, 0, st>>>(pred, target, mask, probseg, c, r, voxels, angular, diff, sums, norms);
  UB_LAUNCH_CHECK();
  return 0;
}

extern "C" int ub_dti_scalar_maps(const float* tensor6, long long voxels, float* fa, float* md, float* ad, float* rd,
                                  float* azimuth, float* inclination, float* rgb, void* stream) {
  if (!tensor6 || voxels <= 0) return fail(-1, "bad arguments to ub_dti_scalar_maps");
  dti_scalar_maps_kernel<<<(unsigned)((voxels + 127) / 128), 128, 0, (cudaStream_t)stream>>>(tensor6, voxels, fa, md, ad, rd,
                                                                                           azimuth, inclination, rgb);
  UB_LAUNCH_CHECK();
  return 0;
}

// --------------------------------------------------------------------------------------------------
// output head: 1x1x1 conv fused with the layout change (ref: BasicUNet.final_conv)
// --------------------------------------------------------------------------------------------------
static const int kC1BwdBlocks = 1184;
static int fill_conv1x1_weights(const float* w, int ci, const float* bias, int co, void* table_dev, cudaStream_t st);

extern "C" long long ub_conv1x1_workspace_bytes(void) {
  // [Conv1x1Weights table | block partials of the backward]
  return (long long)sizeof(Conv1x1Weights) + (long long)kC1BwdBlocks * kC1MaxCo * 33 * 4;
}

// w / bias are DEVICE pointers (the fp32 Parameters); the zero-padded table is built on the device
__global__ void conv1x1_table_kernel(const float* __restrict__ w, int ci, const float* __restrict__ bias, int co,
                                     Conv1x1Weights* __restrict__ T) {
  for (int i = threadIdx.x; i < kC1MaxCo * 32; i += blockDim.x) {
    const int c = i / 32, k = i % 32;
    T->w[c][k] = (c < co && k < ci) ? w[c * ci + k] : 0.f;
  }
  if (threadIdx.x < kC1MaxCo) T->b[threadIdx.x] = (bias != nullptr && (int)threadIdx.x < co) ? bias[threadIdx.x] : 0.f;
}
static int fill_conv1x1_weights(const float* w, int ci, const float* bias, int co, void* table_dev, cudaStream_t st) {
  conv1x1_table_kernel<<<1, 256, 0, st>>>(w, ci, bias, co, reinterpret_cast<Conv1x1Weights*>(table_dev));
  UB_LAUNCH_CHECK();
  return 0;
}

extern "C" int ub_conv1x1_to_ncdhw(const void* u, int cp, const float* w, int ci, const float* bias, int co, int n,
                                   long long voxels, void* workspace, float* out, const ub_deferred_act* u_act,
                                   void* stream) {
  if (!u || !w || !out || !workspace || n <= 0 || n > 65535 || voxels <= 0) return fail(-1, "bad arguments to ub_conv1x1_to_ncdhw");
  if (cp != 32 || ci <= 0 || ci > 32 || co <= 0 || co > kC1MaxCo)
    return fail(-2, "ub_conv1x1_to_ncdhw supports cp = 32, ci <= 32, co <= %d (got cp=%d ci=%d co=%d)", kC1MaxCo, cp, ci, co);
  cudaStream_t st = (cudaStream_t)stream;
  if (int e = fill_conv1x1_weights(w, ci, bias, co, workspace, st)) return e;
  if (voxels >= (1ll << 31)) return fail(-2, "ub_conv1x1_to_ncdhw: sample too large");
  long long blocks = (voxels + 255) / 256;
  const long long cap = (8ll * sm_count() + n - 1) / n;
  if (blocks > cap) blocks = cap;
  const dim3 grid((unsigned)blocks, n);
  const __nv_bfloat16* up = reinterpret_cast<const __nv_bfloat16*>(u);
  const Conv1x1Weights* T = reinterpret_cast<const Conv1x1Weights*>(workspace);
  NormActArgs A;
  memset(&A, 0, sizeof(A));
  if (u_act)
    if (int e = fill_deferred(&A, u_act)) return e;
  if (voxels % 8 == 0 && !env_flag("UB_HEAD_CUDA_CORES")) {
    // warp-level MMA form (head_mma.cuh): a warp takes kHeadFwdUnroll groups of 8 voxels per iteration
    long long mb = (voxels / 8 + 8 * kHeadFwdUnroll - 1) / (8 * kHeadFwdUnroll);
    if (mb > cap) mb = cap;
    const dim3 mgrid((unsigned)mb, n);
    switch (co) {
#define UB_C1_FWD(C_) case C_: \
      if (u_act) head_fwd_mma_kernel<C_, true><<<mgrid, 256, 0, st>>>(up, out, T, (uint32_t)voxels, A); \
      else head_fwd_mma_kernel<C_, false><<<mgrid, 256, 0, st>>>(up, out, T, (uint32_t)voxels, A); \
      break;
      UB_C1_FWD(1) UB_C1_FWD(2) UB_C1_FWD(3) UB_C1_FWD(4) UB_C1_FWD(5) UB_C1_FWD(6) UB_C1_FWD(7) UB_C1_FWD(8)
#undef UB_C1_FWD
    }
    UB_LAUNCH_CHECK();
    return 0;
  }
  switch (co) {
#define UB_C1_FWD(C_) case C_: \
    if (u_act) conv1x1_to_ncdhw_kernel<C_, true><<<grid, 256, 0, st>>>(up, out, T, (uint32_t)voxels, A); \
    else conv1x1_to_ncdhw_kernel<C_, false><<<grid, 256, 0, st>>>(up, out, T, (uint32_t)voxels, A); \
    break;
    UB_C1_FWD(1) UB_C1_FWD(2) UB_C1_FWD(3) UB_C1_FWD(4) UB_C1_FWD(5) UB_C1_FWD(6) UB_C1_FWD(7) UB_C1_FWD(8)
#undef UB_C1_FWD
  }
  UB_LAUNCH_CHECK();
  return 0;
}

extern "C" int ub_conv1x1_from_ncdhw_bwd(const float* dout, int co, const void* u, int cp, const float* w, int ci, int n,
                                         long long voxels, void* workspace, void* du, float* dw, float* db,
                                         const ub_deferred_act* u_act, void* stream) {
  if (!dout || !w || !workspace || n <= 0 || voxels <= 0) return fail(-1, "bad arguments to ub_conv1x1_from_ncdhw_bwd");
  if ((dw || db) && !u) return fail(-1, "ub_conv1x1_from_ncdhw_bwd: weight / bias gradients need the forward input u");
  if (cp != 32 || ci <= 0 || ci > 32 || co <= 0 || co > kC1MaxCo)
    return fail(-2, "ub_conv1x1_from_ncdhw_bwd supports cp = 32, ci <= 32, co <= %d", kC1MaxCo);
  cudaStream_t st = (cudaStream_t)stream;
  if (int e = fill_conv1x1_weights(w, ci, nullptr, co, workspace, st)) return e;
  float* part = reinterpret_cast<float*>(reinterpret_cast<char*>(workspace) + sizeof(Conv1x1Weights));
  const int want_w = (dw || db) ? 1 : 0;
  if (voxels >= (1ll << 31) || n > 65535) return fail(-2, "ub_conv1x1_from_ncdhw_bwd: sample too large");
  long long blocks = (voxels + 127) / 128;
  long long cap = kC1BwdBlocks / n;
  if (cap < 1) cap = 1;
  if (blocks > cap) blocks = cap;
  const dim3 grid((unsigned)blocks, n);
  const __nv_bfloat16* up = reinterpret_cast<const __nv_bfloat16*>(u);
  __nv_bfloat16* dup = reinterpret_cast<__nv_bfloat16*>(du);
  const Conv1x1Weights* T = reinterpret_cast<const Conv1x1Weights*>(workspace);
  NormActArgs A;
  memset(&A, 0, sizeof(A));
  if (u_act)
    if (int e = fill_deferred(&A, u_act)) return e;
  switch (co) {
#define UB_C1_BWD(C_) case C_: \
    if (u_act) conv1x1_from_ncdhw_bwd_kernel<C_, true><<<grid, 256, 0, st>>>(dout, up, dup, T, (uint32_t)voxels, want_w, part, A); \
    else conv1x1_from_ncdhw_bwd_kernel<C_, false><<<grid, 256, 0, st>>>(dout, up, dup, T, (uint32_t)voxels, want_w, part, A); \
    break;
    UB_C1_BWD(1) UB_C1_BWD(2) UB_C1_BWD(3) UB_C1_BWD(4) UB_C1_BWD(5) UB_C1_BWD(6) UB_C1_BWD(7) UB_C1_BWD(8)
#undef UB_C1_BWD
  }
  UB_LAUNCH_CHECK();
  if (want_w) {
    conv1x1_bwd_finish_kernel<<<(kC1MaxCo * 33 + 3) / 4, dim3(32, 4), 0, st>>>(part, (int)(blocks * n), co, ci, dw, db);
    UB_LAUNCH_CHECK();
  }
  return 0;
}

// ---- output head backward fused with the norm backward of the block in front of it (head_mma.cuh) ----
static int head_fused_bps(int n) {
  int b = (2 * 148 + n - 1) / n;     // two resident blocks per SM over the whole grid
  return b < 1 ? 1 : b;
}
extern "C" long long ub_head_bwd_fused_workspace_bytes(int n) {
  const long long recs = (long long)n * head_fused_bps(n);
  // [weight table | dW/db partials | S1/S2 partials | c1 | c2]
  return (long long)sizeof(Conv1x1Weights) + (recs * kC1MaxCo * 33 + recs * 64 + 2ll * n * 32) * 4;
}
extern "C" int ub_head_bwd_fused(const float* dout, int co, const float* w, int ci, int n, long long voxels,
                                 const ub_norm_bwd_fuse* blk, int mode, int c, void* workspace, void* dy,
                                 float* dgamma, float* dbeta, float* dbias, float* dw, float* db, void* stream) {
  if (!dout || !w || !blk || !blk->y || !blk->scale || !blk->shift || !blk->mean || !blk->rstd || !workspace || !dy ||
      n <= 0 || n > 65535 || voxels <= 0)
    return fail(-1, "bad arguments to ub_head_bwd_fused");
  if (ci <= 0 || ci > 32 || co <= 0 || co > kC1MaxCo || c <= 0 || c > 32)
    return fail(-2, "ub_head_bwd_fused supports ci <= 32, co <= %d (got ci=%d co=%d)", kC1MaxCo, ci, co);
  if (voxels % 16 || voxels >= (1ll << 31)) return fail(-2, "ub_head_bwd_fused: voxels per sample must be a multiple of 16");
  if (mode == UB_NORM_NONE) return fail(-2, "ub_head_bwd_fused: the block in front of the head must have a norm");
  cudaStream_t st = (cudaStream_t)stream;
  if (int e = fill_conv1x1_weights(w, ci, nullptr, co, workspace, st)) return e;
  long long bps = head_fused_bps(n);
  const long long max_b = (voxels / 16 + 7) / 8;
  if (bps > max_b) bps = max_b;
  const long long recs = (long long)n * head_fused_bps(n);
  float* part_w = reinterpret_cast<float*>(reinterpret_cast<char*>(workspace) + sizeof(Conv1x1Weights));
  float* part_n = part_w + recs * kC1MaxCo * 33;
  float* c1 = part_n + recs * 64;
  float* c2 = c1 + (size_t)n * 32;
  const Conv1x1Weights* T = reinterpret_cast<const Conv1x1Weights*>(workspace);
  NormActArgs A;
  memset(&A, 0, sizeof(A));
  A.scale = blk->scale; A.shift = blk->shift; A.slope = blk->slope; A.drop_p = blk->drop_p; A.drop_seed = blk->drop_seed;
  A.drop_thresh = drop_thresh(blk->drop_p);
  const int want_w = (dw || db) ? 1 : 0;
  const dim3 grid((unsigned)bps, n);
  const __nv_bfloat16* yp = reinterpret_cast<const __nv_bfloat16*>(blk->y);
  switch (co) {
#define UB_HEAD_K1(C_) case C_: \
    head_bwd_sums_mma_kernel<C_><<<grid, 256, 0, st>>>(dout, yp, T, (uint32_t)voxels, A, blk->mean, blk->rstd, want_w, part_w, part_n); \
    break;
    UB_HEAD_K1(1) UB_HEAD_K1(2) UB_HEAD_K1(3) UB_HEAD_K1(4) UB_HEAD_K1(5) UB_HEAD_K1(6) UB_HEAD_K1(7) UB_HEAD_K1(8)
#undef UB_HEAD_K1
  }
  UB_LAUNCH_CHECK();
  if (want_w) {
    conv1x1_bwd_finish_kernel<<<(kC1MaxCo * 33 + 3) / 4, dim3(32, 4), 0, st>>>(part_w, (int)(bps * n), co, ci, dw, db);
    UB_LAUNCH_CHECK();
  }
  norm_bwd_finalize_kernel<<<1, dim3(32, 32), 0, st>>>(part_n, (int)bps, n, 32, c, (double)voxels, mode, blk->scale, c1, c2,
                                                      dgamma, dbeta, dbias);
  UB_LAUNCH_CHECK();
  NormBwdArgs B;
  memset(&B, 0, sizeof(B));
  B.slope = blk->slope; B.drop_p = blk->drop_p; B.drop_seed = blk->drop_seed; B.drop_thresh = drop_thresh(blk->drop_p);
  B.mean = blk->mean; B.rstd = blk->rstd; B.gscale = blk->scale; B.c1 = c1; B.c2 = c2; B.fshift = blk->shift;
  long long ab = (4ll * sm_count() + n - 1) / n;
  if (ab > max_b) ab = max_b;
  const dim3 agrid((unsigned)ab, n);
  __nv_bfloat16* dyp = reinterpret_cast<__nv_bfloat16*>(dy);
  const bool drop = blk->drop_p > 0.f;
  switch (co) {
#define UB_HEAD_K2(C_) case C_: \
    if (drop) head_bwd_apply_mma_kernel<C_, true><<<agrid, 256, 0, st>>>(dout, yp, dyp, T, (uint32_t)voxels, B); \
    else head_bwd_apply_mma_kernel<C_, false><<<agrid, 256, 0, st>>>(dout, yp, dyp, T, (uint32_t)voxels, B); \
    break;
    UB_HEAD_K2(1) UB_HEAD_K2(2) UB_HEAD_K2(3) UB_HEAD_K2(4) UB_HEAD_K2(5) UB_HEAD_K2(6) UB_HEAD_K2(7) UB_HEAD_K2(8)
#undef UB_HEAD_K2
  }
  UB_LAUNCH_CHECK();
  return 0;
}

// --------------------------------------------------------------------------------------------------
// N3: multi-tensor AdamW (ref:src/model.py:359-361); N4: de-normalised volume in NIfTI storage order
// --------------------------------------------------------------------------------------------------
extern "C" int ub_adamw_step(const ub_adamw_tensor* tensors, int count, double lr, double beta1, double beta2, double eps,
                             double weight_decay, long long step, float grad_scale, void* stream) {
  if (count < 0 || (count > 0 && !tensors) || step < 1) return fail(-1, "bad arguments to ub_adamw_step");
  if (!(beta1 >= 0.0 && beta1 < 1.0 && beta2 >= 0.0 && beta2 < 1.0 && eps >= 0.0 && lr >= 0.0))
    return fail(-1, "ub_adamw_step: invalid hyper-parameters");
  const double bc1 = 1.0 - pow(beta1, (double)step);
  const double bc2 = 1.0 - pow(beta2, (double)step);
  AdamWBatch B;
  B.beta2 = (float)beta2; B.one_minus_beta1 = (float)(1.0 - beta1); B.one_minus_beta2 = (float)(1.0 - beta2);
  B.eps = (float)eps;
  B.decay_mul = (float)(1.0 - lr * weight_decay);
  B.step_size = (float)(lr / bc1);
  B.bc2_sqrt = (float)sqrt(bc2);
  B.grad_scale = grad_scale;
  cudaStream_t st = (cudaStream_t)stream;
  int i = 0;
  while (i < count) {
    B.count = 0;
    B.block_begin[0] = 0;
    while (i < count && B.count < kAdamWMaxTensors) {
      const ub_adamw_tensor& t = tensors[i++];
      if (t.numel == 0) continue;
      if (!t.p || !t.g || !t.m || !t.v || t.numel < 0 || t.numel >= (1ll << 31))
        return fail(-1, "ub_adamw_step: tensor %d has a null pointer or an unsupported size", i - 1);
      const int k = B.count++;
      B.p[k] = t.p; B.g[k] = t.g; B.m[k] = t.m; B.v[k] = t.v;
      B.numel[k] = (int)t.numel;
      B.block_begin[k + 1] = B.block_begin[k] + (int)((t.numel + kAdamWChunk - 1) / kAdamWChunk);
    }
    if (B.count == 0) break;
    adamw_multi_kernel<<<(unsigned)B.block_begin[B.count], 256, 0, st>>>(B);
    UB_LAUNCH_CHECK();
  }
  return 0;
}

extern "C" int ub_bn_running_update(const float* mean, const float* rstd, int c, double count, float eps, float momentum,
                                    float* running_mean, float* running_var, void* stream) {
  if (!mean || !rstd || !running_mean || !running_var || c <= 0 || count <= 0.0) return fail(-1, "bad arguments to ub_bn_running_update");
  bn_running_update_kernel<<<(unsigned)((c + 127) / 128), 128, 0, (cudaStream_t)stream>>>(mean, rstd, c, count, eps, momentum,
                                                                                      running_mean, running_var);
  UB_LAUNCH_CHECK();
  return 0;
}

extern "C" int ub_denorm_to_nifti(const float* src, int c, int x, int y, int z, double scale, double offset, float* dst,
                                  void* stream) {
  if (!src || !dst || c <= 0 || x <= 0 || y <= 0 || z <= 0) return fail(-1, "bad arguments to ub_denorm_to_nifti");
  if ((long long)c * y > 65535) return fail(-2, "ub_denorm_to_nifti: channels x Y must not exceed 65535");
  const dim3 grid((unsigned)((z + 31) / 32), (unsigned)((x + 31) / 32), (unsigned)(c * y));
  denorm_to_nifti_kernel<<<grid, dim3(32, 8), 0, (cudaStream_t)stream>>>(src, dst, x, y, z, scale, offset);
  UB_LAUNCH_CHECK();
  return 0;
}

// --------------------------------------------------------------------------------------------------
// fp32 mode (CUDA-core kernels, NCDHW fp32 tensors): verification path, 1e-5 against the reference
// --------------------------------------------------------------------------------------------------
static int f32_geom(const ub_f32_conv_desc* d, f32::ConvGeom* G) {
  if (!d) return fail(-1, "null fp32 conv descriptor");
  if (d->n <= 0 || d->c0 <= 0 || d->c1 < 0 || d->co <= 0 || d->d <= 0 || d->h <= 0 || d->w <= 0)
    return fail(-1, "fp32 conv: non-positive size");
  if (!((d->k == 1 && d->stride == 1 && d->pad == 0) || (d->k == 3 && d->stride == 1 && d->pad == 1) ||
        (d->k == 4 && d->stride == 2 && d->pad == 1)))
    return fail(-2, "fp32 conv supports (k,s,p) = (1,1,0), (3,1,1), (4,2,1); got (%d,%d,%d)", d->k, d->stride, d->pad);
  G->n = d->n; G->c0 = d->c0; G->c1 = d->c1; G->co = d->co; G->d = d->d; G->h = d->h; G->w = d->w;
  G->k = d->k; G->s = d->stride; G->p = d->pad;
  G->od = (d->d + 2 * d->pad - d->k) / d->stride + 1;
  G->oh = (d->h + 2 * d->pad - d->k) / d->stride + 1;
  G->ow = (d->w + 2 * d->pad - d->k) / d->stride + 1;
  if (G->od <= 0 || G->oh <= 0 || G->ow <= 0) return fail(-2, "fp32 conv: input smaller than the kernel");
  return 0;
}
static unsigned f32_blocks(long long total) { return (unsigned)((total + 255) / 256); }
#define UB_F32_TOTAL_CHECK(t) if ((t) <= 0 || (t) >= (1ll << 39)) return fail(-2, "fp32 path: tensor too large")

extern "C" int ub_f32_conv_fwd(const ub_f32_conv_desc* d, const float* src0, const float* src1, const float* w,
                               const float* bias, float* out, void* stream) {
  f32::ConvGeom G;
  if (int e = f32_geom(d, &G)) return e;
  if (!src0 || !w || !out || (G.c1 > 0 && !src1)) return fail(-1, "bad arguments to ub_f32_conv_fwd");
  const long long total = (long long)G.n * G.co * G.od * G.oh * G.ow;
  UB_F32_TOTAL_CHECK(total);
  f32::conv_fwd_kernel<<<f32_blocks(total), 256, 0, (cudaStream_t)stream>>>(src0, src1, w, bias, out, G, total);
  UB_LAUNCH_CHECK();
  return 0;
}

extern "C" int ub_f32_conv_dgrad(const ub_f32_conv_desc* d, const float* dout, const float* w, float* dsrc0, float* dsrc1,
                                 void* stream) {
  f32::ConvGeom G;
  if (int e = f32_geom(d, &G)) return e;
  if (!dout || !w || !dsrc0 || (G.c1 > 0 && !dsrc1)) return fail(-1, "bad arguments to ub_f32_conv_dgrad");
  const long long total = (long long)G.n * (G.c0 + G.c1) * G.d * G.h * G.w;
  UB_F32_TOTAL_CHECK(total);
  f32::conv_dgrad_kernel<<<f32_blocks(total), 256, 0, (cudaStream_t)stream>>>(dout, w, dsrc0, dsrc1, G, total);
  UB_LAUNCH_CHECK();
  return 0;
}

extern "C" int ub_f32_conv_wgrad(const ub_f32_conv_desc* d, const float* src0, const float* src1, const float* dout,
                                 float* dw, float* dbias, void* stream) {
  f32::ConvGeom G;
  if (int e = f32_geom(d, &G)) return e;
  if (!dout || (dw && (!src0 || (G.c1 > 0 && !src1)))) return fail(-1, "bad arguments to ub_f32_conv_wgrad");
  cudaStream_t st = (cudaStream_t)stream;
  if (dw) {
    const dim3 grid((unsigned)(G.co * (G.c0 + G.c1)), (unsigned)G.k);
    if (G.k == 1) f32::conv_wgrad_kernel<1><<<grid, 128, 0, st>>>(src0, src1, dout, dw, G);
    else if (G.k == 3) f32::conv_wgrad_kernel<3><<<grid, 128, 0, st>>>(src0, src1, dout, dw, G);
    else f32::conv_wgrad_kernel<4><<<grid, 128, 0, st>>>(src0, src1, dout, dw, G);
    UB_LAUNCH_CHECK();
  }
  if (dbias) {
    f32::channel_sum_kernel<<<(unsigned)G.co, 256, 0, st>>>(dout, G.n, G.co, (long long)G.od * G.oh * G.ow, dbias);
    UB_LAUNCH_CHECK();
  }
  return 0;
}

extern "C" int ub_f32_deconv2_fwd(int n, int ci, int co, int d, int h, int w, const float* src, const float* wt,
                                  const float* bias, float* out, void* stream) {
  if (!src || !wt || !out || n <= 0 || ci <= 0 || co <= 0 || d <= 0 || h <= 0 || w <= 0) return fail(-1, "bad arguments to ub_f32_deconv2_fwd");
  const long long total = (long long)n * co * 8 * d * h * w;
  UB_F32_TOTAL_CHECK(total);
  f32::deconv2_fwd_kernel<<<f32_blocks(total), 256, 0, (cudaStream_t)stream>>>(src, wt, bias, out, n, ci, co, d, h, w, total);
  UB_LAUNCH_CHECK();
  return 0;
}

extern "C" int ub_f32_deconv2_dgrad(int n, int ci, int co, int d, int h, int w, const float* dout, const float* wt,
                                    float* dsrc, void* stream) {
  if (!dout || !wt || !dsrc || n <= 0 || ci <= 0 || co <= 0 || d <= 0 || h <= 0 || w <= 0) return fail(-1, "bad arguments to ub_f32_deconv2_dgrad");
  const long long total = (long long)n * ci * d * h * w;
  UB_F32_TOTAL_CHECK(total);
  f32::deconv2_dgrad_kernel<<<f32_blocks(total), 256, 0, (cudaStream_t)stream>>>(dout, wt, dsrc, n, ci, co, d, h, w, total);
  UB_LAUNCH_CHECK();
  return 0;
}

extern "C" int ub_f32_deconv2_wgrad(int n, int ci, int co, int d, int h, int w, const float* src, const float* dout,
                                    float* dw, float* dbias, void* stream) {
  if (!dout || (dw && !src) || n <= 0 || ci <= 0 || co <= 0 || d <= 0 || h <= 0 || w <= 0) return fail(-1, "bad arguments to ub_f32_deconv2_wgrad");
  cudaStream_t st = (cudaStream_t)stream;
  if (dw) {
    f32::deconv2_wgrad_kernel<<<(unsigned)(ci * co), 128, 0, st>>>(src, dout, dw, n, ci, co, d, h, w);
    UB_LAUNCH_CHECK();
  }
  if (dbias) {
    f32::channel_sum_kernel<<<(unsigned)co, 256, 0, st>>>(dout, n, co, (long long)8 * d * h * w, dbias);
    UB_LAUNCH_CHECK();
  }
  return 0;
}

extern "C" int ub_f32_norm_stats(const float* y, int n, int c, long long voxels, int mode, const float* gamma,
                                 const float* beta, float eps, float momentum, float* running_mean, float* running_var,
                                 float* scale, float* shift, float* mean, float* rstd, void* stream) {
  if (!y || !scale || !shift || !mean || !rstd || n <= 0 || c <= 0 || voxels <= 0 || mode < 0 || mode > 2)
    return fail(-1, "bad arguments to ub_f32_norm_stats");
  if (mode == UB_NORM_BATCH_EVAL && (!running_mean || !running_var)) return fail(-1, "eval BatchNorm needs running statistics");
  f32::norm_stats_kernel<<<(unsigned)c, 256, 0, (cudaStream_t)stream>>>(y, n, c, voxels, mode, gamma, beta, eps, momentum,
                                                                        running_mean, running_var, scale, shift, mean, rstd);
  UB_LAUNCH_CHECK();
  return 0;
}

static uint32_t f32_drop_thresh(float p) {
  double t = (double)p * 4294967296.0;
  return t >= 4294967295.0 ? 4294967295u : (uint32_t)t;
}

extern "C" int ub_f32_norm_act_fwd(const float* y, const float* scale, const float* shift, float slope, float drop_p,
                                   uint32_t drop_seed, int n, int c, int d, int h, int w, float* a, float* pooled,
                                   void* stream) {
  if (!y || !a || n <= 0 || c <= 0 || d <= 0 || h <= 0 || w <= 0 || drop_p < 0.f || drop_p >= 1.f || (scale && !shift))
    return fail(-1, "bad arguments to ub_f32_norm_act_fwd");
  cudaStream_t st = (cudaStream_t)stream;
  const long long vol = (long long)d * h * w, total = (long long)n * c * vol;
  UB_F32_TOTAL_CHECK(total);
  f32::norm_act_fwd_kernel<<<f32_blocks(total), 256, 0, st>>>(y, scale, shift, slope, drop_p, drop_seed,
                                                              f32_drop_thresh(drop_p), vol, total, a);
  UB_LAUNCH_CHECK();
  if (pooled) {
    const long long pt = (long long)n * c * (d / 2) * (h / 2) * (w / 2);
    if (pt <= 0) return fail(-2, "MaxPool3d(2) needs every spatial size >= 2");
    f32::maxpool_fwd_kernel<<<f32_blocks(pt), 256, 0, st>>>(a, pooled, d, h, w, pt);
    UB_LAUNCH_CHECK();
  }
  return 0;
}

extern "C" int ub_f32_norm_act_bwd(const float* dA, const float* dP, const float* a, const float* y, int mode,
                                   const float* mean, const float* rstd, const float* scale, const float* shift,
                                   float slope, float drop_p, uint32_t drop_seed, int n, int c, int d, int h, int w,
                                   float* c1c2, float* dy, float* dgamma, float* dbeta, void* stream) {
  if ((!dA && !dP) || !dy || n <= 0 || c <= 0 || d <= 0 || h <= 0 || w <= 0) return fail(-1, "bad arguments to ub_f32_norm_act_bwd");
  const bool has_norm = mode != UB_NORM_NONE;
  if (has_norm && (!y || !mean || !rstd || !scale || !shift || !c1c2)) return fail(-1, "ub_f32_norm_act_bwd: norm modes need y, statistics and the c1c2 workspace");
  if ((dP || (!has_norm && slope != 1.f)) && !a) return fail(-1, "ub_f32_norm_act_bwd: the activations a are required");
  cudaStream_t st = (cudaStream_t)stream;
  const long long vol = (long long)d * h * w, total = (long long)n * c * vol;
  UB_F32_TOTAL_CHECK(total);
  f32::act_bwd_kernel<<<f32_blocks(total), 256, 0, st>>>(dA, dP, a, y, has_norm ? scale : nullptr, shift, slope, drop_p,
                                                         drop_seed, f32_drop_thresh(drop_p), d, h, w, total, dy);
  UB_LAUNCH_CHECK();
  if (!has_norm) return 0;
  float* c1 = c1c2;
  float* c2 = c1c2 + (size_t)n * c;
  f32::norm_bwd_reduce_kernel<<<(unsigned)c, 256, 0, st>>>(dy, y, mean, rstd, n, c, vol, mode, c1, c2, dgamma, dbeta);
  UB_LAUNCH_CHECK();
  f32::norm_bwd_apply_kernel<<<f32_blocks(total), 256, 0, st>>>(dy, y, mean, rstd, scale, c1, c2, vol, total);
  UB_LAUNCH_CHECK();
  return 0;
}
