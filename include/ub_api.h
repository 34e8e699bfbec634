/* libubssfp -- C ABI of the B200-native hot path of SomeUserName1/UNet-bSSFP.
 *
 * The reference has no FFI: the seam is Python class identity (Generator / Discriminator /
 * DownSampleConv / BasicUNet / L1Loss / BCEWithLogitsLoss, ref:src/model.py:15-92,126,155) and the
 * NumPy arithmetic of eval.py (ref:src/eval.py:154-166,217-258). This header is the C boundary a
 * drop-in replacement exports for that path (SURVEY.md section 8b); each entry names the reference
 * op it replaces. Conventions:
 *   - plain C: pointers + sizes, no C++/torch types, no exceptions;
 *   - every entry returns 0 on success, <0 on error; ub_last_error() gives the thread-local message;
 *   - the caller owns ALL device memory (activations, workspaces, outputs);
 *   - all work is enqueued on the caller's cudaStream_t (passed as void*); no internal sync;
 *   - activations and gradients are NDHWC bf16 with the channel count padded to a multiple of 32 ("cp");
 *     the RAW output y of a conv that feeds a normalisation (ub_conv_fwd with stats_partial != NULL) is
 *     NDHWC IEEE fp16 -- it is never a tensor-core operand, only the input of the norm/activation kernels
 *     and of the deferred-activation operand transforms -- so activations are rounded to bf16 once;
 *     tensors at the module boundary are NCDHW fp32 as in the reference;
 *   - there is no CPU fallback and no cuDNN dispatch: an unsupported shape is an error.
 */
#ifndef UB_API_H_
#define UB_API_H_
#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

int ub_version(void);
const char* ub_last_error(void);
/* number of CUDA kernels this library has launched in the process (bench.py reports the delta) */
long long ub_launch_count(void);

/* ---- convolution family ------------------------------------------------------------------ */
enum {
  UB_CONV_K3S1P1 = 0,   /* nn.Conv3d(k=3,s=1,p=1): monai BasicUNet Convolution, ref:model.py:22-28 */
  UB_CONV_K1 = 1,       /* nn.Conv3d(k=1): input heads ref:model.py:19-21, final convs ref:model.py:83 */
  UB_CONV_K4S2P1 = 2,   /* nn.Conv3d(k=4,s=2,p=1): DownSampleConv in the PatchGAN, ref:model.py:50,72-82 */
  UB_DECONV_K2S2 = 3,   /* nn.ConvTranspose3d(k=2,s=2): monai UpSample "deconv" in UpCat */
  UB_CONV_K4S2P1_S2D = 4 /* UB_CONV_K4S2P1 whose source is the space-to-depth layout written by
                            ub_pack_ncdhw_s2d ([n][(pd,ph,pw)][d/2][h/2][w/2][c0p]): the PatchGAN stem d1,
                            ref:model.py:72-73,86. n,d,h,w / c0,c0p describe the ORIGINAL input; the
                            gradient written by ub_conv_dgrad is in the plain NDHWC layout */
};

typedef struct {
  int kind;        /* UB_CONV_* */
  int n, d, h, w;  /* batch and spatial size of the forward INPUT activation */
  int c0, c0p;     /* real / padded channels of input source 0 */
  int c1, c1p;     /* real / padded channels of input source 1 (skip concat [src0, src1]); 0 = none */
  int co, cop;     /* real / padded output channels */
} ub_conv_desc;

/* number of bf16 elements of a packed weight buffer; dir 0 = forward, 1 = dgrad */
long long ub_packed_weight_elems(const ub_conv_desc* d, int dir);
/* OR-ed into `dir` of the pack calls: the K columns of source 0 are written as fp16 (see ub_deferred_act.f16_operand) */
#define UB_PACK_F16_SRC0 2
/* torch-layout fp32 weights ([co][ci][k..] or [ci][co][2][2][2] for the transposed conv) -> packed bf16 */
int ub_pack_conv_weights(const ub_conv_desc* d, int dir, const float* w, void* packed, void* stream);
/* the same for `count` weights in as few launches as the pointer table allows (`items` is a HOST array; only kind
 * and the channel fields of desc are used). The modules re-pack every weight of a network at the start of each
 * forward / backward pass from the live fp32 Parameters (~25 us for the generator), so no cached operand copy can
 * go stale behind an out-of-band write to parameter memory. */
typedef struct {
  ub_conv_desc desc;
  int dir;
  const float* w;
  void* packed;
} ub_weight_pack_item;
int ub_pack_conv_weights_multi(const ub_weight_pack_item* items, int count, void* stream);

/* number of output tiles of the forward launch == rows of the statistics partial buffer */
int ub_conv_num_tiles(const ub_conv_desc* d);
/* A DEFERRED ACTIVATION: the activations a = LeakyReLU_slope(Dropout_p(y * scale + shift)) of a
 * conv -> norm -> dropout -> LeakyReLU block (monai Convolution -> ADN("NDA"), ref:model.py:22-28), given by the
 * block's raw conv output y (NDHWC fp16, 32 padded channels) and these constants instead of a materialised
 * tensor. Consumers that accept one apply it on their operand path (in shared memory between the TMA arrival
 * and the tcgen05.mma for the convolutions, in registers for the memory-bound kernels), so the tensor `a` is
 * never written to or read from HBM. All consumers evaluate the same function bit for bit. */
typedef struct {
  const float* scale;      /* [n][32] gamma * rstd   (ub_norm_finalize) */
  const float* shift;      /* [n][32] */
  float slope, drop_p;
  uint32_t drop_seed;
  int f16_operand;         /* ub_conv_fwd only: evaluate the activations in packed fp16 arithmetic and multiply them
                              as an fp16 x fp16 tensor-core operand (three instructions per element pair instead of the
                              fp32 path's conversions; relative error ~3 * 2^-12, below bf16 rounding). The weights
                              must be packed with UB_PACK_F16_SRC0. For passes without a backward (inference, the
                              generator forward of the discriminator phase): a backward would need the bf16 form. */
} ub_deferred_act;
/* 1 when source 0 of this convolution may be a deferred activation in ub_conv_fwd AND ub_conv_wgrad (3x3x3 convs
 * with 32 output channels and a 32-channel source 0: the full-resolution layers), else 0 */
int ub_conv_deferred_src0_ok(const ub_conv_desc* d);
/* out = conv(cat[src0, src1]) + bias; optional LeakyReLU; optional per-tile sum / sumsq partials
 * stats_partial: [ub_conv_num_tiles][2][cop] floats or NULL. With stats_partial the output is the raw input y of
 * a normalisation and is written as fp16 (statistics from the fp32 accumulators); otherwise bf16.
 * src0_act != NULL: src0 points at the producer's y (fp16) and is a deferred activation. */
/* src0_f16 != 0: src0 is a MATERIALISED fp16 activation tensor (ub_norm_act_fwd's a_f16 output) and the weights were
 * packed with UB_PACK_F16_SRC0: its K chunks run as fp16 x fp16 MMAs into the same fp32 accumulators (the forward
 * pass then carries 1/8 of bf16's operand rounding on those layers). Same availability as a deferred source. */
int ub_conv_fwd(const ub_conv_desc* d, const void* src0, const void* src1, const void* w_packed,
                const float* bias, int act, float slope, void* out, float* stats_partial,
                const ub_deferred_act* src0_act, int src0_f16, void* stream);
/* d src = conv_transpose(dy); dsrc1 may be NULL when the op has one source */
int ub_conv_dgrad(const ub_conv_desc* d, const void* dy, const void* w_packed_dgrad, void* dsrc0,
                  void* dsrc1, void* stream);
/* Optional epilogue fusion of ub_conv_dgrad_fused: dsrc0 is the gradient dA of the activations of a
 * conv -> norm -> dropout -> LeakyReLU block (the "producer"); while writing it the epilogue also
 * accumulates that block's norm-backward reductions S1 = sum dz, S2 = sum dz * xhat per (n, c), with
 * dz = dA * lrelu'(y * scale + shift) * dropout_mask / (1 - p), into per-CTA records
 * partial[ub_conv_dgrad_fuse_records(desc)][2][32]. Pass them to ub_norm_act_bwd (ext_partial) and its
 * reduction pass over dA and y is skipped. Available where ub_conv_dgrad_fuse_records() > 0 (3x3x3
 * convs with one 32-channel source, i.e. the full-resolution layers). */
typedef struct {
  const void* y;           /* producer's raw conv output, NDHWC fp16, 32 channels */
  const float* scale;      /* [n][32] gamma * rstd          (ub_norm_finalize) */
  const float* shift;      /* [n][32] */
  const float* mean;       /* [n][32] */
  const float* rstd;       /* [n][32] */
  float slope, drop_p;
  uint32_t drop_seed;
  float* partial;          /* out: [records][2][32] */
} ub_norm_bwd_fuse;
int ub_conv_dgrad_fuse_records(const ub_conv_desc* d);   /* records (n-major, records / n per sample); 0 = unsupported */
int ub_conv_dgrad_fused(const ub_conv_desc* d, const void* dy, const void* w_packed_dgrad, void* dsrc0,
                        void* dsrc1, const ub_norm_bwd_fuse* fuse, void* stream);
/* which kernel serves (desc, dir), dir 0 forward / 1 dgrad / 2 wgrad: 0 igemm_fwd_kernel (generic tap-table
 * implicit GEMM), 1 igemm_march_kernel, 2 wgrad_march_kernel, 3 igemm_wgrad_kernel (profiling / roofline tables) */
int ub_conv_kernel_class(const ub_conv_desc* d, int dir);
/* dw (fp32, torch layout) = sum_voxels src (x) dy; workspace holds the split-K partials */
long long ub_conv_wgrad_workspace_bytes(const ub_conv_desc* d);
/* src0_act != NULL: src0 points at the producer's y (fp16) and is a deferred activation (ub_conv_deferred_src0_ok) */
int ub_conv_wgrad(const ub_conv_desc* d, const void* src0, const void* src1, const void* dy,
                  void* workspace, float* dw, const ub_deferred_act* src0_act, void* stream);

/* ---- layout at the module boundary --------------------------------------------------------- */
/* cat[a (ca ch), b (cb ch)] NCDHW fp32 -> NDHWC bf16 with cp channels (b may be NULL); replaces the
 * torch.cat of ref:model.py:86 and Lightning's host tensor layout. a_bf16 != 0: `a` is NCDHW bf16 (a loader that
 * ships the conditioning input in bf16 halves its host-to-device bytes; the result is bit-identical because fp32
 * inputs are rounded to bf16 by this very kernel) */
int ub_pack_ncdhw(const void* a, int a_bf16, int ca, const float* b, int cb, int n, long long voxels, int cp,
                  void* out, void* stream);
/* same, but the destination is the parity-planar space-to-depth layout
 * [n][(pd,ph,pw)][d/2][h/2][w/2][cp] (eight dense half-resolution sub-volumes per sample) read by
 * UB_CONV_K4S2P1_S2D (the PatchGAN stem d1, ref:model.py:72-73,86); d, h, w must be even */
int ub_pack_ncdhw_s2d(const void* a, int a_bf16, int ca, const float* b, int cb, int n, int d, int h, int w, int cp,
                      void* out, void* stream);
/* NDHWC bf16 (n, d, h, w, cp) -> the same tensor in the parity-planar space-to-depth layout
 * [n][(pd,ph,pw)][d/2][h/2][w/2][cp] (a permuting copy; d, h, w even). The PatchGAN body d2 .. d5 (ref:model.py:74-82)
 * reads its input this way through UB_CONV_K4S2P1_S2D instead of strided TMA boxes. */
int ub_to_s2d(const void* src, int n, int d, int h, int w, int cp, void* dst, void* stream);
/* Sliding-window inference (ref:model.py:315-333, ref:data_module.py:168-183; torchio==0.19.6
 * GridSampler / GridAggregator, any patch_overlap). ub_pack_patches gathers n (<= 64) d x h x w patches of
 * an NCDHW fp32 volume into one NDHWC bf16 batch: patch i starts at element offsets[i] (HOST array) of `a`,
 * its element (c,z,y,x) is at + c*stride_c + z*stride_d + y*stride_h + x. ub_unpack_patch writes channels
 * [c_begin, c_begin+c) of batch sample `sample` into the volume region at dst + dst_offset (same
 * addressing); calling it in sampler order reproduces "the later patch wins". */
int ub_pack_patches(const float* a, int ca, int n, const long long* offsets, int d, int h, int w,
                    long long stride_c, long long stride_d, long long stride_h, int cp, void* out, void* stream);
int ub_unpack_patch(const void* src, int cp, int c_begin, int c, int sample, int d, int h, int w, float* dst,
                    long long dst_offset, long long stride_c, long long stride_d, long long stride_h, void* stream);
/* the same aggregation for an NCDHW fp32 patch [c][d][h][w] (the output of ub_conv1x1_to_ncdhw) */
int ub_paste_patch(const float* src, int c, int d, int h, int w, float* dst, long long dst_offset,
                   long long stride_c, long long stride_d, long long stride_h, void* stream);
/* GridAggregator.add_batch for one batch of n (<= 64) NCDHW fp32 patches src [n][c <= 8][pd][ph][pw], in sampler
 * order, in ONE launch. origins (HOST, [n][3]): patch origins (z, y, x) in the volume; boxes (HOST, [n][6] z0 y0 x0
 * z1 y1 x1, half-open, inside the patch; NULL = the whole patch): the region each patch writes. out [c][d][h][w] and
 * weight [d][h][w] are contiguous fp32 volumes. mode 0 'crop': the last patch whose box holds a voxel is assigned
 * (weight unused); mode 1 'average': out += p, weight += 1; mode 2 'hann': out += p * w, weight += w with
 * w = (wz[z] * wy[y]) * wx[x] read from window (DEVICE, pd + ph + pw floats: wz, wy, wx). Each voxel sums its
 * patches in order with separately rounded fp32 multiplies and adds, so launches in sampler order reproduce
 * torchio's tensors bit for bit. ub_blend_finish: out /= weight (every channel) after the last batch. */
int ub_blend_patches(const float* src, int n, int c, int pd, int ph, int pw, const int* origins, const int* boxes,
                     int mode, const float* window, float* out, float* weight, int d, int h, int w, void* stream);
int ub_blend_finish(float* out, const float* weight, int c, long long voxels, void* stream);
/* NDHWC bf16 (cp channels) -> NCDHW fp32, channels [c_begin, c_begin + c) */
int ub_unpack_ncdhw(const void* src, int cp, int c_begin, int c, int n, long long voxels, float* out,
                    void* stream);

/* ---- output head: 1x1x1 conv to <= 8 channels fused with the layout change ------------------------- */
/* monai BasicUNet.final_conv = nn.Conv3d(32, 6, 1) (ref:model.py:22-28) followed by the module boundary:
 * out (NCDHW fp32 [n][co][voxels]) = W u + b straight from the NDHWC bf16 activations u (cp = 32), instead of a
 * padded 32-channel bf16 tensor + unpack. w [co][ci] / bias [co] are the fp32 parameters (device pointers).
 * workspace: ub_conv1x1_workspace_bytes() bytes. */
long long ub_conv1x1_workspace_bytes(void);
/* u_act != NULL (both calls): u points at the last block's y (fp16) and is a deferred activation */
int ub_conv1x1_to_ncdhw(const void* u, int cp, const float* w, int ci, const float* bias, int co, int n,
                        long long voxels, void* workspace, float* out, const ub_deferred_act* u_act, void* stream);
/* its backward in ONE pass over dout (NCDHW fp32) and u: du = W^T dout (NDHWC bf16, may be NULL),
 * dw [co][ci] = sum dout (x) u and db [co] = sum dout (fp32, may be NULL; u may be NULL when both are) */
int ub_conv1x1_from_ncdhw_bwd(const float* dout, int co, const void* u, int cp, const float* w, int ci, int n,
                              long long voxels, void* workspace, void* du, float* dw, float* db,
                              const ub_deferred_act* u_act, void* stream);
/* The backward of the head when its input is the DEFERRED activation of a conv -> norm -> dropout -> LeakyReLU block
 * (`blk`: that block's y (fp16, 32 channels), scale / shift / mean / rstd [n][32]; blk->partial is not used), fused
 * with that block's norm backward: returns the block's dy (NDHWC bf16) straight from dout, without materialising du
 * (two passes over dout and y instead of three passes over du, dA and y), plus the block's dgamma / dbeta / dbias
 * ([c], may be NULL) and the head's dw [co][ci] / db [co] (may be NULL). mode: UB_NORM_* of the block; c: its real
 * channels. voxels per sample must be a multiple of 16. workspace: ub_head_bwd_fused_workspace_bytes(n) bytes.
 * ref: monai BasicUNet.final_conv after upcat_1 (TwoConv -> ADN "NDA"), ref:model.py:22-28 */
long long ub_head_bwd_fused_workspace_bytes(int n);
int ub_head_bwd_fused(const float* dout, int co, const float* w, int ci, int n, long long voxels,
                      const ub_norm_bwd_fuse* blk, int mode, int c, void* workspace, void* dy, float* dgamma,
                      float* dbeta, float* dbias, float* dw, float* db, void* stream);

/* ---- normalisation + dropout + activation --------------------------------------------------- */
enum { UB_NORM_INSTANCE = 0, UB_NORM_BATCH_TRAIN = 1, UB_NORM_BATCH_EVAL = 2, UB_NORM_NONE = 3 };
/* InstanceNorm3d(affine) / BatchNorm3d statistics from the conv epilogue partials.
 * scale/shift/mean/rstd: [n][cp] floats. running_* updated in UB_NORM_BATCH_TRAIN (momentum 0.1,
 * unbiased variance), read in UB_NORM_BATCH_EVAL. ref: monai ADN "N"; ref:model.py:53-54 */
int ub_norm_finalize(const float* stats_partial, int tiles_per_sample, int n, int cp, int c,
                     double voxels_per_sample, const float* gamma, const float* beta, float eps, int mode,
                     float momentum, float* running_mean, float* running_var, float* scale, float* shift,
                     float* mean, float* rstd, void* stream);
/* BatchNorm running statistics from the batch statistics a UB_NORM_BATCH_TRAIN finalize saved (mean / rstd: the
 * first c entries of its outputs) when it was called with running_mean = running_var = NULL:
 * running = (1 - momentum) * running + momentum * {mean, unbiased variance}; count = n * voxels. Decouples the
 * update from the forward pass so that independent passes can run on different streams and still update in the
 * reference's order (ref:src/model.py:184-186: fake branch, then real branch). */
int ub_bn_running_update(const float* mean, const float* rstd, int c, double count, float eps, float momentum,
                         float* running_mean, float* running_var, void* stream);
/* a = LeakyReLU_slope(Dropout_p(y * scale + shift)); pooled (may be NULL) = MaxPool3d(2)(a). y is fp16, a and
 * pooled bf16. scale == NULL: no normalisation. a may be NULL when pooled or a_f16 is given (the activations stay
 * deferred / only the requested copies are materialised). ref: monai ADN "NDA" + Down.max_pooling */
/* a_f16 (may be NULL): the SAME fp32 values rounded to fp16 -- the operand copy for a forward conv called with
 * src0_f16 (the bf16 copy `a` is what the weight gradient needs; a pass without a backward writes only a_f16) */
int ub_norm_act_fwd(const void* y, const float* scale, const float* shift, float slope, float drop_p,
                    uint32_t drop_seed, int n, int d, int h, int w, int cp, void* a, void* a_f16, void* pooled,
                    void* stream);
long long ub_norm_act_bwd_workspace_bytes(int n, int cp);
/* backward of the block above: dy from dA; dgamma/dbeta/dbias (fp32 [c]) may be NULL.
 * mean == NULL (UB_NORM_NONE): plain activation backward (reads a).
 * shift != NULL (norm modes): the LeakyReLU branch is recomputed as sign(y * scale + shift) -- the
 * forward's own fma -- and `a` is not read (may be NULL): 10 instead of 14 bytes per element. */
int ub_norm_act_bwd(const void* dA, const void* a, const void* y, int mode, const float* mean,
                    const float* rstd, const float* scale, const float* shift, float slope, float drop_p,
                    uint32_t drop_seed,
                    int n, long long voxels, int cp, int c, void* workspace, void* dy, float* dgamma,
                    float* dbeta, float* dbias, const float* ext_partial, int ext_records_per_sample, void* stream);
/* ext_partial != NULL: per-sample partial records [n * ext_records_per_sample][2][cp] produced by
 * ub_conv_dgrad_fused replace the reduction pass. */
/* MaxPool3d(2) backward; accumulate != 0 adds onto the gradient already in dA (skip path).
 * a_act != NULL: `a` points at the block's y (fp16) and is a deferred activation */
int ub_maxpool_bwd(const void* a, const void* dP, void* dA, int accumulate, int n, int d, int h, int w,
                   int cp, const ub_deferred_act* a_act, void* stream);
/* The same routing for a conv -> norm -> dropout -> LeakyReLU block whose dA is COMPLETE after this pass (skip
 * gradient + routed pool gradient: the second conv of every encoder level), fused with that block's norm-backward
 * reduction: the activations are recomputed from fuse->y (cp channels here, constants [n][cp]) and the kernel also
 * accumulates S1 / S2 (see ub_norm_bwd_fuse) into fuse->partial[ub_maxpool_bwd_fuse_records()][2][cp]; pass them to
 * ub_norm_act_bwd as ext_partial. ref: monai Down = MaxPool3d(2) + TwoConv, ref:model.py:22-28 */
int ub_maxpool_bwd_fuse_records(int n, int d, int h, int w, int cp);   /* n-major; 0 = unsupported shape */
int ub_maxpool_bwd_fused(const void* dP, void* dA, int accumulate, int n, int d, int h, int w, int cp,
                         const ub_norm_bwd_fuse* fuse, void* stream);
/* out[c] = sum over rows of x[rows][cp] (bias gradients of convs without a following norm) */
long long ub_colsum_workspace_bytes(int cp);
int ub_colsum(const void* x, long long rows, int cp, int c, void* workspace, float* out, void* stream);

/* ---- losses -------------------------------------------------------------------------------------- */
long long ub_l1_workspace_bytes(void);
/* nn.L1Loss (mean), ref:model.py:126,136 */
int ub_l1_fwd(const float* a, const float* b, long long numel, void* workspace, float* loss, void* stream);
int ub_l1_bwd(const float* a, const float* b, const float* grad_out, long long numel, float* da, void* stream);
/* nn.BCEWithLogitsLoss (mean), ref:model.py:155,173-175,187-192. target: per-element tensor, or NULL
 * to use target_const (the reference only ever passes all-ones / all-zeros);
 * dx_unit (may be NULL) = d loss / d x for an upstream gradient of 1 */
int ub_bce_logits(const float* x, const float* target, float target_const, int numel, float* loss,
                  float* dx_unit, void* stream);
int ub_scale(const float* x, const float* scalar, long long numel, float* y, void* stream);

/* ---- evaluation -------------------------------------------------------------------------------- */
/* ref:eval.py:154-166 (relative / angular error map) fused with ref:eval.py:217-258 (masked,
 * probseg-weighted ROI means). Volumes are channel-last [X][Y][Z][C] fp32. diff, mask, probseg may be
 * NULL. sums: [r][c] doubles, norms: [r] doubles (zeroed by the call). c <= 8, r <= 3. */
int ub_relerr_map_reduce(const float* pred, const float* target, const unsigned char* mask,
                         const float* probseg, int c, int r, long long voxels, int angular, float* diff,
                         double* sums, double* norms, void* stream);

/* ref:eval.py:73-116 (do_calc_scalar_maps): per-voxel symmetric 3x3 eigen-decomposition of the diffusion
 * tensor (channel-last [voxels][6] = dxx,dxy,dxz,dyy,dyz,dzz, fp32) and the derived maps FA, MD, AD, RD
 * ([voxels]), azimuth / inclination of the principal axis in degrees ([voxels]) and the FA-weighted RGB map
 * ([voxels][3]). Any output may be NULL. Arithmetic in fp64 like the reference. The principal eigenvector is
 * oriented with v_z >= 0 (LAPACK leaves the sign implementation-defined). */
int ub_dti_scalar_maps(const float* tensor6, long long voxels, float* fa, float* md, float* ad, float* rd,
                       float* azimuth, float* inclination, float* rgb, void* stream);

/* ---- optimiser (SURVEY.md 8f N3) ------------------------------------------------------------------ */
/* torch.optim.AdamW (ref:src/model.py:144,164,359-361: lr 1e-3, betas (0.9, 0.999), eps 1e-8, weight decay 0.01)
 * over `count` parameter tensors in as few launches as the pointer table allows. `tensors` is a HOST array;
 * p / g / m / v are device pointers to fp32 arrays of numel elements (parameter, gradient, exp_avg, exp_avg_sq),
 * updated in place. step >= 1 is the number of this update (bias corrections 1 - beta^step, computed on the
 * host; the hyper-parameters are doubles because torch derives 1 - beta from Python floats). grad_scale multiplies the gradient first (1 / world_size after a SUM all-reduce; otherwise 1). */
typedef struct {
  float* p;
  const float* g;
  float* m;
  float* v;
  long long numel;
} ub_adamw_tensor;
int ub_adamw_step(const ub_adamw_tensor* tensors, int count, double lr, double beta1, double beta2, double eps,
                  double weight_decay, long long step, float grad_scale, void* stream);

/* ---- prediction volume -> NIfTI storage order (SURVEY.md 8f N4) ------------------------------------- */
/* ref:src/model.py:335-357 (save_predicitions: np.moveaxis(volume, 0, -1) -> Nifti1Image) followed by
 * ref:src/eval.py:39-47 (do_invert_dwi_tensor_norm: v * |max - min| + min in float64, stored as the header's
 * float32). src: one volume in module layout [c][x][y][z] fp32 (z fastest); dst: the data block of a NIfTI-1
 * file holding the channel-last array (x, y, z, c), i.e. [c][z][y][x] with x fastest. scale = 1, offset = 0
 * gives the plain layout change. */
int ub_denorm_to_nifti(const float* src, int c, int x, int y, int z, double scale, double offset, float* dst,
                       void* stream);

/* ---- fp32 mode ------------------------------------------------------------------------------------ */
/* north_star: "agree within 1e-2 relative (bf16) or 1e-5 (fp32 mode)". The same operators on the CUDA cores
 * (fp32 products, fp64 sums), tensors in the reference's own NCDHW fp32 layout with REAL channel counts and
 * torch weight layouts ([co][ci][k][k][k]; [ci][co][2][2][2] for the transposed conv). A verification path for
 * small volumes: no tensor cores, no roofline claim. */
typedef struct {
  int n, c0, c1, co;   /* batch; channels of source 0 / source 1 (skip concat [src0, src1], c1 = 0: none); output channels */
  int d, h, w;         /* input spatial size */
  int k, stride, pad;  /* (1,1,0), (3,1,1) or (4,2,1): the three Conv3d shapes of ref:model.py */
} ub_f32_conv_desc;
int ub_f32_conv_fwd(const ub_f32_conv_desc* d, const float* src0, const float* src1, const float* w, const float* bias,
                    float* out, void* stream);
int ub_f32_conv_dgrad(const ub_f32_conv_desc* d, const float* dout, const float* w, float* dsrc0, float* dsrc1,
                      void* stream);
/* dw and / or dbias may be NULL */
int ub_f32_conv_wgrad(const ub_f32_conv_desc* d, const float* src0, const float* src1, const float* dout, float* dw,
                      float* dbias, void* stream);
/* ConvTranspose3d(kernel 2, stride 2); d, h, w = INPUT spatial size */
int ub_f32_deconv2_fwd(int n, int ci, int co, int d, int h, int w, const float* src, const float* wt, const float* bias,
                       float* out, void* stream);
int ub_f32_deconv2_dgrad(int n, int ci, int co, int d, int h, int w, const float* dout, const float* wt, float* dsrc,
                         void* stream);
int ub_f32_deconv2_wgrad(int n, int ci, int co, int d, int h, int w, const float* src, const float* dout, float* dw,
                         float* dbias, void* stream);
/* statistics straight from y [n][c][voxels] (two passes, fp64); mode = UB_NORM_INSTANCE / BATCH_TRAIN / BATCH_EVAL;
 * scale / shift / mean / rstd: [n][c] */
int ub_f32_norm_stats(const float* y, int n, int c, long long voxels, int mode, const float* gamma, const float* beta,
                      float eps, float momentum, float* running_mean, float* running_var, float* scale, float* shift,
                      float* mean, float* rstd, void* stream);
/* a = LeakyReLU(Dropout(y * scale + shift)) (scale NULL: no norm); pooled (may be NULL) = MaxPool3d(2)(a) */
int ub_f32_norm_act_fwd(const float* y, const float* scale, const float* shift, float slope, float drop_p,
                        uint32_t drop_seed, int n, int c, int d, int h, int w, float* a, float* pooled, void* stream);
/* backward of the block above, including the max-pool routing: dA (gradient of a) and dP (gradient of pooled) may
 * each be NULL (not both). mode UB_NORM_NONE: activation backward only. c1c2: workspace of 2*n*c floats. */
int ub_f32_norm_act_bwd(const float* dA, const float* dP, const float* a, const float* y, int mode, const float* mean,
                        const float* rstd, const float* scale, const float* shift, float slope, float drop_p,
                        uint32_t drop_seed, int n, int c, int d, int h, int w, float* c1c2, float* dy, float* dgamma,
                        float* dbeta, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* UB_API_H_ */
