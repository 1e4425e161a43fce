/* mvtb.h — C ABI of libmvtb.so: B200 (sm_100a) kernels for the MRI artifact transforms of
 * yanielc/medical-vision-textural-bias.
 *
 * The reference is pure Python and has no FFI of its own; these entry points are what a
 * binding for its hot path (source_code/filters_and_operators.py = F, stylization_layers.py = S)
 * calls.  Each entry cites the reference routine whose arithmetic it replaces.
 *
 * Conventions
 *   - every function returns 0 (MVTB_OK) on success, a negative MVTB_E* code for argument
 *     errors, or a positive cudaError_t; nothing throws, nothing calls exit();
 *   - all work is enqueued asynchronously on the caller's stream (`stream` is a cudaStream_t
 *     passed as void*); plan_create/plan_destroy synchronise; a transform call blocks the host only when a workspace has to grow
 *     (first call of a plan on a larger batch) or a pinned staging slot is still in flight (INTEGRATION.md);
 *   - the caller owns every in/out/u/minmax device buffer; the plan owns its tables and
 *     workspace; a plan is used from one stream at a time;
 *   - tensors are contiguous row-major fp32; a "volume" is one block of the last `ndim_fft`
 *     axes (the unit the reference FFTs), e.g. one channel of a (C,H,W,D) sample for the
 *     3-D transforms, or one batch item (C,H,W,D) for the 4-D FFT of GibbsNoiseLayer.
 */
#ifndef MVTB_H
#define MVTB_H
#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MVTB_VERSION 200

#define MVTB_OK 0
#define MVTB_EINVAL (-1)        /* bad argument (null pointer, non-positive size, ...) */
#define MVTB_EUNSUPPORTED (-2)  /* shape / option outside what the kernels implement */
#define MVTB_ENOMEM (-3)
#define MVTB_ENODEVICE (-4)     /* no usable CUDA device: there is no CPU fallback */
#define MVTB_ETIMEOUT (-5)      /* a tensor-core kernel of an EARLIER call on this plan gave up on an mbarrier wait (that call's output is
                                   invalid); the plan has switched to the CUDA-core kernels.  Never seen outside a protocol bug. */

#define MVTB_MAX_FFT_DIMS 4
#define MVTB_MAX_SPIKES 8

/* mask_kind */
#define MVTB_MASK_NONE 0
/* keep  <=>  sum_d (i_d - floor(N_d/2))^2 <= mask_thresh   (disk_mask, F:165-197; the fp32
 * comparison `< r**2` is turned into this integer threshold on the host, SURVEY A.1) */
#define MVTB_MASK_DISK 1
/* keep  <=>  sum_d (2 i_d - (N_d-1))^2 <= mask_thresh   (GibbsNoise F:686-698 and
 * GibbsNoiseLayer S:99-109; i_d = fftshift-ed index; threshold found on the host by evaluating
 * the reference's own fp64 / fp32 predicate, which is monotone in the sum) */
#define MVTB_MASK_CENTRED 2
/* keep  <=>  mask_u[fftshift-ed index] > mask_p, mask_u a device array of the volume's full k-space shape: RandZF's
 * random zero-filling (50_reconstruction/reconGan/utils2.py:34-74: `mask = torch.rand(k.size()); k[mask <= p] = 0`).
 * The mask is not Hermitian; as for every mask the real part taken afterwards makes it (M(f) + M(-f)) / 2.  General
 * FFT path only; mask_ndim is ignored (the array covers all FFT axes). */
#define MVTB_MASK_UNIFORM 3

typedef struct mvtb_spike {
    int32_t idx[MVTB_MAX_FFT_DIMS]; /* fftshift-ed k-space index per FFT axis, outermost first
                                       (what the reference writes to: F:387, F:975-983) */
    float amplitude;                /* exp(log-intensity) in fp32 (F:389, F:942) */
    int32_t reserved;
} mvtb_spike;

/* One fused k-space pass:  out = Re ifftn( W * ( M * fftn(x) with spikes set ) )
 * = RandFourierDiskMaskd (F:236-252) / GibbsNoise (F:663-705) / GibbsNoiseLayer (S:79-116)
 *   -> RandPlaneWaves_ellipsoid (F:370-393) / KSpaceSpikeNoise (F:906-945)
 *   -> WrapArtifact (F:503-515), each stage optional, in that order. */
typedef struct mvtb_chain_desc {
    int32_t mask_kind;
    int32_t mask_ndim;     /* number of trailing axes in the distance (<= ndim_fft) */
    int64_t mask_thresh;   /* integer threshold; negative keeps nothing */
    int32_t inside_off;    /* 1: mask = 1 - mask (F:194-195) */
    int32_t n_spikes;      /* 0..MVTB_MAX_SPIKES, distinct locations */
    float wrap_alpha;      /* weight of odd fftshift-ed indices (F:509-511) */
    int32_t wrap_naxes;    /* 0 = no wrap; else the trailing wrap_naxes axes are weighted (3 in the reference) */
    mvtb_spike spikes[MVTB_MAX_SPIKES];
    const float* mask_u;   /* MVTB_MASK_UNIFORM: device pointer to this volume's uniform field (else NULL) */
    float mask_p;          /* MVTB_MASK_UNIFORM: threshold */
    int32_t reserved;
} mvtb_chain_desc;

typedef struct mvtb_plan mvtb_plan;

int mvtb_version(void);
/* copies the calling thread's last error text; returns its length */
int mvtb_last_error(char* buf, int n);

/* FFT plan over the last ndim_fft (2..4) axes, fft_shape outermost first.  chunk_volumes =
 * how many volumes are in flight between kernels (workspace = chunk_volumes half-spectra).
 * Every axis length must factor into primes <= 31 (240, 155, 128, 64, ... do). */
int mvtb_plan_create(mvtb_plan** out, int ndim_fft, const int* fft_shape, int chunk_volumes, int device);
int mvtb_plan_destroy(mvtb_plan* plan);
size_t mvtb_plan_workspace_bytes(const mvtb_plan* plan);

/* Fused chain over n_volumes volumes.  desc: host array of n_desc entries, n_desc == 1
 * (shared) or n_volumes.  minmax_out (nullable): device float[2*n_samples], receives
 * (min, max) of `out` per sample, a sample being vols_per_sample consecutive volumes
 * (what SaltAndPepper's x.min()/x.max() needs, F:476).  in == out is allowed. */
int mvtb_kspace_chain_f32(mvtb_plan* plan, const float* in, float* out, int n_volumes,
                          const mvtb_chain_desc* desc, int n_desc,
                          float* minmax_out, int vols_per_sample, void* stream);

/* mvtb_kspace_chain_f32 followed by mvtb_salt_pepper_sparse_f32(out, vols_per_sample * volume, n_volumes /
 * vols_per_sample samples, seed, offset, p, minmax_out): the whole 127-series chain (F:236-252 -> F:370-393 ->
 * F:503-515 -> F:465-482) in one call, with bit-identical results to the two calls.  When the mask keeps a small
 * ball (band-limited path) the select pass runs inside the inverse kernel, on output lines that are still in L2,
 * instead of as a second pass over HBM.  minmax_out (required): device float[2 * n_samples].  n_volumes must be a
 * multiple of vols_per_sample.  in == out is allowed. */
int mvtb_kspace_chain_sp_f32(mvtb_plan* plan, const float* in, float* out, int n_volumes,
                             const mvtb_chain_desc* desc, int n_desc, float* minmax_out, int vols_per_sample,
                             float p, uint64_t seed, uint64_t offset, void* stream);

/* The general form: optional intensity prologue map on the way in (pre_abt: device float[3 * n_volumes], one (a, b, t)
 * per volume from mvtb_intensity_prologue_coeffs_f32, y = x != 0 ? a x + b : t; NULL = none), the chain, and an
 * optional sparse salt-and-pepper pass on the way out (sp: NULL = none; then minmax_out may be NULL too).
 * mvtb_kspace_chain_f32 / _sp_f32 are this call with the corresponding arguments NULL. */
typedef struct mvtb_sp_params {
    float p;
    uint64_t seed, offset;
} mvtb_sp_params;
int mvtb_kspace_chain_ex_f32(mvtb_plan* plan, const float* in, float* out, int n_volumes,
                             const mvtb_chain_desc* desc, int n_desc, const float* pre_abt,
                             float* minmax_out, int vols_per_sample, const mvtb_sp_params* sp, void* stream);
/* mvtb_kspace_chain_ex_f32 with the distance between samples' Philox span counters set: span s of sample i uses counter
 * offset + i * sample_stride + s (0 = ceil(voxels per sample / MVTB_SP_SPAN), which is mvtb_kspace_chain_ex_f32; a nonzero
 * stride must not be below that span count).  One call over a batch then draws the hits that one call per sample would draw
 * with `offset` advanced by sample_stride between calls -- SaltAndPepper(rng="philox-sparse") advances it by
 * ceil(voxels / 256) per call.  The select pass runs where mvtb_kspace_chain_ex_f32 runs it (fused into the inverse kernel
 * when it can be). */
int mvtb_kspace_chain_ex_strided_f32(mvtb_plan* plan, const float* in, float* out, int n_volumes,
                                     const mvtb_chain_desc* desc, int n_desc, const float* pre_abt,
                                     float* minmax_out, int vols_per_sample, const mvtb_sp_params* sp,
                                     uint64_t sample_stride, void* stream);

/* sum over the full (unshifted, unnormalised) spectrum of log(|k| + 1e-10) per volume, into
 * device double[n_volumes]; the caller divides by the volume size and multiplies by 2.5
 * (KSpaceSpikeNoise default intensity F:932-933, RandKSpaceSpikeNoise default range F:1127-1130). */
int mvtb_kspace_logabs_sum_f32(mvtb_plan* plan, const float* in, int n_volumes, double* sums_out, void* stream);

/* (min, max) per sample of n_per_sample contiguous floats -> device float[2*n_samples] (F:476) */
int mvtb_minmax_f32(const float* in, size_t n_per_sample, int n_samples, float* minmax_out, void* stream);

/* SaltAndPepper.salt_and_pepper (F:465-482): y = u <= p/2 ? min/2 : (u <= p ? max/2 : x), with
 * (min,max) per sample read from minmax (device, from mvtb_minmax_f32 or the chain).
 * u: device uniforms of the same shape (bit-exact parity with the reference given its mask),
 * or NULL -> counter-based Philox4x32-10 keyed by `seed`, element i of the whole buffer uses
 * counter (offset + i/4), lane i%4.  in == out allowed. */
int mvtb_salt_pepper_f32(const float* in, float* out, size_t n_per_sample, int n_samples,
                         const float* u, uint64_t seed, uint64_t offset, float p,
                         const float* minmax, void* stream);

/* In-place salt-and-pepper whose cost is proportional to p: instead of one uniform per voxel, every span of
 * MVTB_SP_SPAN consecutive voxels of a sample is walked from hit to hit by one warp, with geometric gaps drawn from
 * Philox4x32-10 by inverse CDF against the integer table of mvtb_sparse_table (exact integer compares), plus one random
 * bit per hit for salt vs pepper.  The voxels hit are i.i.d. Bernoulli(p) exactly as with `u <= p`, and half of them get
 * min/2, half max/2 (F:478-479).  Deterministic in (seed, offset, p); a different random field than
 * mvtb_salt_pepper_f32's.  Span s of sample i uses the Philox counters (offset + i * ceil(n_per_sample / MVTB_SP_SPAN)
 * + s, ...): advance `offset` by at least n_samples * ceil(n_per_sample / MVTB_SP_SPAN) between calls.
 * table_dev: device scratch of MVTB_SP_BLOCK uint32 owned by the caller. */
#define MVTB_SP_BLOCK 256
#define MVTB_SP_SPAN 8192
int mvtb_salt_pepper_sparse_f32(float* x, size_t n_per_sample, int n_samples, uint64_t seed, uint64_t offset,
                                float p, const float* minmax, unsigned* table_dev, void* stream);
/* T[k] = floor(2^32 (1 - (1-p)^(k+1))), k < MVTB_SP_BLOCK (host memory) */
int mvtb_sparse_table(float p, unsigned* table_out);

/* the uniforms mvtb_salt_pepper_f32 uses when u == NULL (for tests and for feeding the oracle) */
int mvtb_philox_uniform_f32(float* out, size_t n, uint64_t seed, uint64_t offset, void* stream);

/* ---- intensity prologue: NormalizeIntensityd(nonzero=True, channel_wise=True) -> RandScaleIntensityd ->
 * RandShiftIntensityd, the MONAI 0.5 transforms in front of the chain in every training script of the reference
 * (10_scripts/127_.../stylized_gibbs12p5_spikes15_wrap0p5_sap0p05_FLAIR.py:134-136).  Per channel c with m = x != 0:
 *   y = m ? ((x - mean(x[m])) / std(x[m])) * scale[c] + shift[c] : shift[c]     (population std; 1 if it is 0)
 * mvtb_intensity_prologue_coeffs_f32: one read of the data -> stats_out[c] = (count, mean, std) (device double[3C],
 *   nullable) and abt_out[c] = (a, b, t) with y = m ? a x + b : t (device float[3C], nullable).  scale / shift: device
 *   float[C] (1 + factor and offset of the two random transforms; NULL = not applied).  scratch: device buffer of
 *   mvtb_intensity_scratch_bytes(C) bytes.  Deterministic (fixed-order reduction in double).
 * mvtb_intensity_affine_f32: the map on its own, in == out allowed.
 * mvtb_kspace_chain_ex_f32 (below) applies the map while the chain reads the volume (one triple per volume). */
size_t mvtb_intensity_scratch_bytes(int n_channels);
int mvtb_intensity_prologue_coeffs_f32(const float* in, size_t n_per_channel, int n_channels, const float* scale,
                                       const float* shift, double* stats_out, float* abt_out, void* scratch, void* stream);
int mvtb_intensity_affine_f32(const float* in, float* out, size_t n_per_channel, int n_channels, const float* abt,
                              void* stream);

/* ---- Dice loss / metric reductions behind the hot path (MONAI 0.5 DiceLoss(sigmoid=True, squared_pred=True),
 * Activations(sigmoid) -> AsDiscrete(0.5) -> DiceMetric; 10_scripts/127_.../...FLAIR.py:216, 266-283).
 * mvtb_dice_sums_f32: one pass over x (logits if from_logits, else probabilities / binary predictions) and target,
 *   n_vols = B*C volumes of n_per_vol voxels -> sums_out[6 v ..] = sum t p, sum p^2, sum t^2, sum t q, sum q, sum t
 *   (p = sigmoid(x) or x, q = [p >= 0.5]) as device doubles; deterministic.  scratch: mvtb_dice_scratch_bytes(n_vols).
 * mvtb_dice_grad_f32: grad_out_i = (coef[2v] t_i + coef[2v+1] p_i) * (from_logits ? p_i (1 - p_i) : 1). */
size_t mvtb_dice_scratch_bytes(int n_vols);
int mvtb_dice_sums_f32(const float* x, const float* target, size_t n_per_vol, int n_vols, int from_logits,
                       double* sums_out, void* scratch, void* stream);
int mvtb_dice_grad_f32(const float* x, const float* target, size_t n_per_vol, int n_vols, int from_logits,
                       const float* coef, float* grad_out, void* stream);

/* sum_i (a_i - b_i)^2 -> device double (deterministic).  scratch: mvtb_dice_scratch_bytes(1) bytes.  With fftn
 * unnormalised over (H, W), MSE(Re fftn a, Re fftn b) + MSE(Im fftn a, Im fftn b) = H W MSE(a, b) (Parseval): the
 * frequency-consistency loss of 50_reconstruction/reconGan/reconGan_freq.py:134-140 needs no transform. */
int mvtb_sqdiff_sum_f32(const float* a, const float* b, size_t n, double* sum_out, void* scratch, void* stream);

/* RandSpatialCropd / CenterSpatialCropd followed by RandFlipd (MONAI 0.5; 127_...FLAIR.py:130-133, :153) as one gather on a
 * (C, H, W, D) sample:  out[c][i][j][k] = in[c][o0 + (f0 ? s0-1-i : i)][o1 + (f1 ? s1-1-j : j)][o2 + (f2 ? s2-1-k : k)],
 * in_shape = (H, W, D), out_shape = (s0, s1, s2), offset = (o0, o1, o2) with o + s <= N on every axis, flip_axes_mask bit a =
 * spatial axis a reversed (np.flip after the crop).  The host draws offsets and flips in MONAI's order. in != out. */
int mvtb_crop_flip_f32(const float* in, float* out, int n_channels, const int32_t* in_shape, const int32_t* out_shape,
                       const int32_t* offset, int flip_axes_mask, void* stream);
/* the same for n_samples samples of one shape in one launch, each with its own window and flips: offsets_dev[3 n_samples] and
 * flips_dev[n_samples] are int32 arrays ON THE DEVICE (windows are not range-checked). */
int mvtb_crop_flip_batch_f32(const float* in, float* out, int n_samples, int n_channels, const int32_t* in_shape,
                             const int32_t* out_shape, const int32_t* offsets_dev, const int32_t* flips_dev, void* stream);
/* The same gather for a batch whose samples come from a ragged cache (the training loader's device-resident sample cache):
 *   out[b][c] = flip_b(entry[entry_dev[b]][channels[c]][start_b : start_b + out_shape])
 * Entry e holds n_channels_in channels of spatial shape entry_shape_dev[3e .. 3e+2], C-contiguous, starting at element
 * entry_offset_dev[e] of `cache`.  channels: host array of n_channels_out (<= MVTB_GATHER_MAX_CHANNELS) indices into the
 * stored channels, in any order, or NULL for all of them (then n_channels_out == n_channels_in): a SelectChanneld in front
 * of the crop costs nothing, the unselected channels are never read.  out_shape: host, every axis >= 1.  out: (n_samples,
 * n_channels_out, s0, s1, s2), cache != out.  entry_dev[n_samples], starts_dev[3 n_samples] and flips_dev[n_samples] (bit a =
 * spatial axis a; bits above 2 are ignored) are int32 arrays ON THE DEVICE, as are the int64 entry_offset_dev and the int32
 * entry_shape_dev tables: none of them is checked here.  The caller guarantees that every entry index is valid and that
 * 0 <= start_b and start_b + out_shape <= the entry's shape on every axis (mvtb/train_stage.py checks each window on the
 * host before it uploads them). */
#define MVTB_GATHER_MAX_CHANNELS 8
int mvtb_crop_flip_gather_f32(const float* cache, float* out, int n_samples, int n_channels_out, const int64_t* entry_offset_dev,
                              const int32_t* entry_shape_dev, int n_channels_in, const int32_t* channels, const int32_t* out_shape,
                              const int32_t* entry_dev, const int32_t* starts_dev, const int32_t* flips_dev, void* stream);

/* Spacingd -> Orientationd (MONAI 0.5, 127_...FLAIR.py:120-129: pixdim (1.5, 1.5, 2.0), modes bilinear / nearest,
 * border padding, align_corners=False; then axcodes "RAS"), optionally followed by a crop and flip, as one gather from
 * the loaded volume.  in: (n_volumes, H, W, D), out: (n_volumes, s0, s1, s2), contiguous fp32, in != out.
 * Output index j -> index q in Spacingd's output grid:  q[g] = base[g] + step[g] * j[axis[g]]  (axis a permutation,
 * step +-1, every q inside grid_shape).  q -> source taps along each source axis k, then clipped to [0, n_k - 1]:
 *   taps != NULL (separable transform): source axis k reads taps[tap_off[k] + q[tap_grid[k]]] (device array of n_taps
 *     entries built on the host from torch's own coordinates; its indices are not range-checked here);
 *   taps == NULL (general): coordinate k = matrix[4k] q0 + matrix[4k+1] q1 + matrix[4k+2] q2 + matrix[4k+3] in fp64.
 * NEAREST rounds half to even and copies one voxel; BILINEAR is trilinear in fp32 with the taps' weights. */
#define MVTB_RESAMPLE_BILINEAR 0
#define MVTB_RESAMPLE_NEAREST 1
typedef struct mvtb_resample_tap {
    int32_t i0, i1;          /* source indices of the low and high tap (i1 = min(i0 + 1, n - 1); nearest reads i0) */
    float w0, w1;            /* their weights */
} mvtb_resample_tap;
typedef struct mvtb_resample_geom {
    int32_t in_shape[3];     /* source (H, W, D) */
    int32_t grid_shape[3];   /* Spacingd's output grid */
    int32_t out_shape[3];    /* (s0, s1, s2) */
    int32_t axis[3], base[3], step[3];
    int32_t mode;            /* MVTB_RESAMPLE_* */
    int32_t n_taps;
    int32_t tap_grid[3], tap_off[3];
    const mvtb_resample_tap* taps;
    double matrix[12];
} mvtb_resample_geom;
int mvtb_resample_f32(const float* in, float* out, int n_volumes, const mvtb_resample_geom* geom, void* stream);

/* The decode half of LoadImaged -> AsChannelFirstd: a NIfTI-1/2 payload already on the device (raw: the vox_offset-th byte
 * of the file, aligned to its element size) -> out (C, X, Y, Z) C-contiguous float32, out[c][i][j][k] = file element
 * ((c Z + k) Y + j) X + i.  dims = (X, Y, Z, C), a host array; X Y Z <= 2^31.  datatype: a NIfTI code below (others:
 * MVTB_EUNSUPPORTED); swap_bytes: the file's byte order is not the device's.  scaled = 0: float(raw), rounded to nearest
 * even; scaled != 0: raw * slope + inter in float32 (8/16-bit integers, float32) or float64 (32-bit integers, float64),
 * the multiply and the add rounded separately, then rounded to float32.  raw != out. */
#define MVTB_NIFTI_UINT8 2
#define MVTB_NIFTI_INT16 4
#define MVTB_NIFTI_INT32 8
#define MVTB_NIFTI_FLOAT32 16
#define MVTB_NIFTI_FLOAT64 64
#define MVTB_NIFTI_INT8 256
#define MVTB_NIFTI_UINT16 512
#define MVTB_NIFTI_UINT32 768
int mvtb_nifti_decode_f32(const void* raw, float* out, int32_t datatype, int32_t swap_bytes, const int64_t* dims, double slope,
                          double inter, int32_t scaled, void* stream);

/* WrapArtifact (F:503-515) on (C,H,W,D) when H, W and D are all even: the image-domain fold
 * out = prod_axes (c0 + s c1 Roll_{N/2}) x, c0=(1+alpha)/2, c1=(1-alpha)/2, s=(-1)^(N/2)
 * (SURVEY A.3).  Returns MVTB_EUNSUPPORTED for an odd axis (use the chain). in != out. */
int mvtb_wrap_fold_f32(const float* in, float* out, int n_volumes, int H, int W, int D, float alpha, void* stream);

/* WrapArtifact.__call__ (F:503-515) on (H, W, D) volumes with even H and W and any D (BraTS: 240 x 240 x 155, where
 * the odd D has no half shift): H and W are folded in the image domain, D is filtered row by row (forward FFT,
 * parity weight, inverse FFT in one kernel).  16 B/voxel instead of the chain's five passes.  plan: a 3-D plan of
 * that shape.  MVTB_EUNSUPPORTED for odd H or W (use the chain with wrap weights).  in != out. */
int mvtb_wrap_odd_last_f32(mvtb_plan* plan, const float* in, float* out, int n_volumes, float alpha, void* stream);

/* ---- measurement hooks (bench.py): per-kernel device time from cudaEvents recorded on the
 * launching stream around every launch a plan makes, and a process-wide launch counter. */
#define MVTB_K_ROWS_FWD 0
#define MVTB_K_AXIS_FWD 1
#define MVTB_K_AXIS_MID 2
#define MVTB_K_AXIS_INV 3
#define MVTB_K_ROWS_INV 4
#define MVTB_K_BL_FWD_H 5
#define MVTB_K_BL_FWD_W 6
#define MVTB_K_BL_MID 7
#define MVTB_K_BL_INV_W 8
#define MVTB_K_BL_INV_H 9
#define MVTB_K_SPIKE_REDUCE 10
#define MVTB_K_SPIKE_APPLY 11
#define MVTB_K_ROWS_WRAP 12
#define MVTB_K_BL_INV_SP 13
#define MVTB_K_BL_FWD_TC 14
#define MVTB_K_BL_INV_TC 15
#define MVTB_K_BL_MM_TC 16     /* k_bl_inv_tc<NF, 0>: compute-only pass, per-sample (min, max) */
#define MVTB_K_SP_BITS 17      /* k_sp_bits: the select pass's coordinates as 2 bits per voxel */
#define MVTB_K_KINDS 18
int mvtb_plan_profile(mvtb_plan* plan, int enable);   /* 1: reset + start recording, 0: stop */
/* synchronises the recorded events; fills ms_sum[kind] / counts[kind] (arrays of MVTB_K_KINDS) */
int mvtb_plan_profile_read(mvtb_plan* plan, double* ms_sum, int* counts);
const char* mvtb_kernel_name(int kind);
unsigned long long mvtb_launch_count(void);           /* kernels launched by this library so far */

/* Which kernels the chain uses: 0 = automatic (the band-limited pruned-DFT path when the mask is a
 * small disk, else the general FFT path), 1 = always the general FFT path.  Both produce the same
 * result to fp32 rounding; the switch exists for tests and measurements. */
#define MVTB_PATH_AUTO 0
#define MVTB_PATH_GENERAL 1
#define MVTB_PATH_BL_PAIRS 2   /* automatic, but the band-limited H kernels use pair folding even when H % 4 == 0 */
#define MVTB_PATH_BL_SPLIT 3   /* automatic, but the band-limited W axis, D axis and pointwise stage run as three kernels */
int mvtb_plan_set_path(mvtb_plan* plan, int path);
#define MVTB_PATH_BL_CUDACORE 4 /* automatic, with both band-limited H-axis passes on the CUDA cores */
#define MVTB_PATH_BL_TC 5       /* automatic, with both band-limited H-axis passes on the tensor cores (tcgen05, 3xTF32); AUTO runs
                                   the forward pass there (faster) and the inverse pass on the CUDA cores (MVTB_TC / MVTB_TC_INV) */

/* Synchronises the device and returns 0, or a positive code if a tensor-core kernel of this plan gave up on one of
 * its (bounded) mbarrier waits -- a protocol bug; results of that call are then invalid.  For tests. */
int mvtb_plan_tc_status(mvtb_plan* plan);

#ifdef __cplusplus
}
#endif
#endif /* MVTB_H */
