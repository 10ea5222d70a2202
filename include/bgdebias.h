/*
 * bgdebias.h -- C ABI of libbgdebias_b200.so
 *
 * B200 (sm_100a) replacement for the background-debiasing data path of
 * NinV/Background-Debiased-Video-CIL.  Plain pointers and sizes only: no torch types, no C++
 * types.  Every entry point names the reference code it replaces (paths relative to the
 * reference repository root).
 *
 * Conventions
 *   - every function returns a bgd_status (0 = BGD_OK); on failure bgd_last_error() holds a
 *     message for the calling thread.  The reference signals errors with Python exceptions;
 *     the Python host layer turns a non-zero status into RuntimeError/ValueError.
 *   - "d_" pointers are device memory on the current CUDA device, "h_" pointers are host memory.
 *   - device entry points are stream-ordered: they enqueue work on `stream` (a cudaStream_t,
 *     NULL = default stream) and return without synchronising.  Host entry points copy in,
 *     compute, copy out and return when the result is in the host buffer.
 *   - there is no CPU fallback: without a usable sm_100 device every compute call fails with
 *     BGD_ERR_NO_DEVICE / BGD_ERR_CUDA.
 */
#ifndef BGDEBIAS_H_
#define BGDEBIAS_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define BGD_ABI_VERSION 1

typedef enum bgd_status {
    BGD_OK = 0,
    BGD_ERR_INVALID = 1,      /* bad argument (null pointer, T == 0, negative size, ...) */
    BGD_ERR_CUDA = 2,         /* a CUDA runtime call failed; see bgd_last_error() */
    BGD_ERR_UNSUPPORTED = 3,  /* valid request this build cannot serve */
    BGD_ERR_NO_DEVICE = 4     /* no CUDA device / not an sm_100 device */
} bgd_status;

/* Output layouts of the blend.  NTCHW is what the reference's DataLoader hands the model:
 * per-sample FormatShape('NCHW') gives [T,3,H,W] and default_collate stacks to [B,T,3,H,W]
 * (libs/cil/cil.py:203-210).  NCTHW is the permuted variant BASELINE.json mentions.  NTHWC ([B][T][H][W][3], the
 * *_out entry points only) is channels-last storage of both: its permute(0,1,4,2,3) is the logical [B,T,3,H,W] batch,
 * whose flatten(0, 1) is torch.channels_last-contiguous, and its permute(0,4,1,2,3) is [B,3,T,H,W] in
 * torch.channels_last_3d strides. */
#define BGD_LAYOUT_NTCHW 0
#define BGD_LAYOUT_NCTHW 1
#define BGD_LAYOUT_NTHWC 2

/* Output element types of the *_out blend entry points.  The blend is computed in fp32 as in the *_f32 entry points; a
 * 16-bit output is that value rounded once to nearest even (__float2bfloat16_rn / __float2half_rn), which equals torch's
 * .to(torch.bfloat16) / .to(torch.float16) of the fp32 result bit for bit.  Normalised values lie in about [-2.2, 2.7],
 * far inside the fp16 range. */
#define BGD_OUT_F32  0
#define BGD_OUT_BF16 1
#define BGD_OUT_F16  2

/* Median kernel variants (for differential testing; AUTO is the product path). */
#define BGD_MEDIAN_AUTO      0
#define BGD_MEDIAN_SWAR      1   /* thread-per-4-columns byte-SIMD binary search; any T, any N */
#define BGD_MEDIAN_BITSLICED 2   /* TMA-staged cooperative bit-sliced select; needs N % 16 == 0 */
#define BGD_MEDIAN_COLPLANE  3   /* TMA-staged thread-per-column bit-plane select (AUTO's choice for 512 < T <= 544) */
#define BGD_MEDIAN_LDSM      4   /* TMA-staged, transposing shared-memory loads, POPC counting (AUTO's choice for
                                    T <= 512; longer videos of the same call take COLPLANE) */

/* ---- library / device ------------------------------------------------------------------ */

int bgd_abi_version(void);
const char *bgd_last_error(void);

/* Properties of CUDA device `device`; any out pointer may be NULL. */
int bgd_device_info(int device, int *sm_count, int *cc_major, int *cc_minor,
                    int64_t *smem_optin_bytes, int64_t *total_mem_bytes);

/* Number of kernels this library has launched since load (all threads). */
int64_t bgd_kernel_launch_count(void);

/* Select the median kernel variant used by the entry points below (process-wide). */
int bgd_median_set_variant(int variant);
int bgd_median_get_variant(void);

/* ---- temporal median ---------------------------------------------------------------------
 * Replaces   median_frame = np.median(frames, axis=0).astype(dtype=np.uint8)
 *   cil_tools/extract_background.py:73   (CLI variant of bg_extraction_tmf, :42-75)
 *   libs/loader/comix_loader.py:161      (rawframes variant, :148-164)
 * Semantics (bit-exact): out[n] = (s[(T-1)/2] + s[T/2]) >> 1 with s = sort(frames[:, n]).
 * A video is a [T][N] uint8 matrix, N = H*W*3 bytes per frame, rows contiguous.
 */

/* One video resident in device memory. d_frames [T][N], d_out [N]. */
int bgd_temporal_median_u8(const uint8_t *d_frames, int64_t T, int64_t N, uint8_t *d_out,
                           void *stream);

/* V videos concatenated along T (same N): video v owns rows h_offsets[v] .. h_offsets[v+1]-1.
 * This is one call for what bg_extract_multiple (extract_background.py:102-109) does video by
 * video.  h_offsets is a HOST array of V+1 non-decreasing row indices; every video needs at
 * least one frame.  d_out [V][N]. */
int bgd_temporal_median_varlen_u8(const uint8_t *d_frames, const int64_t *h_offsets, int64_t V,
                                  int64_t N, uint8_t *d_out, void *stream);

/* Host-buffer form of the same computation: the frames are T separately allocated host
 * buffers of N bytes each (the `frames` list of extract_background.py:48-60; pass pointers
 * into one block if they are contiguous).  Stages through pinned memory, runs the kernel,
 * copies the [N] result back to h_out.  `device` = CUDA device ordinal. */
int bgd_temporal_median_u8_host(const uint8_t *const *h_frame_ptrs, int64_t T, int64_t N,
                                uint8_t *h_out, int device);

/* Host-buffer form for a batch of videos in one contiguous host block h_frames [sum T][N]
 * (pinned or pageable); results to h_out [V][N].  Copies and kernels are pipelined in chunks
 * of whole videos through a pinned double buffer.  This is the call a worker of
 * extract_background.py:154-162 would make for its slice of the video list. */
int bgd_temporal_median_varlen_u8_host(const uint8_t *h_frames, const int64_t *h_offsets,
                                       int64_t V, int64_t N, uint8_t *h_out, int device);

/* ---- NaN-masked temporal median / mean (simulated-camera-motion extraction) ---------------
 * Replaces   ave_frame = np.nanmedian(transform_frames, axis=0).astype(np.uint8)   (avg_method 0)
 *            ave_frame = np.nanmean(transform_frames, axis=0).astype(np.uint8)     (avg_method 1)
 *   cil_tools/extract_background.py:94-98 (sim_cam_motion_bg_extract, :78-99); with zero_is_missing != 0
 *   also the `frame[frame == 0] = np.nan` of :91.
 * d_frames [T][N] float32 (N = 100*100*3 after RandomResizedCrop(100)); NaN (and 0) = missing.
 * Median of n valid values: f32((s[(n-1)/2] + s[n/2]) / 2); mean: float32 running sum in frame order,
 * f32(f64(sum) / f64(n)); n == 0: NaN.  d_out_u8 [N] receives the uint8 cast (truncation, NaN -> 0; the
 * value domain is 0 <= v < 256), d_out_f32 [N] the float result; either may be NULL. */
int bgd_nan_temporal_reduce_f32(const float *d_frames, int64_t T, int64_t N, int avg_method,
                                int zero_is_missing, uint8_t *d_out_u8, float *d_out_f32, void *stream);

/* V frame folders in one launch: d_frames [sum T][N], video v = rows h_offsets[v] .. h_offsets[v+1]-1 (HOST
 * array of V+1 row indices, V <= 65535), outputs [V][N].  What bg_extract_multiple
 * (extract_background.py:102-109) does folder by folder with --method sim_cam. */
int bgd_nan_temporal_reduce_varlen_f32(const float *d_frames, const int64_t *h_offsets, int64_t V, int64_t N,
                                       int avg_method, int zero_is_missing, uint8_t *d_out_u8,
                                       float *d_out_f32, void *stream);

/* ---- ActorCutMix blend -----------------------------------------------------------------------
 * Replaces, for all frames of a clip in one launch,
 *   actor_cut_mix = actor_img * actor_mask + scene_img * (1 - actor_mask)   libs/loader/actor_cut_mix_loader.py:143-148
 *   foreground_area += human_mask[:, :, 0].sum()                            :154-163 (_calc_foreground_ratio)
 * d_actor, d_mask, d_scene, d_out: n uint8 elements each ([T][H][W][3], channel innermost), 16-byte aligned;
 * numpy's uint8 (wrapping) arithmetic, exact for any mask value.  d_mask_sum (device uint64, may be NULL)
 * receives the sum of the mask bytes of channel 0 (elements with index % 3 == 0). */
int bgd_actor_cut_mix_u8(const uint8_t *d_actor, const uint8_t *d_mask, const uint8_t *d_scene, int64_t n,
                         uint8_t *d_out, uint64_t *d_mask_sum, void *stream);

/* ---- BG-mix blend ------------------------------------------------------------------------
 * Replaces, for a whole batch in one launch,
 *   libs/loader/comix_loader.py:138-145   BackgroundMixDataset._mix_background
 *       bg    = Normalize(RandomCrop(Resize(bg)))                      (bg_pipeline, :72-75)
 *       blend = imgs * (1 - alpha) + bg.view(1, 3, H, W) * alpha        (:142)
 *   plus the mmaction Normalize + FormatShape('NCHW') that produced `imgs` from uint8 frames
 *   (configs/ucf101/bgmix_plus_randAug/..._bgmix_plus_randAug.py:137-138), folded in as a
 *   per-channel 256-entry table (d_fg_lut) so the foreground travels as uint8.
 *
 *   d_fg      [B][T][H][W][3] uint8 RGB        foreground clips after the geometric pipeline
 *   d_bg_pool [P][3][Hb][Wb]  fp32             backgrounds AFTER Resize (values 0..255, not normalised)
 *   d_bg_idx  [B] int32   pool slot per sample (ignored where apply == 0)
 *   d_top, d_left [B] int32   RandomCrop offsets: rows top..top+H-1, cols left..left+W-1
 *   d_apply   [B] uint8   1 = blend, 0 = foreground normalisation only (sample not mixed)
 *   d_fg_lut  [3][256] fp32   normalised value of every uint8 level per channel
 *   h_bg_mean, h_bg_std [3]  HOST fp32 arrays, torchvision Normalize parameters
 *   alpha     blend weight of the background; (1 - alpha) is computed in double then rounded
 *   d_out     fp32, BGD_LAYOUT_NTCHW: [B][T][3][H][W];  BGD_LAYOUT_NCTHW: [B][3][T][H][W]
 * Arithmetic per element (each operation rounded to fp32, no FMA contraction):
 *   fg = lut[c][x];  bg = (p - mean[c]) / std[c];  out = fg * f32(1-alpha) + bg * f32(alpha)
 */
int bgd_bgmix_blend_f32(const uint8_t *d_fg, int64_t B, int64_t T, int64_t H, int64_t W,
                        const float *d_bg_pool, int64_t P, int64_t Hb, int64_t Wb,
                        const int32_t *d_bg_idx, const int32_t *d_top, const int32_t *d_left,
                        const uint8_t *d_apply, const float *d_fg_lut, const float *h_bg_mean,
                        const float *h_bg_std, double alpha, int layout, float *d_out,
                        void *stream);

/* bgd_bgmix_blend_f32 with a choice of pool and output: replaces the same reference code
 * (libs/loader/comix_loader.py:138-145 with :72-75, and config ..._bgmix_plus_randAug.py:137-138) and hands the model
 * the tensor it consumes.  d_bg_pool is fp32 (pool_is_u8 == 0) or uint8 (pool_is_u8 != 0) [P][3][Hb][Wb]; a uint8 pool
 * (values already at crop scale, images that need no Resize) takes 4x less memory and traffic;
 *   layout     BGD_LAYOUT_NTCHW, BGD_LAYOUT_NCTHW or BGD_LAYOUT_NTHWC ([B][T][H][W][3])
 *   out_dtype  BGD_OUT_F32, BGD_OUT_BF16 or BGD_OUT_F16: element type of d_out
 * Every other argument and the arithmetic as bgd_bgmix_blend_f32. */
int bgd_bgmix_blend_out(const uint8_t *d_fg, int64_t B, int64_t T, int64_t H, int64_t W,
                        const void *d_bg_pool, int pool_is_u8, int64_t P, int64_t Hb, int64_t Wb,
                        const int32_t *d_bg_idx, const int32_t *d_top, const int32_t *d_left,
                        const uint8_t *d_apply, const float *d_fg_lut, const float *h_bg_mean,
                        const float *h_bg_std, double alpha, int layout, int out_dtype, void *d_out,
                        void *stream);

/* Foreground already normalised: d_fg_norm fp32 [B][T][3][H][W] is the `imgs` tensor the reference's
 * pipeline hands to _mix_background (libs/loader/comix_loader.py:142); no table is involved.
 * out = fg * f32(1 - alpha) + bg_norm * f32(alpha) where apply != 0, a copy elsewhere.
 * d_bg_pool is fp32 (pool_is_u8 == 0) or uint8 (pool_is_u8 != 0) [P][3][Hb][Wb]. */
int bgd_bgmix_blend_normfg_f32(const float *d_fg_norm, int64_t B, int64_t T, int64_t H, int64_t W,
                               const void *d_bg_pool, int pool_is_u8, int64_t P, int64_t Hb,
                               int64_t Wb, const int32_t *d_bg_idx, const int32_t *d_top,
                               const int32_t *d_left, const uint8_t *d_apply,
                               const float *h_bg_mean, const float *h_bg_std, double alpha,
                               int layout, float *d_out, void *stream);

/* Host-buffer form: foreground batch and per-sample parameters live in host memory (what a
 * DataLoader collate hands over), the pool and the LUT are device resident.  Copies the inputs
 * in, blends, leaves the training tensor in d_out (device) and returns after the stream is
 * idle.  If h_checksum is not NULL it receives the sum of all output elements (double),
 * computed on device and copied back. */
int bgd_bgmix_blend_f32_host(const uint8_t *h_fg, int64_t B, int64_t T, int64_t H, int64_t W,
                             const float *d_bg_pool, int64_t P, int64_t Hb, int64_t Wb,
                             const int32_t *h_bg_idx, const int32_t *h_top, const int32_t *h_left,
                             const uint8_t *h_apply, const float *d_fg_lut, const float *h_bg_mean,
                             const float *h_bg_std, double alpha, int layout, float *d_out,
                             double *h_checksum, int device);

/* ---- BG-mix over a ragged uint8 pool: Resize + RandomCrop + Normalize + blend ---------------------
 * Replaces the same reference code as bgd_bgmix_blend_f32 (libs/loader/comix_loader.py:138-145 with the
 * bg_pipeline of :72-75) for pools the uniform [P][3][Hb][Wb] form cannot hold:
 *   - backgrounds of different sizes (the reference resizes and crops each image at its own size; the HMDB51 and
 *     Sth-Sth-v2 pools of configs/HMDB51/bgmix_seed_1000_inc_5_stages_bgmix_plus_randAug.py and
 *     configs/sth-sthv2/seed_1000_inc_9_stages_bgmix_plus_randAug.py have mixed widths),
 *   - pools too large to keep resized in fp32 (uint8 at native size is ~4.6x smaller),
 *   - the random-frame mode of _get_bg_image (:133-136, back_ground_from_bg_dir=False): the frames a batch drew,
 *     shipped with the batch, are its pool.
 * d_pool is one byte buffer; image s is planar uint8 [3][h][w] (torchvision.io.read_image's layout) at
 * d_slots[s].offset.  Resize(bg_resize) is evaluated inside the launch with the arithmetic of torchvision's
 * antialiased bilinear resize on float tensors (ATen UpSampleKernel.cpp, third-party): per-axis weight tables from
 * bgd_aa_resize_table, horizontal pass then vertical pass, products and sums rounded as that kernel rounds them
 * (csrc/raggedmix.cu states the order); an axis whose size does not change has no table (-1) and is skipped. */
typedef struct bgd_ragged_slot {
    int64_t offset;      /* bytes from d_pool to the image's first byte */
    int32_t h, w;        /* stored (native) size */
    int32_t Hb, Wb;      /* size after Resize; top/left of the crop refer to this image */
    int32_t xtab, ytab;  /* word offsets of the column / row tables in d_tables; -1 = that axis keeps its size */
    int32_t kx, ky;      /* taps per entry of those tables */
} bgd_ragged_slot;

/* HOST function, no device needed: weight table of one axis for in_size -> out_size.  *taps receives K; when h_words is
 * not NULL it receives out_size entries of (2 + K) 32-bit words: {first source index, tap count, K float weights}. */
int bgd_aa_resize_table(int64_t in_size, int64_t out_size, int32_t *taps, int32_t *h_words, int64_t cap_words);

/* Resize alone (what Resize(bg_resize) of comix_loader.py:72 returns for read_image(...).float()):
 * image at d_pool + h_slot->offset -> d_out fp32 [3][Hb][Wb].  h_slot is a HOST pointer. */
int bgd_aa_resize_u8_f32(const uint8_t *d_pool, const bgd_ragged_slot *h_slot, const int32_t *d_tables,
                         float *d_out, void *stream);

/* The blend; arguments as bgd_bgmix_blend_f32 except the pool: d_slots [P] (device), d_tables (device). */
int bgd_bgmix_blend_ragged_f32(const uint8_t *d_fg, int64_t B, int64_t T, int64_t H, int64_t W,
                               const uint8_t *d_pool, const bgd_ragged_slot *d_slots, int64_t P,
                               const int32_t *d_tables, const int32_t *d_bg_idx, const int32_t *d_top,
                               const int32_t *d_left, const uint8_t *d_apply, const float *d_fg_lut,
                               const float *h_bg_mean, const float *h_bg_std, double alpha, int layout,
                               float *d_out, void *stream);

/* bgd_bgmix_blend_ragged_f32 with a choice of output (replaces libs/loader/comix_loader.py:72-75, :126-136 and :138-145
 * as that entry point does): layout and out_dtype as bgd_bgmix_blend_out, every other argument as
 * bgd_bgmix_blend_ragged_f32. */
int bgd_bgmix_blend_ragged_out(const uint8_t *d_fg, int64_t B, int64_t T, int64_t H, int64_t W,
                               const uint8_t *d_pool, const bgd_ragged_slot *d_slots, int64_t P,
                               const int32_t *d_tables, const int32_t *d_bg_idx, const int32_t *d_top,
                               const int32_t *d_left, const uint8_t *d_apply, const float *d_fg_lut,
                               const float *h_bg_mean, const float *h_bg_std, double alpha, int layout,
                               int out_dtype, void *d_out, void *stream);

/* ---- RandomResizedCrop of a batch of frames (simulated-camera-motion extraction) --------------------
 * Replaces, for every frame of many frame folders in one launch,
 *   cil_tools/extract_background.py:81     cam_motion_pipeline = Compose([RandomResizedCrop(size=100)])
 *   cil_tools/extract_background.py:89-90  frame = cam_motion_pipeline(read_image(f).float()).permute(1, 2, 0)
 * The random draws (top, left, h, w) are made on the host, with the torch RNG, as RandomResizedCrop.get_params makes them;
 * this call evaluates torchvision's resized_crop(frame, top, left, h, w, (out_h, out_w), bilinear, antialias=True) for
 * each frame: the window [:, top:top+h, left:left+w] through ATen's antialiased bilinear resize (third-party,
 * UpSampleKernel.cpp) with the arithmetic of bgd_aa_resize_u8_f32 -- per-axis weight tables from bgd_aa_resize_table
 * (in = crop size, out = output size), horizontal pass then vertical, products and sums rounded as that kernel rounds them
 * (csrc/raggedmix.cu states the order); an axis whose crop size equals the output size has no table (-1) and is skipped.
 *
 *   d_src       frames, planar uint8 [3][H][W] each (torchvision.io.read_image's layout), at any byte offsets
 *   src_bytes   size of d_src; every frame must lie inside it
 *   h_desc      HOST array of n descriptors (validated, then copied to the device on `stream`)
 *   d_tables    int32 weight tables (device), table_words words; may be NULL when no descriptor has a table
 *   d_out       float32 [n][out_h][out_w][3], channels last
 * n < 2^31, and ceil(out_h / 32) * ceil(out_w / 32) <= 65535. */
typedef struct bgd_crop_desc {
    int64_t offset;          /* bytes from d_src to the frame's first byte */
    int32_t H, W;            /* frame size */
    int32_t top, left;       /* crop window: rows top .. top+h-1, columns left .. left+w-1, inside the frame */
    int32_t h, w;
    int32_t xtab, ytab;      /* word offsets in d_tables of the w -> out_w and h -> out_h tables; -1 = no table */
    int32_t kx, ky;          /* taps per entry of those tables (what bgd_aa_resize_table reports for the sizes) */
} bgd_crop_desc;

int bgd_resized_crop_aa_u8_f32(const uint8_t *d_src, int64_t src_bytes, const bgd_crop_desc *h_desc, int64_t n,
                               const int32_t *d_tables, int64_t table_words, int64_t out_h, int64_t out_w,
                               float *d_out, void *stream);

/* ---- foreground pipeline tail: Resize -> Normalize -> FormatShape (-> blend) -----------------
 * Replaces the tail of the reference's training pipeline
 *   dict(type='Resize', scale=(224, 224), keep_ratio=False), Normalize, FormatShape('NCHW')
 *   configs/ucf101/bgmix_plus_randAug/bgmix_seed_1000_inc_10_stages_bgmix_plus_randAug.py:136-138
 * so that the DataLoader can ship the uint8 crops MultiScaleCrop (:129-135) produces.  Resize is mmaction2 0.x ->
 * mmcv.imresize -> cv2.resize(img, (W, H), interpolation=cv2.INTER_LINEAR) (third-party, not in the reference tree);
 * results are bit-equal to cv2.resize for uint8 RGB images.
 *
 *   d_src     packed uint8 source pixels, 4-byte aligned, src_bytes a multiple of 4
 *   h_geom    HOST int64 [B][5]: {byte offset of the clip's first crop pixel in d_src, crop height, crop width,
 *             row stride in bytes, frame stride in bytes}; a clip is T frames, pixels RGB interleaved.  A crop of one
 *             column needs 3 readable bytes after each row (the kernel reads pixel pairs).
 *   d_out     uint8 [B][T][H][W][3]
 */
int bgd_resize_bilinear_u8(const uint8_t *d_src, int64_t src_bytes, const int64_t *h_geom, int64_t B,
                           int64_t T, int64_t H, int64_t W, uint8_t *d_out, void *stream);

/* Resize + the blend of bgd_bgmix_blend_f32 in one launch: the [B][T][H][W][3] uint8 intermediate never exists.
 * Source arguments as bgd_resize_bilinear_u8, blend arguments and arithmetic as bgd_bgmix_blend_f32;
 * d_bg_pool is fp32 (pool_is_u8 == 0) or uint8 (pool_is_u8 != 0) [P][3][Hb][Wb]. */
int bgd_bgmix_resize_blend_f32(const uint8_t *d_src, int64_t src_bytes, const int64_t *h_geom, int64_t B,
                               int64_t T, int64_t H, int64_t W, const void *d_bg_pool, int pool_is_u8,
                               int64_t P, int64_t Hb, int64_t Wb, const int32_t *d_bg_idx,
                               const int32_t *d_top, const int32_t *d_left, const uint8_t *d_apply,
                               const float *d_fg_lut, const float *h_bg_mean, const float *h_bg_std,
                               double alpha, int layout, float *d_out, void *stream);

/* bgd_bgmix_resize_blend_f32 with a choice of output (replaces config ..._bgmix_plus_randAug.py:136-138 and
 * libs/loader/comix_loader.py:138-145 as that entry point does): layout and out_dtype as bgd_bgmix_blend_out, every
 * other argument as bgd_bgmix_resize_blend_f32. */
int bgd_bgmix_resize_blend_out(const uint8_t *d_src, int64_t src_bytes, const int64_t *h_geom, int64_t B,
                               int64_t T, int64_t H, int64_t W, const void *d_bg_pool, int pool_is_u8,
                               int64_t P, int64_t Hb, int64_t Wb, const int32_t *d_bg_idx,
                               const int32_t *d_top, const int32_t *d_left, const uint8_t *d_apply,
                               const float *d_fg_lut, const float *h_bg_mean, const float *h_bg_std,
                               double alpha, int layout, int out_dtype, void *d_out, void *stream);

/* bgd_resize_bilinear_u8 and bgd_bgmix_resize_blend_out with a choice of geometry form: h_geom is HOST int64
 * [B][geom_cols], geom_cols 5 (the form of those entry points, same results) or 11, the training pipeline's
 * Resize(scale=(-1, S)) -> MultiScaleCrop -> Resize((W, H), keep_ratio=False) of mmaction2 0.x:
 *   {the five columns of bgd_resize_bilinear_u8, Hr, Wr, y0, x0, ch, cw}
 * Entry b is cv2.resize(cv2.resize(frame, (Wr, Hr))[y0:y0+ch, x0:x0+cw], (W, H)) of every frame of its clip, both
 * resizes INTER_LINEAR and bit-exact, the first rounded to uint8 as cv2 rounds it; the intermediate images never exist.
 * Needs Hr, Wr, ch, cw >= 1, y0, x0 >= 0, y0 + ch <= Hr, x0 + cw <= Wr and (h - 1) * row stride + 3 * max(w, 2) < 2^31.
 * Every other argument as bgd_resize_bilinear_u8 / bgd_bgmix_resize_blend_out. */
int bgd_resize_bilinear_cols_u8(const uint8_t *d_src, int64_t src_bytes, const int64_t *h_geom, int geom_cols,
                                int64_t B, int64_t T, int64_t H, int64_t W, uint8_t *d_out, void *stream);
int bgd_bgmix_resize_blend_cols_out(const uint8_t *d_src, int64_t src_bytes, const int64_t *h_geom, int geom_cols,
                                    int64_t B, int64_t T, int64_t H, int64_t W, const void *d_bg_pool,
                                    int pool_is_u8, int64_t P, int64_t Hb, int64_t Wb, const int32_t *d_bg_idx,
                                    const int32_t *d_top, const int32_t *d_left, const uint8_t *d_apply,
                                    const float *d_fg_lut, const float *h_bg_mean, const float *h_bg_std,
                                    double alpha, int layout, int out_dtype, void *d_out, void *stream);

/* The evaluation pipeline's tail, with no blend: Resize(scale=(-1, S), keep_ratio=True) -> CenterCrop / ThreeCrop ->
 * Normalize(to_bgr=False) -> FormatShape('NCHW') of mmaction2 0.x (the val / test / feature datasets of a CIL run), so that
 * the DataLoader can ship the decoded uint8 frames.  Each output entry resizes one source clip to Hr x Wr (cv2.resize,
 * INTER_LINEAR, bit-exact) and emits the H x W window at (top, left) of that resized image, normalised through d_fg_lut;
 * the resized image never exists.  The crops of one clip are entries with the same source offset.
 *
 *   d_src      as bgd_resize_bilinear_u8
 *   h_geom     HOST int64 [n][9]: the five columns of bgd_resize_bilinear_u8, then {Hr, Wr, top, left}; needs
 *              Hr, Wr >= 1, top, left >= 0, top + H <= Hr and left + W <= Wr
 *   d_fg_lut   fp32 [3][256] normalisation table, as bgd_bgmix_blend_f32
 *   layout     BGD_LAYOUT_NTCHW ([n][T][3][H][W]) or BGD_LAYOUT_NTHWC ([n][T][H][W][3]); BGD_LAYOUT_NCTHW is rejected
 *   out_dtype  as bgd_bgmix_blend_out
 * With the entries of a batch ordered clip-major, then crop, d_out [n][T][3][H][W] is [B][K*T][3][H][W]: mmaction's
 * crop-major ThreeCrop list after FormatShape('NCHW') and default_collate. */
int bgd_resize_crop_normalize_out(const uint8_t *d_src, int64_t src_bytes, const int64_t *h_geom, int64_t n,
                                  int64_t T, int64_t H, int64_t W, const float *d_fg_lut, int layout,
                                  int out_dtype, void *d_out, void *stream);

/* Host-buffer form of bgd_bgmix_resize_blend_f32, as bgd_bgmix_blend_f32_host is for the blend: the packed crops
 * (h_src, pinned or pageable) and the per-sample draws live in host memory -- what a DataLoader collate hands over when
 * the pipeline stops after MultiScaleCrop (config :129-135) -- the fp32 pool and the table are device resident.  Copies in,
 * runs the fused launch, leaves the training tensor in d_out and returns when the stream is idle; h_checksum (may be NULL)
 * receives the sum of the output elements. */
int bgd_bgmix_resize_blend_f32_host(const uint8_t *h_src, int64_t src_bytes, const int64_t *h_geom, int64_t B,
                                    int64_t T, int64_t H, int64_t W, const float *d_bg_pool, int64_t P,
                                    int64_t Hb, int64_t Wb, const int32_t *h_bg_idx, const int32_t *h_top,
                                    const int32_t *h_left, const uint8_t *h_apply, const float *d_fg_lut,
                                    const float *h_bg_mean, const float *h_bg_std, double alpha, int layout,
                                    float *d_out, double *h_checksum, int device);

/* ---- batched ragged gather (owner side of the sharded background pool's exchange) --------------------
 * Replaces, for the images of a batch that one rank owns, the per-sample background read of the reference
 *   libs/loader/comix_loader.py:126-131   bg_idx = torch.randint(len(self.bg_files)); read_image(self.bg_files[bg_idx])
 * when the pool is sharded across ranks: the owner copies every requested native image into one send buffer in one launch,
 * and a single all_to_all_single delivers it (bgdebias_b200.pool.ShardedPool.fetch).
 *
 *   d_src        the owner's pool bytes (a RaggedPool buffer), 16-byte aligned
 *   h_segments   HOST int64 [n][3]: {source byte offset, destination byte offset, bytes}; both offsets 16-byte aligned, every
 *                segment inside d_src[0, src_bytes) and d_out[0, out_bytes); validated, then copied to the device on `stream`
 *   d_out        destination buffer, 16-byte aligned; bytes outside every segment are left untouched
 * n <= 65535; n == 0 (or only empty segments) launches nothing. */
int bgd_ragged_pack_u8(const uint8_t *d_src, int64_t src_bytes, const int64_t *h_segments, int64_t n, uint8_t *d_out,
                       int64_t out_bytes, void *stream);

/* ---- multi-source ragged gather over peer-mapped shards (bgdebias_b200.pool.PeerPool.gather) ---------------------------
 * The receiving form of the same replacement (libs/loader/comix_loader.py:126-131) on one node: every rank's shard is mapped
 * into every other rank once (bgd_ipc_export / bgd_ipc_open), and a rank copies the images its batch drew straight from their
 * owners' memory into one buffer, in one launch, with no collective and no host synchronisation.
 *
 *   d_bases       DEVICE table of n_bases source base pointers (a rank's own buffer or a peer mapping), each 16-byte aligned
 *   h_base_bytes  HOST int64 [n_bases]: readable bytes from each base
 *   h_segments    HOST int64 [n][4]: {source index, source byte offset, destination byte offset, bytes}; both offsets 16-byte
 *                 aligned, every segment inside its source's [0, h_base_bytes) and inside d_out[0, out_bytes)
 *   d_out         destination buffer, 16-byte aligned; bytes outside every segment are left untouched
 * Every segment is validated on the host before anything is launched (BGD_ERR_INVALID names the first bad one); the table then
 * travels through the per-thread workspace ring, so the call does not wait for the stream.  n <= 65535; n == 0 (or only
 * empty segments) launches nothing. */
int bgd_ragged_gather_u8(const uint8_t *const *d_bases, const int64_t *h_base_bytes, int64_t n_bases, const int64_t *h_segments,
                         int64_t n, uint8_t *d_out, int64_t out_bytes, void *stream);

/* Export the allocation that holds d_ptr (device memory of the current device) to other processes of this host: handle
 * receives the 64-byte cudaIpcMemHandle_t of the allocation's base (found with cuMemGetAddressRange), offset the byte offset
 * of d_ptr from that base.  BGD_ERR_UNSUPPORTED when the memory cannot be exported: it must come from cudaMalloc (torch's
 * native caching allocator without expandable_segments; not the cudaMallocAsync backend, not cuMemCreate mappings). */
int bgd_ipc_export(const void *d_ptr, uint8_t *handle, int64_t *offset);

/* Map a handle of bgd_ipc_export from ANOTHER process into this process on `device` (cudaIpcOpenMemHandle with
 * cudaIpcMemLazyEnablePeerAccess); *d_base receives the mapped allocation base.  A handle cannot be opened in the process
 * that exported it.  BGD_ERR_UNSUPPORTED when the mapping fails (e.g. the two devices cannot access each other). */
int bgd_ipc_open(const uint8_t *handle, int device, void **d_base);

/* Unmap a base returned by bgd_ipc_open.  The exporter must keep its allocation alive until every mapping is closed. */
int bgd_ipc_close(void *d_base);

#ifdef __cplusplus
}
#endif
#endif /* BGDEBIAS_H_ */
