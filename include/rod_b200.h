/* rod_b200.h -- C ABI of the B200-native corruption pipeline (librod_b200.so).
 *
 * Drop-in boundary for the hot path of ysbbin/Robust-Object-Detection:
 * scripts/augmentations.py (apply_noise :30-33, apply_motion_blur :36-38,
 * apply_lowres :41-45, _apply_random_corruption :48-56) and its batch twin
 * scripts/build_corrupted_testsets.py:41-59,108-124.
 *
 * Plain pointers and sizes only; no torch / C++ types.  Every function returns a
 * rod_status (0 = ok) and never throws.  "Device" pointers are CUDA device
 * addresses on the current device; `stream` is a cudaStream_t passed as void*
 * (NULL = the legacy default stream).  All device work is stream-ordered and the
 * library never synchronises unless the function name ends in _host.
 *
 * A rod_plan may be used from one host thread at a time (it caches tables, tile lists and scratch buffers lazily);
 * launches issued from it on different streams may overlap on the device.  Different plans are independent.
 *
 * Images are HWC uint8 with 3 interleaved channels (BGR for the reference's
 * callers; every operation is per channel).  A batch is described by a table of
 * rod_image_desc: byte offsets into one source and one destination buffer, so
 * ragged (mixed-resolution) batches are one flat buffer + a descriptor table.
 */
#ifndef ROD_B200_H
#define ROD_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(__GNUC__)
#define ROD_API __attribute__((visibility("default")))
#else
#define ROD_API
#endif

typedef enum rod_status {
    ROD_OK = 0,
    ROD_ERR_INVALID_ARG = 1,  /* bad shape / pitch / NULL pointer                     */
    ROD_ERR_UNSUPPORTED = 2,  /* parameter outside the exact-parity domain            */
    ROD_ERR_CUDA = 3,         /* a CUDA call failed; see rod_last_cuda_error()        */
    ROD_ERR_NO_DEVICE = 4,    /* no CUDA device: there is NO CPU fallback             */
    ROD_ERR_OOM = 5
} rod_status;

/* Op-codes of the random one-of-three apply (augmentations.py:50-56); 0 = not applied. */
enum { ROD_OP_NONE = 0, ROD_OP_NOISE = 1, ROD_OP_BLUR = 2, ROD_OP_LOWRES = 3 };

typedef struct rod_image_desc {
    uint64_t src_offset; /* byte offset of pixel (0,0) channel 0 from the src base pointer */
    uint64_t dst_offset; /* same for the dst base pointer                                   */
    int32_t  height;     /* rows    (>= 1)                                                  */
    int32_t  width;      /* pixels  (>= 1); a row holds 3*width bytes                       */
    int64_t  src_pitch;  /* bytes between consecutive source rows, >= 3*width              */
    int64_t  dst_pitch;  /* bytes between consecutive destination rows, >= 3*width         */
} rod_image_desc;

typedef struct rod_plan rod_plan; /* opaque: device descriptor table + tile lists + resize tables */

/* Library / device probing ------------------------------------------------------------ */
ROD_API const char* rod_version(void);
ROD_API int         rod_device_count(void);           /* 0 when no GPU is visible */
ROD_API int         rod_last_cuda_error(void);        /* cudaError_t of the last failing CUDA call (thread local) */
ROD_API const char* rod_status_string(int status);

/* Plans ------------------------------------------------------------------------------- */
/* Uploads the descriptor table (host array) to the current device and precomputes the
 * per-op tile lists.  The plan can be reused for any number of launches on any stream. */
ROD_API int  rod_plan_create(const rod_image_desc* images, int n_images, rod_plan** out_plan);
ROD_API void rod_plan_destroy(rod_plan* plan);
ROD_API int  rod_plan_num_images(const rod_plan* plan);
/* Sum over images of 3*H*W: bytes one full-resolution pass reads (and writes). */
ROD_API uint64_t rod_plan_payload_bytes(const rod_plan* plan);
/* Number of kernels one call of the given op launches (for launch accounting; the counter memsets and the copies of
 * the host entry points are not counted).  ROD_OP_LOWRES: 1 until the first LowRes call built the resize tables, then
 * one per non-empty tile list.  That is exact when the source base pointer of the call is 4-byte aligned and, if the
 * plan has images for the staged exact-2x kernels, so is the destination base.  Otherwise one strip-kernel launch
 * replaces all the exact-2x band and strip launches, and the call launches fewer kernels than this count.
 * The combined entry points have codes of their own: 100 = rod_corrupt_batch_u8 (copy, noise, blur, then the LowRes
 * lists), 101 = rod_corrupt_letterbox_f16 on its unfused path (noise, blur, LowRes lists, letterbox) and 102 =
 * rod_corrupt_chw_f32 (noise, blur, LowRes lists, conversion); each is 3 + the ROD_OP_LOWRES count, with the same
 * base-pointer caveat.  rod_corrupt_letterbox_f16 on its fused path launches 1 kernel, plus the ROD_OP_LOWRES count
 * when the LowRes images do not run inside that kernel. */
ROD_API int  rod_plan_launches(const rod_plan* plan, int op);

/* a1: apply_noise (augmentations.py:30-33).
 * compat mode (noise != NULL): `noise` is a device float32 array holding, image after
 *   image in plan order, the H*W*3 field the reference would have drawn; result is
 *   uint8(trunc(clamp(float(src) + noise, 0, 255))) -- bit-exact with the reference.
 * philox mode (noise == NULL): the field is generated in registers from Philox4x32-10 blocks
 *   (key = seed, counter = (group, first_image_index + i, offset)).  Two Gaussian generators (csrc/rod_core.h defines
 *   both; the oracle restates both):
 *     table      (3 <= sigma <= 20; default there): integer arithmetic only -- one block serves a group of 16 consecutive
 *                elements; each Philox word gives four 8-bit draws from a 256-entry table of N(0, sigma^2/4) (1/256
 *                units; 2nd/4th/6th moments exact) and the four are mixed by a 4 x 4 Hadamard transform,
 *                k = floor((xa +- xb +- xc +- xd) / 256): uncorrelated, 2^32 equally likely values each, tails to 6.2 sigma;
 *     Box-Muller (sigma <= 2048; default outside [3, 20], rod_plan_set_gaussian_generator(ROD_GAUSS_BOXMULLER), and always
 *                on the training path rod_corrupt_letterbox_f16): groups of 8 elements, 16-bit stratified radius with a
 *                32-bit tail refinement, 16-bit angle.
 *   result is clamp(src + floor(noise), 0, 255).  Reproducible for any batch split / GPU count;
 *   validated statistically (not bit-identical to NumPy's stream).  The first launch with a new sigma uploads
 *   the table synchronously: call rod_noise_prewarm(sigma) first when the launch is to be captured in a CUDA graph.
 * opcodes (device uint8[n_images], may be NULL): when given, only images whose
 *   op-code equals ROD_OP_NOISE are processed; the others are left untouched. */
ROD_API int rod_noise_u8(const rod_plan* plan, const uint8_t* src, uint8_t* dst, const float* noise,
                 float sigma, uint64_t seed, uint64_t first_image_index, uint32_t offset,
                 const uint8_t* opcodes, void* stream);
/* The float32 field philox mode adds (same layout as `noise` above); for tests/resume. */
ROD_API int rod_noise_field_f32(const rod_plan* plan, float* out_field, float sigma, uint64_t seed,
                        uint64_t first_image_index, uint32_t offset, void* stream);
/* Philox-mode Gaussian generator of this plan: ROD_GAUSS_AUTO (0, default: table when 3 <= sigma <= 20, else
 * Box-Muller), ROD_GAUSS_BOXMULLER (1) or ROD_GAUSS_TABLE_PHILOX7 (2: like AUTO with the table generator on
 * Philox4x32-7, the smallest round count that passes BigCrush in Salmon et al. 2011 -- a different, equally valid stream). */
#define ROD_GAUSS_AUTO 0
#define ROD_GAUSS_BOXMULLER 1
#define ROD_GAUSS_TABLE_PHILOX7 2
ROD_API int rod_plan_set_gaussian_generator(rod_plan* plan, int generator);
/* Builds and uploads the table-generator table of `sigma` on `device` now (synchronous), so that later Philox-mode
 * launches with this sigma issue no allocation or blocking copy and can be captured in a CUDA graph.  No-op for sigma
 * outside the table generator's range.  (augmentations.py:30-33 has no such state: NumPy draws on the host.) */
ROD_API int rod_noise_prewarm(int device, float sigma);
/* The 256 entries of that table (int32, host pointer): for tests and for restating the stream. */
ROD_API int rod_gauss_table_i32(float sigma, int32_t* out256);

/* The HOST generator of compat mode: the field `np.random.normal(0, sigma, shape).astype(np.float32)` of
 * augmentations.py:31, regenerated bit for bit from NumPy's legacy generator state (MT19937 + polar Gaussian) with the
 * per-pair work spread over `threads` host threads (0 = all).  key[624], *pos, *has_gauss, *cached are
 * np.random.get_state()[1:5] on entry and the state NumPy itself would have after the call on return (feed them to
 * np.random.set_state), so later draws continue on the same stream.  Pure host code (no GPU work).  It is the reference
 * the device generator below is tested against, and the field source of the host-buffer paths (rod_apply_host). */
ROD_API int rod_numpy_legacy_normal_f32(uint32_t* key, int32_t* pos, int32_t* has_gauss, double* cached, double sigma,
                                uint64_t n, float* out, int threads);
/* The same stream drawn on the GPU (csrc/legacy_rng.cu): the values go into n_seg device segments in order, segment s
 * getting seg_counts[s] consecutive floats at out + seg_offsets[s] (segments sorted and disjoint, else
 * ROD_ERR_INVALID_ARG; floats between them are not written), so the fields of several images are one draw.  The state
 * arguments are those of rod_numpy_legacy_normal_f32; sigma must be finite and >= 0.  Returns once the state after the
 * call is known: one host wait on `stream` per round (one round unless the call exceeds 256 x 128 blocks of 624 words,
 * about 2.6 fields of 1360x765x3).  The few values whose float32 could depend on the last ulps of the device log() are
 * recomputed on the host with libm log() and written by a kernel queued on `stream`; *host_fixups (may be NULL) gets
 * their number.  A total count of 0 changes no state. */
ROD_API int rod_numpy_legacy_normal_f32_device(uint32_t* key, int32_t* pos, int32_t* has_gauss, double* cached,
                                double sigma, const uint64_t* seg_offsets, const uint64_t* seg_counts, int n_seg,
                                float* out, int* host_fixups, void* stream);

/* a2+a3: apply_motion_blur(img, k, angle_deg) (augmentations.py:21-38) for angle_deg == 0:
 * horizontal k-tap box, BORDER_REFLECT_101, out = (2S + k) / (2k).  k odd, 1 <= k <= 31;
 * anything else returns ROD_ERR_UNSUPPORTED (never an approximation). */
ROD_API int rod_blur_h_u8(const rod_plan* plan, const uint8_t* src, uint8_t* dst, int k, double angle_deg,
                  const uint8_t* opcodes, void* stream);

/* a2+a3 at angle_deg != 0 (SURVEY 8f): install the k x k float32 kernel that
 * _motion_blur_kernel(k, angle_deg) builds (augmentations.py:21-27; `kernel` is a HOST pointer, row-major).  While
 * installed, every ROD_OP_BLUR of this plan (rod_blur_h_u8 with the same k, rod_corrupt_batch_u8, rod_apply_host,
 * rod_corrupt_letterbox_f16) is cv2.filter2D(img, -1, kernel), bit-exact for k*k < 130 (OpenCV's direct filter
 * engine; larger kernels use DFT-based convolution there and return ROD_ERR_UNSUPPORTED here).  NULL removes it. */
ROD_API int rod_set_blur_kernel(rod_plan* plan, const float* kernel, int k);

/* a4+a5: apply_lowres(img, factor) (augmentations.py:41-45): INTER_AREA down to
 * (max(1,int(W*factor)), max(1,int(H*factor))) then 8-bit INTER_LINEAR back, fused: the
 * low-resolution intermediate lives in shared memory only.  0 < factor <= 1. */
ROD_API int rod_lowres_u8(rod_plan* plan, const uint8_t* src, uint8_t* dst, double factor,
                  const uint8_t* opcodes, void* stream);

/* a6-a9: one launch group that applies opcodes[i] to image i (ROD_OP_NONE = byte copy),
 * with the reference's constants unless overridden: sigma, k, factor.  Noise is philox
 * mode unless `noise` is given. */
ROD_API int rod_corrupt_batch_u8(rod_plan* plan, const uint8_t* src, uint8_t* dst, const uint8_t* opcodes,
                         const float* noise, float sigma, int k, double factor, uint64_t seed,
                         uint64_t first_image_index, uint32_t offset, void* stream);

/* Training path (BASELINE config 5): corruption fused with the detector-input formatting
 * of Ultralytics' LetterBox + Format + preprocess_batch: INTER_LINEAR resize-to-fit of the
 * CORRUPTED pixels, constant pad, BGR->RGB, HWC->CHW, half(float(u8)/255).  `out` is a
 * device fp16 array [n_images, 3, out_h, out_w].  Any 2-byte aligned `out` is accepted; the fused kernel stores pairs
 * of halves, so it runs only when `out` is 4-byte aligned (and out_w is even), otherwise the unfused path computes the
 * same bytes. */
ROD_API int rod_corrupt_letterbox_f16(rod_plan* plan, const uint8_t* src, const uint8_t* opcodes,
                              void* out_f16, int out_h, int out_w, int pad_value,
                              const float* noise, float sigma, int k, double factor, uint64_t seed,
                              uint64_t first_image_index, uint32_t offset, void* stream);

/* Faster R-CNN loader (augmentations.py:60-74 RandomCorruption inside train_frcnn_augmented.py:61-67's
 * Compose([RandomCorruption(0.5), ToImage(), ToDtype(float32, scale=True)])) for a batch: opcodes[i] picks the corruption
 * of image i exactly as rod_corrupt_batch_u8 does (same parameters and checks; Philox noise uses the plan's own generator),
 * then BGR -> RGB, HWC -> CHW and fl(float(v) * fl(1/255)) per element, torchvision's to_dtype_image arithmetic.
 * Output layout: `out` is one flat device float32 buffer (256-byte aligned, else ROD_ERR_INVALID_ARG); image i is the
 * contiguous [3, H_i, W_i] block at float offset rod_plan_chw_offset(plan, i), in plan order, each block starting at a
 * multiple of 64 floats (256 bytes); rod_plan_chw_offset(plan, n_images) is the buffer's size in floats.  The gaps
 * between blocks are not written.  Clean images are read from `src` in place; corrupted ones go through the plan's
 * scratch buffer (the dst descriptors' layout). */
ROD_API int rod_corrupt_chw_f32(rod_plan* plan, const uint8_t* src, const uint8_t* opcodes, float* out, const float* noise,
                        float sigma, int k, double factor, uint64_t seed, uint64_t first_image_index, uint32_t offset,
                        void* stream);
/* Float offset of image i's block in the output of rod_corrupt_chw_f32 (0 <= i <= n_images; 0 otherwise). */
ROD_API uint64_t rod_plan_chw_offset(const rod_plan* plan, int i);

/* SURVEY 8f rank 4 -- RestorationDataset.__getitem__ (scripts/train_restoration.py:104-129) for a batch of patches.
 * The plan's source descriptors are the crops (offset + pitch into the device-resident images; one patch size per
 * batch); flips[i] != 0 applies cv2.flip(patch, 1) first; opcodes[i] picks the corruption (1..3; 0 = none).
 * Outputs are device float32 [n,3,P,P] RGB planes of value / 255.0f: the corrupted input and the clean target. */
ROD_API int rod_restoration_pairs_f32(rod_plan* plan, const uint8_t* src, const uint8_t* flips, const uint8_t* opcodes,
                              float* corrupted_out, float* clean_out, const float* noise, float sigma, int k,
                              double factor, uint64_t seed, uint64_t first_image_index, uint32_t offset, void* stream);

/* The resize-first branch of RestorationDataset._random_crop / _center_crop (scripts/train_restoration.py:79-81,
 * 88-90): frames smaller than the patch are enlarged with cv2.resize(img, (max(w, size), max(h, size))), i.e. OpenCV's
 * 8-bit fixed-point INTER_LINEAR, before the crop.  One HWC uint8 image, device pointers, pitches in bytes; (nh, nw) must
 * not be smaller than (h, w) in either axis (a 2x reduction would switch OpenCV to INTER_AREA: ROD_ERR_UNSUPPORTED). */
ROD_API int rod_resize_linear_u8(const uint8_t* src, int h, int w, int64_t src_pitch, uint8_t* dst, int nh, int nw,
                         int64_t dst_pitch, void* stream);

/* SURVEY 8f rank 1 -- `cv2.imwrite(str(dst_img_dir / img_path.name), out)` (scripts/build_corrupted_testsets.py:124, :164)
 * for a device-resident batch: baseline JPEG encoding whose bytes equal OpenCV 4.13.0's (libjpeg-turbo defaults: YCbCr
 * 4:2:0, quality 95, standard Huffman tables, islow DCT).  `images`: the pixels to encode (src_offset / src_pitch /
 * height / width; HWC BGR uint8).  `header`: the bytes SOI .. SOS OpenCV itself writes with the wanted parameters (any
 * image size): its DQT / DHT segments define the tables; ROD_ERR_UNSUPPORTED unless it is baseline 4:2:0 without restart
 * markers.  After rod_jpeg_encode() the device array rod_jpeg_stream_base() + rod_jpeg_stream_offset(i) holds the
 * entropy-coded segment + EOI of image i and rod_jpeg_stream_lengths()[i] (device uint32) its length, 0xFFFFFFFF if it did
 * not fit its buffer; the file is OpenCV's header for that image size followed by those bytes. */
typedef struct rod_jpeg_encoder rod_jpeg_encoder;
ROD_API int rod_jpeg_create(const rod_image_desc* images, int n_images, const uint8_t* header, uint64_t header_len,
                    rod_jpeg_encoder** out_enc);
ROD_API void rod_jpeg_destroy(rod_jpeg_encoder* enc);   /* its large device buffers go to a cache for the next encoder */
ROD_API void rod_jpeg_trim(void);                         /* frees that cache */
ROD_API int rod_jpeg_encode(rod_jpeg_encoder* enc, const uint8_t* pixels, void* stream);
ROD_API uint64_t rod_jpeg_stream_offset(const rod_jpeg_encoder* enc, int i);
ROD_API const uint8_t* rod_jpeg_stream_base(const rod_jpeg_encoder* enc);
ROD_API const uint32_t* rod_jpeg_stream_lengths(const rod_jpeg_encoder* enc);
/* lengths and streams to the host: host_len[n_images]; image i's bytes at host_out + rod_jpeg_stream_offset(enc, i)
 * (host_out holds rod_jpeg_stream_offset(enc, n_images) bytes); returns when the copies are complete */
ROD_API int rod_jpeg_download(rod_jpeg_encoder* enc, uint8_t* host_out, uint32_t* host_len, void* stream);

/* SURVEY 8f rank 1, the reading side -- `img = cv2.imread(str(img_path))` (scripts/build_corrupted_testsets.py:109, :149)
 * for a batch of files: baseline JPEG decoding whose pixels equal OpenCV 4.13.0's (libjpeg-turbo defaults: islow IDCT, fancy
 * chroma upsampling, BGR output) straight into a device-resident HWC batch.  Decodable here: baseline sequential, 8 bit,
 * one scan (restart markers are fine), no EXIF rotation, either Y Cb Cr with the luma sampled 2x2 (4:2:0, what OpenCV's own
 * encoder writes), 2x1 (4:2:2) or 1x1 (4:4:4) against 1x1 chroma, or greyscale; subsampled files need width >= 5.  Every
 * other file is REPORTED (status >= 10), never approximated: the caller reads it with the host codec.
 * The _ex forms also take PROGRESSIVE files (SOF2, same frame layouts, Huffman coded, table slots 0..3, restart markers
 * fine) when `formats` has ROD_JPEGDEC_PROGRESSIVE: every scan is checked as libjpeg-turbo's jdphuff.c does, and a file
 * whose scans leave a coefficient bit unknown (libjpeg would block-smooth it) or redefine a quantisation table in use is
 * reported as 12; one without EOI behind its last scan as 13.  A complete progressive file decodes to the pixels of its
 * baseline twin.  The plain forms are the _ex forms with ROD_JPEGDEC_BASELINE.
 *   rod_jpegdec_probe        host only: ROD_OK + (height, width) when the device decoder takes the file, else
 *                            ROD_ERR_UNSUPPORTED
 *   rod_jpegdec_probe_ex     the same for the formats in `formats` (a progressive file is walked to its EOI)
 *   rod_jpegdec_create       host work for a batch (markers, tables, scans without byte stuffing into page-locked memory,
 *                            on `host_threads` threads); image i will be written at pixels + dst_offsets[i] with row pitch
 *                            dst_pitches[i] bytes (NULL or 0: 3 * width)
 *   rod_jpegdec_create_ex    the same for the formats in `formats`; baseline and progressive files mix in one batch
 *   rod_jpegdec_host_status  the verdict of create per image (0: decodable; 11: not a JPEG; 12: unsupported layout;
 *                            13: scan does not end in EOI) and the sizes of the decodable ones
 *   rod_jpegdec_decode       upload + Huffman decoding + IDCT + upsampling / colour conversion on `stream`; returns when the
 *                            Huffman stage has synchronised (a few host round trips), the rest is asynchronous
 *   rod_jpegdec_status       waits for `stream`; per image 0: decoded; 1 / 2: corrupt / truncated entropy data (pixels
 *                            undefined); >= 10: as above */
typedef struct rod_jpeg_decoder rod_jpeg_decoder;
#define ROD_JPEGDEC_BASELINE 1
#define ROD_JPEGDEC_PROGRESSIVE 2
ROD_API int rod_jpegdec_probe(const uint8_t* file, uint64_t n, int* height, int* width);
ROD_API int rod_jpegdec_probe_ex(const uint8_t* file, uint64_t n, int formats, int* height, int* width);
ROD_API int rod_jpegdec_create(const uint8_t* const* files, const uint64_t* lens, int n_images, const uint64_t* dst_offsets,
                       const int64_t* dst_pitches, int host_threads, rod_jpeg_decoder** out_dec);
ROD_API int rod_jpegdec_create_ex(const uint8_t* const* files, const uint64_t* lens, int n_images, const uint64_t* dst_offsets,
                          const int64_t* dst_pitches, int host_threads, int formats, rod_jpeg_decoder** out_dec);
ROD_API void rod_jpegdec_destroy(rod_jpeg_decoder* dec);   /* its device / page-locked buffers go to caches for the next decoder */
ROD_API void rod_jpegdec_trim(void);                          /* frees the page-locked cache (the device cache: rod_jpeg_trim) */
ROD_API int rod_jpegdec_host_status(const rod_jpeg_decoder* dec, int32_t* status, int32_t* heights, int32_t* widths);
ROD_API int rod_jpegdec_decode(rod_jpeg_decoder* dec, uint8_t* pixels, void* stream);
ROD_API int rod_jpegdec_status(rod_jpeg_decoder* dec, int32_t* status, void* stream);

/* Host-buffer entry points (what a per-image Python/cgo/JNI caller binds): src/dst are HOST
 * pointers laid out by the plan's descriptors; the call stages through pinned memory,
 * overlaps H2D / kernel / D2H in chunks of images, and returns after dst is complete. */
ROD_API int rod_apply_host(rod_plan* plan, int op, const uint8_t* src_host, uint8_t* dst_host,
                   const float* noise_host, float sigma, int k, double factor, uint64_t seed,
                   uint64_t first_image_index, uint32_t offset);

#ifdef __cplusplus
}
#endif
#endif /* ROD_B200_H */
