// rod_internal.h -- host-side plan object shared by the translation units of librod_b200.so.
#pragma once
#include <cuda_runtime.h>

#include <atomic>
#include <mutex>
#include <utility>
#include <vector>

#include "../../include/rod_b200.h"
#include "rod_core.h"

namespace rod {

constexpr unsigned int kCounterRing = 4096;  // rod_plan::d_counters

// Tile geometry shared by the host tile builders and the kernels.
constexpr int kNoiseSpan = 16384;  // elements (bytes) per noise work item
constexpr int kBlurRowsPerTile = 8;  // one row per warp, 8 warps per CTA
constexpr int kLowresTH = 32;      // output rows per lowres tile
constexpr int kLowresTWB = 480;    // output BYTES per lowres tile row (byte columns); its ~250 low-res byte columns fit one pass of 256 threads
constexpr int kLbTH = 32;          // letterbox output tile
constexpr int kLbTW = 64;
constexpr int kMaxAreaTaps = 8;
constexpr int kF2dTH = 16;         // general 2-D filter tile: rows x output bytes
constexpr int kF2dTWB = 768;
constexpr int kF2dMaxElems = 130;  // cv::filter2D uses DFT-based convolution from 130 kernel elements on (8U)
constexpr int kChwBandRows = 8;    // CHW conversion: rows per work item, one per warp
constexpr size_t kFusedMaxSmem = 227 * 1024;  // fused letterbox: dynamic shared memory one CTA may use

struct HostShape {
    int h, w;
};

// Letterbox geometry + tables of one source shape.
struct DevLetterbox {
    int32_t h, w, new_h, new_w, top, left;
    int32_t area2;             // 1: exact 2x2 decimation (cv::resize rewrites INTER_LINEAR to INTER_AREA)
    int32_t identity;          // 1: new size == source size
    uint32_t lx_s0, lx_a;      // int32 s0[new_w], uint32 (a0 | a1<<16)[new_w]
    uint32_t ly_s, ly_b;       // uint32 (s0 | s1<<16)[new_h], uint32 (b0 | b1<<16)[new_h]
    uint32_t lx_pack;          // uint2 per OUTPUT column X of the padded row: {3 * s0 (0xFFFFFFFF: padding column), a0 | a1<<16}
    int32_t lane_group;        // fused kernel: lanes l and l + lane_group would read the same shared-memory bank (0: no such period)
};

// A tile list on the device, in image order: the tiles of image i are d[start[i], start[i + 1]).
struct TileList {
    Tile* d = nullptr;
    int n = 0;
    std::vector<int> start;
    // first tile and tile count of images [lo, hi)
    std::pair<const Tile*, int> range(int lo, int hi) const {
        if (n == 0) return {d, 0};
        return {d + start[lo], start[hi] - start[lo]};
    }
};

// The LowRes tile lists, one per kernel and copy unit (lowres.cu launch_lowres_lists)
enum LowresList {
    LR_GENERIC,                       // lowres_kernel: shapes that are not exact-2x in x
    LR_X2_STRIP,                      // lowres_x2_kernel over every exact-2x image (base pointers not 4-byte aligned)
    LR_X2_REST,                       // lowres_x2_kernel over the exact-2x images no band kernel takes
    LR_X2W8, LR_X2W4,                 // lowres_x2w_kernel: 8-byte aligned rows and w % 8 == 0 (64-bit loads), the others
    LR_X2P16, LR_X2P8, LR_X2P4,       // lowres_x2p_kernel (exact 2x in both axes) by copy unit: 16, 8, 4 bytes
    LR_X2F16, LR_X2F8, LR_X2F4,       // lowres_x2f_kernel (exact-2x width, float y taps)
    LR_X2H16, LR_X2H8, LR_X2H4,       // lowres_x2h_kernel (... with the regular three-tap y structure)
    LR_X2G,                           // lowres_x2g_kernel: odd widths at factor 0.5
    LR_X2I_CARRY, LR_X2I_EVEN,        // lowres_x2i_kernel: odd widths with a regular y axis, odd h / even h
    LR_NUM_LISTS
};

}  // namespace rod

struct rod_plan {
    int device = 0;
    int n_images = 0;
    int sm_count = 148;
    std::vector<rod_image_desc> descs;
    std::vector<rod::DevImage> h_images;
    std::vector<rod::HostShape> shapes;  // distinct (h, w)
    uint64_t payload_bytes = 0;
    int max_w = 0;
    bool all_contiguous = true;
    uint64_t src_extent = 0, dst_extent = 0;  // bytes spanned by the descriptors in src / dst
    uint64_t src_min_offset = 0;               // smallest src_offset (start of the span a host upload must cover)

    rod::DevImage* d_images = nullptr;
    rod::TileList noise_tiles, blur_tiles;
    rod::TileList lowres[rod::LR_NUM_LISTS];  // indexed by rod::LowresList
    size_t lowres_x2_smem = 0;
    // ring of work counters for dynamically scheduled kernels, one per launch: launches of one plan may be in flight
    // on several streams / from several host threads, so the slot index is taken atomically and the ring is long
    // enough (4096 launches) that a slot is never reused while its launch is still pending
    unsigned int* d_counters = nullptr;
    // the blur launches' own ring of counter pairs (blur.cu): zeroed once here, and every launch leaves its pair at 0
    unsigned int* d_blur_counters = nullptr;
    mutable std::atomic<unsigned int> launch_seq{0};
    bool monotonic = true;  // image extents are disjoint and increasing in both src and dst
    int gauss_generator = ROD_GAUSS_AUTO;  // Philox-mode Gaussian generator (rod_plan_set_gaussian_generator)

    // lowres tables, rebuilt when the factor changes
    double lowres_factor = -1.0;
    rod::DevShape* d_shapes = nullptr;
    uint32_t* d_tab = nullptr;
    bool lowres_all_identity = false;
    bool lowres_all_x2w = false;  // every shape is either an identity or eligible for the exact-2x in-register / in-smem path
    int lowres_half_rows = 0, lowres_half_cols = 0;  // worst-case low-res rows / cols one tile touches
    int lowres_src_rows = 0;                          // worst-case source rows one generic tile reads

    // letterbox tables, rebuilt when (out_h, out_w) changes
    int lb_out_h = 0, lb_out_w = 0;
    rod::DevLetterbox* d_lb = nullptr;
    uint32_t* d_lb_tab = nullptr;
    bool lb_all_linear = false;  // every shape is a plain INTER_LINEAR letterbox (fused kernel eligible)
    rod::TileList lb_tiles;
    uint8_t* d_scratch = nullptr;  // corrupted full-res images for the letterbox and CHW paths
    uint64_t scratch_bytes = 0;

    // float32 CHW output (rod_corrupt_chw_f32): float offset of image i's [3,H,W] block, i = n: the total (rod_plan_create);
    // its device copy and the row bands are uploaded on first use
    std::vector<uint64_t> chw_off;
    uint64_t* d_chw_off = nullptr;
    rod::TileList chw_tiles;

    // general 2-D blur kernel override (rod_set_blur_kernel): non-zero taps in row-major order
    float4* d_f2d_taps = nullptr;
    int f2d_ntaps = 0, f2d_k = 0;
    rod::TileList f2d_tiles;

    // restoration pairs (rod_restoration_pairs_f32): contiguous-patch plan + two uint8 patch buffers
    rod_plan* inner = nullptr;
    uint8_t* d_patch_clean = nullptr;
    uint8_t* d_patch_corrupted = nullptr;

    // host-buffer (e2e) staging
    uint8_t* d_stage_src = nullptr;
    uint8_t* d_stage_dst = nullptr;
    float* d_stage_noise = nullptr;
    uint8_t* d_stage_ops = nullptr;
    cudaStream_t streams[3] = {nullptr, nullptr, nullptr};
    // fork/join of the per-op kernels of a mixed batch (small batches do not fill the GPU one op at a time)
    cudaStream_t aux_streams[2] = {nullptr, nullptr};
    cudaEvent_t ev_fork = nullptr, ev_join[2] = {nullptr, nullptr};
    // device arrays that came from the block cache (plan.cu plan_alloc), with their sizes
    mutable std::mutex cached_mutex;
    mutable std::vector<std::pair<void*, size_t>> cached_blocks;
    // fork/join of the LowRes launches of one call (several tile lists: lowres.cu launch_lowres); created on first use
    mutable std::mutex lr_mutex;
    mutable cudaStream_t lr_streams[2] = {nullptr, nullptr};
    mutable cudaEvent_t lr_ev_fork = nullptr, lr_ev_join[2] = {nullptr, nullptr};
};

namespace rod {
extern thread_local int g_last_cuda_error;
inline int cuda_fail(cudaError_t e) {
    g_last_cuda_error = (int)e;
    return e == cudaErrorMemoryAllocation ? ROD_ERR_OOM : ROD_ERR_CUDA;
}
#define ROD_CUDA(call)                                  \
    do {                                                \
        cudaError_t _e = (call);                        \
        if (_e != cudaSuccess) return rod::cuda_fail(_e); \
    } while (0)

int grid_for(const rod_plan* plan, int n_tiles, int ctas_per_sm);

// cache of large device blocks keyed by (device, rounded size) (jpeg.cu): cudaMalloc / cudaFree synchronise the device
cudaError_t block_cache_alloc(int dev, void** p, size_t n);
void block_cache_free(int dev, void* p, size_t n);

// kernel launchers (one per .cu)
int launch_noise(const rod_plan* plan, int mode, const uint8_t* src, uint8_t* dst, const float* noise,
                 float* field_out, float sigma, uint64_t seed, uint64_t first_image, uint32_t offset,
                 const uint8_t* opcodes, int my_op, cudaStream_t stream, int img_lo, int img_hi,
                 int generator = -1 /* -1: plan->gauss_generator */);
int launch_blur(const rod_plan* plan, const uint8_t* src, uint8_t* dst, int k, const uint8_t* opcodes,
                cudaStream_t stream, int img_lo, int img_hi);
int launch_lowres(const rod_plan* plan, const uint8_t* src, uint8_t* dst, const uint8_t* opcodes,
                  cudaStream_t stream, int img_lo, int img_hi);
int launch_filter2d(const rod_plan* plan, const uint8_t* src, uint8_t* dst, const uint8_t* opcodes, cudaStream_t stream,
                    int img_lo, int img_hi);
int launch_gather_patches(const rod_plan* plan, const rod_plan* inner, const uint8_t* src, uint8_t* clean,
                          const uint8_t* flips, cudaStream_t stream);
int launch_resize_linear(const uint8_t* src, int h, int w, int64_t src_pitch, uint8_t* dst, int nh, int nw, int64_t dst_pitch,
                         cudaStream_t stream);
int launch_format_pairs(const rod_plan* inner, const uint8_t* clean, const uint8_t* corrupted, float* clean_out,
                        float* corrupted_out, cudaStream_t stream);
// dynamic shared memory of the fused letterbox kernel for this plan (row buffers sized by its widest image); the fused
// path is taken only when it is at most kFusedMaxSmem
size_t fused_letterbox_smem(const rod_plan* plan);
int launch_fused_letterbox(const rod_plan* plan, const uint8_t* src, const uint8_t* scratch, const uint8_t* opcodes,
                           const float* noise, void* out_f16, int pad_value, float sigma, int k, uint64_t seed,
                           uint64_t first_image, uint32_t offset, bool lowres_in_kernel, cudaStream_t stream);
int launch_letterbox(const rod_plan* plan, const uint8_t* img, const uint8_t* src, const uint8_t* opcodes, void* out_f16,
                     int pad_value, cudaStream_t stream);
int launch_chw_f32(const rod_plan* plan, const uint8_t* src, const uint8_t* scratch, const uint8_t* opcodes, float* out,
                   cudaStream_t stream);

int gauss_table_for(int device, float sigma, const int32_t** out);  // noise.cu: device copy of the Philox-mode table
int ensure_lowres_tables(rod_plan* plan, double factor);
int ensure_letterbox_tables(rod_plan* plan, int out_h, int out_w);
int ensure_chw_tables(rod_plan* plan);

enum NoiseMode { NOISE_COMPAT = 0, NOISE_PHILOX = 1, NOISE_COPY = 2, NOISE_FIELD = 3 };
}  // namespace rod
