// chw.cu -- the detector input of the torchvision Faster R-CNN loader: HWC uint8 BGR -> float32 [3,H,W] RGB planes.
//
// Reference: train_frcnn_augmented.py:61-67 -- Compose([RandomCorruption(0.5), ToImage(), ToDtype(torch.float32,
// scale=True)]).  torchvision's to_dtype_image computes image.to(float32).mul_(1.0 / 255): one product
// fl(float(v) * fl(1/255)) per element.  (That is not v / 255.0f for every v, so the lookup table of format_pairs_kernel,
// restoration.cu, does not apply here.)
//
// chw_f32_kernel: persistent CTAs over bands of kChwWarps rows, one row per warp.  Image i is read from `src` when its
// op-code is ROD_OP_NONE, else from the scratch the corruption kernels wrote (dst descriptors); clean images are never
// copied.  Image i's planes start at out + chw_off[i] + c * H * W (rod_plan_chw_offset: 256-byte aligned blocks), so when
// H * W % 4 != 0 the three planes of one row sit at three different float4 phases.  A warp therefore stages a segment of
// its row in shared memory (coalesced 16-byte loads at whatever byte phase the row has), and each plane then reads its
// own pixel window from there: lane l writes the aligned float4 slot covering pixels [4s - m, 4s - m + 4) of plane row
// phase m, with scalar stores only for the partial slots at both ends of the row.  The shared-memory reads are bytes at
// a stride of 3 (12 bytes per lane): conflict-free.
#include "rod_internal.h"

namespace rod {

constexpr int kChwSeg = 512;   // pixels per staged row segment: 4 float4 slots per lane and plane
constexpr int kChwLead = 3;    // pixels staged before a segment (a plane's slot may begin up to 3 pixels before it)
// byte phase (< 16) + 3 * (kChwSeg + kChwLead) bytes, in whole 16-byte chunks
constexpr int kChwStageChunks = (15 + 3 * (kChwSeg + kChwLead) + 15) / 16;
constexpr int kChwCtasPerSm = 6;  // 1536 threads per SM (40 registers: no spills); 6 x 12.5 KB of shared memory

struct ChwParams {
    const DevImage* images;
    const Tile* tiles;      // {image, first row, end row, 0}
    int n_tiles;
    const uint8_t* src;     // clean images (src descriptors)
    const uint8_t* scratch; // corrupted images (dst descriptors)
    const uint8_t* opcodes;
    const uint64_t* out_off;  // float offset of image i's [3,H,W] block
    float* out;
};

__device__ __forceinline__ float to_unit(uint32_t v) {
    // float(v) for a byte v: 2^23 + v has v in its low mantissa bits, minus 2^23 is exact; then torchvision's product
    const float f = __fsub_rn(__uint_as_float(0x4B000000u | v), 8388608.0f);
    return __fmul_rn(f, 1.0f / 255.0f);
}

__global__ void __launch_bounds__(32 * kChwBandRows, kChwCtasPerSm) chw_f32_kernel(ChwParams p) {
    __shared__ __align__(16) uint8_t stage[kChwBandRows][kChwStageChunks * 16];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    uint8_t* sm = stage[warp];
    for (int t = blockIdx.x; t < p.n_tiles; t += gridDim.x) {
        const Tile tl = p.tiles[t];
        const int y = tl.a + warp;
        if (y >= tl.b) continue;
        const DevImage im = p.images[tl.img];
        const bool clean = p.opcodes[tl.img] == ROD_OP_NONE;
        const uint8_t* row = clean ? p.src + im.src_off + (int64_t)y * im.src_pitch
                                   : p.scratch + im.dst_off + (int64_t)y * im.dst_pitch;
        const int w = im.w;
        const uint64_t plane = (uint64_t)im.h * w;
        float* orow = p.out + p.out_off[tl.img] + (uint64_t)y * w;
        const uintptr_t rbeg = (uintptr_t)row, rend = rbeg + 3u * (uint32_t)w;
        for (int x0 = 0; x0 < w + kChwLead; x0 += kChwSeg) {
            // stage the bytes of pixels [x0 - 3, x0 + kChwSeg): only chunks that hold bytes of the row are read
            const uintptr_t g = rbeg + 3 * (intptr_t)(x0 - kChwLead);
            const uintptr_t a = g & ~(uintptr_t)15;
            const int phase = (int)(g - a);
            for (int q = lane; q < kChwStageChunks; q += 32) {
                const uintptr_t c = a + 16 * (uintptr_t)q;
                if (c + 16 > rbeg && c < rend) *reinterpret_cast<uint4*>(sm + 16 * q) = __ldg(reinterpret_cast<const uint4*>(c));
            }
            __syncwarp();
#pragma unroll
            for (int c = 0; c < 3; ++c) {  // BGR -> RGB: plane c is channel 2 - c
                float* prow = orow + c * plane;
                const int m = (int)((c * plane + (uint64_t)y * w) & 3);  // chw_off[i] is a multiple of 64 floats
                const uint8_t* sb = sm + phase + 3 * (kChwLead - x0) + (2 - c);  // byte of channel 2 - c of pixel x: sb[3x]
#pragma unroll
                for (int j = 0; j < kChwSeg / 128; ++j) {
                    const int x = x0 + 128 * j + 4 * lane - m;  // first pixel of this lane's slot
                    if (x >= w) break;
                    float v[4];
#pragma unroll
                    for (int i = 0; i < 4; ++i) v[i] = to_unit(sb[3 * (x + i)]);
                    if (x >= 0 && x + 4 <= w) {
                        *reinterpret_cast<float4*>(prow + x) = make_float4(v[0], v[1], v[2], v[3]);
                    } else {
#pragma unroll
                        for (int i = 0; i < 4; ++i)
                            if (x + i >= 0 && x + i < w) prow[x + i] = v[i];
                    }
                }
            }
            __syncwarp();
        }
    }
}

int launch_chw_f32(const rod_plan* plan, const uint8_t* src, const uint8_t* scratch, const uint8_t* opcodes, float* out,
                   cudaStream_t stream) {
    ChwParams p;
    p.images = plan->d_images;
    p.tiles = plan->chw_tiles.d;
    p.n_tiles = plan->chw_tiles.n;
    p.src = src; p.scratch = scratch; p.opcodes = opcodes;
    p.out_off = plan->d_chw_off;
    p.out = out;
    chw_f32_kernel<<<grid_for(plan, p.n_tiles, kChwCtasPerSm), 32 * kChwBandRows, 0, stream>>>(p);
    ROD_CUDA(cudaGetLastError());
    return ROD_OK;
}

}  // namespace rod
