// filter2d.cu -- a2+a3 for angles other than 0: general k x k float32 kernel (SURVEY 8f rank 3, sm_100a).
//
// Reference: scripts/augmentations.py:21-38 -> cv2.filter2D(img, -1, kernel) with the line kernel rotated by
// cv2.warpAffine.  For k*k < 130 OpenCV 4.13.0 runs its direct FilterEngine (filter.simd.hpp Filter2D +
// FilterVec_8u): per output byte the non-zero taps are accumulated in float32 in row-major kernel order from 0,
// BORDER_REFLECT_101 on both axes, cvRound + saturate.  The vectorised part of a row (flat byte index below
// 4 * (3W / 4)) uses fused multiply-add, the scalar tail (last 3W % 4 bytes) a separate multiply and add -- both
// reproduced here, so the result is bit-exact (tests/golden/golden_angles.npz).
//
// Unlike the angle-0 box (blur.cu, HBM-bound) this op is FMA-issue-bound: ~23 dependent-order FMAs per byte for
// the 45-degree 9 x 9 kernel.  A CTA stages a tile plus halo as float32 in shared memory once; each thread then
// owns 3 byte columns x 2 rows (6 independent accumulation chains), reading conflict-free (lane = byte column).
#include "rod_internal.h"

namespace rod {

constexpr int kF2dCols = 3;  // byte columns per thread (256 apart)

struct Filter2dParams {
    const DevImage* images;
    const Tile* tiles;  // a = first row, b = first byte column of the tile
    int n_tiles;
    const uint8_t* src;
    uint8_t* dst;
    const uint8_t* opcodes;
    const float4* taps;  // {dy, 3 * dx (int bits), weight, -} non-zero kernel entries in row-major order
    int n_taps, k;
    int tile_pitch;  // floats per staged row
};

__global__ void __launch_bounds__(256) filter2d_kernel(Filter2dParams p) {
    extern __shared__ __align__(16) uint8_t smem[];
    float4* s_taps = reinterpret_cast<float4*>(smem);
    float* tile = reinterpret_cast<float*>(smem + (size_t)p.n_taps * sizeof(float4));
    for (int i = threadIdx.x; i < p.n_taps; i += 256) s_taps[i] = p.taps[i];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int r = p.k >> 1, tp = p.tile_pitch;
    __syncthreads();
    for (int ti = blockIdx.x; ti < p.n_tiles; ti += gridDim.x) {
        const Tile t = p.tiles[ti];
        if (p.opcodes != nullptr && p.opcodes[t.img] != ROD_OP_BLUR) continue;
        const DevImage im = p.images[t.img];
        const uint8_t* simg = p.src + im.src_off;
        uint8_t* dimg = p.dst + im.dst_off;
        const int n = 3 * im.w, y0 = t.a, b0 = t.b;
        const int th = min(kF2dTH, im.h - y0), twb = min(kF2dTWB, n - b0);
        // ---- stage rows [y0 - r, y0 + th + r) x byte columns [b0 - 3r, b0 + twb + 3r) as floats, reflect-101 per pixel
        const int ncols = twb + 6 * r;
        for (int rr = warp; rr < th + 2 * r; rr += 8) {
            const uint8_t* srow = simg + (int64_t)reflect101(y0 + rr - r, im.h) * im.src_pitch;
            float* trow = tile + rr * tp;
            // columns [c_lo, c_hi) lie inside the row: 32-bit loads over their 4-byte aligned middle, bytes at the ends;
            // the columns outside are reflected border pixels (per pixel, not per byte)
            const int c_lo = max(0, 3 * r - b0), c_hi = min(ncols, n + 3 * r - b0);
            const uint8_t* s0 = srow + (b0 - 3 * r);  // s0[ci] is the source byte of column ci
            const int c_al = min(c_hi, c_lo + (int)((4u - (uint32_t)((uintptr_t)(s0 + c_lo) & 3u)) & 3u));
            const int n_words = (c_hi - c_al) >> 2;
            for (int q = lane; q < n_words; q += 32) {
                const uint32_t v = __ldg(reinterpret_cast<const uint32_t*>(s0 + c_al) + q);
                float* t4 = trow + c_al + 4 * q;
                t4[0] = (float)(v & 0xFFu); t4[1] = (float)((v >> 8) & 0xFFu); t4[2] = (float)((v >> 16) & 0xFFu); t4[3] = (float)(v >> 24);
            }
            for (int ci = lane; ci < ncols; ci += 32) {
                if (ci >= c_al && ci < c_al + 4 * n_words) continue;  // done above
                const int i = b0 + ci - 3 * r;  // byte position in the row
                if (i >= 0 && i < n) {
                    trow[ci] = (float)srow[i];
                } else {
                    const int j = i + 3 * r, px = j / 3, c = j - 3 * px;  // j >= 0; pixel px - r
                    trow[ci] = (float)srow[3 * reflect101(px - r, im.w) + c];
                }
            }
        }
        __syncthreads();
        // ---- accumulate
        const int n_vec = n & ~3;  // bytes at or beyond it belong to OpenCV's scalar tail
        for (int ry = 0; ry < th; ry += 2) {
            float acc[2][kF2dCols];
#pragma unroll
            for (int q = 0; q < 2; ++q)
#pragma unroll
                for (int i = 0; i < kF2dCols; ++i) acc[q][i] = 0.f;
            const float* base = tile + ry * tp + threadIdx.x;
            for (int tt = 0; tt < p.n_taps; ++tt) {
                const float4 tap = s_taps[tt];
                const float* q0 = base + __float_as_int(tap.x) * tp + __float_as_int(tap.y);
#pragma unroll
                for (int q = 0; q < 2; ++q)
#pragma unroll
                    for (int i = 0; i < kF2dCols; ++i) acc[q][i] = fmaf(q0[q * tp + 256 * i], tap.z, acc[q][i]);
            }
#pragma unroll
            for (int i = 0; i < kF2dCols; ++i) {
                const int x = (int)threadIdx.x + 256 * i;
                if (x >= twb) continue;
                const bool tail = (b0 + x) >= n_vec;
#pragma unroll
                for (int q = 0; q < 2; ++q) {
                    if (ry + q >= th) continue;
                    float s = acc[q][i];
                    if (tail) {  // scalar tail of the row: separate multiply and add
                        s = 0.f;
                        for (int tt = 0; tt < p.n_taps; ++tt) {
                            const float4 tap = s_taps[tt];
                            s = fadd(s, fmul(tile[(ry + q + __float_as_int(tap.x)) * tp + x + __float_as_int(tap.y)], tap.z));
                        }
                    }
                    float v = frint(s);
                    v = v < 0.f ? 0.f : (v > 255.f ? 255.f : v);
                    dimg[(int64_t)(y0 + ry + q) * im.dst_pitch + b0 + x] = (uint8_t)(int)v;
                }
            }
        }
        __syncthreads();  // the tile is restaged
    }
}

int launch_filter2d(const rod_plan* plan, const uint8_t* src, uint8_t* dst, const uint8_t* opcodes, cudaStream_t stream,
                    int img_lo, int img_hi) {
    const auto [tiles, n_tiles] = plan->f2d_tiles.range(img_lo, img_hi);
    if (n_tiles == 0 || plan->f2d_ntaps == 0) return ROD_OK;
    Filter2dParams p;
    p.images = plan->d_images;
    p.tiles = tiles;
    p.n_tiles = n_tiles;
    p.src = src; p.dst = dst; p.opcodes = opcodes;
    p.taps = plan->d_f2d_taps;
    p.n_taps = plan->f2d_ntaps;
    p.k = plan->f2d_k;
    p.tile_pitch = kF2dTWB + 3 * (p.k - 1);
    const size_t smem = (size_t)p.n_taps * sizeof(float4) + (size_t)(kF2dTH + p.k - 1) * p.tile_pitch * sizeof(float);
    if (smem > 227 * 1024) return ROD_ERR_UNSUPPORTED;
    ROD_CUDA(cudaFuncSetAttribute(filter2d_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    int per_sm = (int)((227 * 1024) / (smem + 1024));
    per_sm = per_sm < 1 ? 1 : (per_sm > 4 ? 4 : per_sm);
    filter2d_kernel<<<grid_for(plan, p.n_tiles, per_sm), 256, smem, stream>>>(p);
    ROD_CUDA(cudaGetLastError());
    return ROD_OK;
}

}  // namespace rod
