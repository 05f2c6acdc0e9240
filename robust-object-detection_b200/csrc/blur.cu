// blur.cu -- a2+a3: horizontal k-tap motion blur (angle 0) on interleaved 3-channel rows (sm_100a).
//
// Reference: scripts/augmentations.py:21-38 -> cv2.filter2D(img, -1, kernel) with the angle-0
// kernel = k taps of float32(1/k) on one row, BORDER_REFLECT_101, i.e. per channel
//     out[x] = round(sum_{j=-r..r} in[reflect101(x + j)] / k)  ==  (2 S + k) / (2 k)   (odd k).
//
// Rows are independent, so one warp owns one row at a time: the row is staged in shared
// memory with 16-byte cp.async copies at the SAME 16-byte phase as its destination address,
// the reflected halo is written next to it, and every lane then produces 16 output bytes per
// step from three 128-bit shared-memory loads and stores them with one 128-bit global store.
// No block-level barrier is used (warps never share data), only __syncwarp().

#include "rod_internal.h"

namespace rod {

struct BlurParams {
    const DevImage* images;
    const Tile* tiles;
    int n_tiles;
    const uint8_t* src;
    uint8_t* dst;
    const uint8_t* opcodes;
    int k;
    int row_buf_bytes;  // shared bytes per warp
    unsigned int* counter;  // zeroed before the launch
};

constexpr int kBlurLeft = 64;  // bytes in front of the 16-byte block that holds pixel 0 (>= 3*15 halo + 16)

__device__ __forceinline__ void cp_async16(uint32_t smem_addr, const void* gptr) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(smem_addr), "l"(gptr) : "memory");
}
__device__ __forceinline__ void cp_async_wait_all() {
    asm volatile("cp.async.commit_group;\ncp.async.wait_group 0;" ::: "memory");
}
__device__ __forceinline__ void stg16_blur(void* p, uint4 v) {
    asm volatile("st.global.L1::no_allocate.v4.u32 [%0], {%1,%2,%3,%4};" ::"l"(p), "r"(v.x), "r"(v.y), "r"(v.z),
                 "r"(v.w)
                 : "memory");
}

template <int K>  // K == 9: specialised fast path; K == 0: generic odd k
__global__ void __launch_bounds__(256, 4) blur_rows_kernel(BlurParams p) {
    extern __shared__ __align__(16) uint8_t smem[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    uint8_t* buf = smem + (size_t)warp * p.row_buf_bytes;
    const uint32_t buf_s = (uint32_t)__cvta_generic_to_shared(buf);
    const int k = (K == 0) ? p.k : K;
    const int halo = 3 * (k >> 1);

    // each warp takes a whole tile (8 consecutive rows) at a time from a shared counter and filters its rows one by one
    for (int sub = 8, ti = 0;;) {
        if (sub >= 8) {
            if (lane == 0) ti = (int)atomicAdd(p.counter, 1u);
            ti = __shfl_sync(0xFFFFFFFFu, ti, 0);
            sub = 0;
        }
        if (ti >= p.n_tiles) break;
        const Tile t = p.tiles[ti];
        const int wr = sub++;
        if (p.opcodes != nullptr && p.opcodes[t.img] != ROD_OP_BLUR) { sub = 8; continue; }
        if (wr >= t.b) { sub = 8; continue; }
        const DevImage im = p.images[t.img];
        const int y = t.a + wr;
        const int n = 3 * im.w;
        const uint8_t* srow = p.src + im.src_off + (int64_t)y * im.src_pitch;
        uint8_t* drow = p.dst + im.dst_off + (int64_t)y * im.dst_pitch;
        const int shift = (int)((uintptr_t)drow & 15);
        uint8_t* row = buf + kBlurLeft + shift;  // byte of pixel 0
        // chunk j covers row positions [16j - shift, 16j - shift + 16); chunks [jf0, jf1) lie fully inside [0, n)
        const int jf0 = (shift != 0) ? 1 : 0;
        const int jf1 = (n + shift) >> 4;
        const bool right_edge = ((n + shift) & 15) != 0;

        // ---- stage the row: smem byte (kBlurLeft + shift + i) = in[i]
        if ((((uintptr_t)srow ^ (uintptr_t)drow) & 15) == 0) {
            const uint8_t* sal = srow - shift;  // 16-byte aligned
            for (int j = jf0 + lane; j < jf1; j += 32) cp_async16(buf_s + kBlurLeft + 16 * j, sal + 16 * j);
            // the (at most two) partial chunks: one byte per lane
            const int i = (lane < 16) ? (lane - shift) : (16 * jf1 - shift + lane - 16);
            if (((lane < 16) ? (shift != 0) : right_edge) && i >= 0 && i < n) row[i] = srow[i];
            cp_async_wait_all();
        } else {
            for (int i = lane; i < n; i += 32) row[i] = srow[i];
        }
        __syncwarp();
        // ---- reflected halo (BORDER_REFLECT_101 per pixel, not per byte)
        if (lane < 2 * halo || K == 0) {
            for (int q = lane; q < 2 * halo; q += 32) {
                const int i = (q < halo) ? (q - halo) : (n + q - halo);  // row position outside [0, n)
                const int px = (i >= 0) ? i / 3 : -((-i + 2) / 3);       // floor(i / 3)
                const int c = i - 3 * px;
                int rp;
                if (im.w > (k >> 1)) rp = (px < 0) ? -px : 2 * (im.w - 1) - px;  // single reflection
                else rp = reflect101(px, im.w);                                   // tiny rows: periodic
                row[i] = row[3 * rp + c];
            }
        }
        __syncwarp();
        // ---- compute + store
        uint8_t* dal = drow - shift;
        if (K == 9) {
            for (int j = jf0 + lane; j < jf1; j += 32) {
                const uint4* wp = reinterpret_cast<const uint4*>(buf + kBlurLeft + 16 * j - 16);
                const uint4 a = wp[0], b = wp[1], c = wp[2];
                const uint32_t w[12] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w, c.x, c.y, c.z, c.w};
                uint32_t out[4];
                blur9_chunk16(w, out);
                stg16_blur(dal + 16 * j, make_uint4(out[0], out[1], out[2], out[3]));
            }
            // partial chunks: lane 0 takes the left one, lane 1 the right one
            if (lane < 2 && ((lane == 0) ? (shift != 0) : right_edge)) {
                const int j = (lane == 0) ? 0 : jf1;
                const uint4* wp = reinterpret_cast<const uint4*>(buf + kBlurLeft + 16 * j - 16);
                const uint4 a = wp[0], b = wp[1], c = wp[2];
                const uint32_t w[12] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w, c.x, c.y, c.z, c.w};
                uint32_t out[4];
                blur9_chunk16(w, out);
                const int lo = 16 * j - shift;
                for (int bb = 0; bb < 16; ++bb) {
                    const int i = lo + bb;
                    if (i >= 0 && i < n) drow[i] = (uint8_t)(out[bb >> 2] >> (8 * (bb & 3)));
                }
            }
        } else {
            const int nchunks = (shift + n + 15) >> 4;
            for (int j = lane; j < nchunks; j += 32) {
                const int lo = 16 * j - shift;
                uint32_t out[4];
#pragma unroll
                for (int g = 0; g < 4; ++g) {
                    uint32_t o = 0;
#pragma unroll
                    for (int b = 0; b < 4; ++b) {
                        const int i = lo + 4 * g + b;
                        const uint32_t v = (i >= 0 && i < n) ? blur_byte_generic(row, i, k) : 0u;
                        o |= v << (8 * b);
                    }
                    out[g] = o;
                }
                if (lo >= 0 && lo + 16 <= n) {
                    stg16_blur(dal + 16 * j, make_uint4(out[0], out[1], out[2], out[3]));
                } else {
                    for (int b = 0; b < 16; ++b) {
                        const int i = lo + b;
                        if (i >= 0 && i < n) drow[i] = (uint8_t)(out[b >> 2] >> (8 * (b & 3)));
                    }
                }
            }
        }
        __syncwarp();  // the row buffer is reused by this warp's next row
    }
}

int launch_blur(const rod_plan* plan, const uint8_t* src, uint8_t* dst, int k, const uint8_t* opcodes,
                cudaStream_t stream, int img_lo, int img_hi) {
    const auto [tiles, n_tiles] = plan->blur_tiles.range(img_lo, img_hi);
    if (n_tiles == 0) return ROD_OK;
    BlurParams p;
    p.images = plan->d_images;
    p.tiles = tiles;
    p.n_tiles = n_tiles;
    p.src = src; p.dst = dst; p.opcodes = opcodes; p.k = k;
    // per-warp buffer: kBlurLeft | (shift + 3w rounded up to 16) | 16 (right window) + halo, 16-byte multiple
    const int row_bytes = 3 * plan->max_w;
    p.row_buf_bytes = kBlurLeft + ((15 + row_bytes + 15) & ~15) + 64;
    // one row buffer per warp: very wide rows run with fewer warps per CTA (the kernel has no block-level coupling)
    int warps = kBlurRowsPerTile;
    while (warps > 1 && (size_t)p.row_buf_bytes * warps > 227 * 1024) --warps;
    const size_t smem = (size_t)p.row_buf_bytes * warps;
    if (smem > 227 * 1024) return ROD_ERR_UNSUPPORTED;  // a single row does not fit: wider than ~77 000 pixels
    int ctas_per_sm = (int)((227 * 1024) / (smem + 1024));
    if (ctas_per_sm < 1) ctas_per_sm = 1;
    // measured on B200 (256 x 1360x765): 4 resident CTAs (32 warps) per SM -> 5.79 TB/s; 5 -> 5.62; 6 -> 5.57; 3 -> 5.66
    if (ctas_per_sm > 4) ctas_per_sm = 4;
    p.counter = plan->d_counters + (plan->launch_seq.fetch_add(1u) & (kCounterRing - 1u));
    ROD_CUDA(cudaMemsetAsync(p.counter, 0, sizeof(unsigned int), stream));
    const int grid = grid_for(plan, (p.n_tiles + warps - 1) / warps, ctas_per_sm);
    if (k == 9) {
        ROD_CUDA(cudaFuncSetAttribute(blur_rows_kernel<9>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        blur_rows_kernel<9><<<grid, 32 * warps, smem, stream>>>(p);
    } else {
        ROD_CUDA(cudaFuncSetAttribute(blur_rows_kernel<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        blur_rows_kernel<0><<<grid, 32 * warps, smem, stream>>>(p);
    }
    ROD_CUDA(cudaGetLastError());
    return ROD_OK;
}

}  // namespace rod
