// jpegdec.cu -- f1: device-side baseline JPEG DECODER whose pixels equal cv2.imread's (sm_100a).
//
// Reference: scripts/build_corrupted_testsets.py:109 / :149 (`img = cv2.imread(str(img_path))`): with corruption and encoding
// on the GPU, decoding the source frames on host threads is what the test-set build spends its time in.  The arithmetic
// is rod_jpegdec.h (libjpeg-turbo's integer algorithms, checked on the CPU against cv2.imdecode by tests/emu); this file
// is the batch machinery:
//   host    rod_jpegdec_create: per file (on `host_threads` threads) walk the markers, build the decoding tables, copy the
//           entropy-coded segment without its 0xFF00 stuffing into one page-locked buffer; equal table sets are shared
//   device  Huffman decoding of a scan -- one serial bit stream when there are no restart markers -- in parallel by
//           self-synchronisation (rod_jpegdec.h decode_span): a thread per 1024-bit subsequence, the image's table set in
//           shared memory
//             jpegdec_guess_kernel   end state of every subsequence from a guessed start state
//             jpegdec_sync_kernel    re-decodes the subsequences whose predecessor's end state changed (each thread up to
//                                    eight times per launch); launched until one launch changes nothing
//             jpegdec_scan_kernel    first block of every subsequence (prefix sum of the block counts, a CTA per image)
//             jpegdec_write_kernel   decodes from the now exact start states and stores the coefficients (int16, natural
//                                    order, per-component block rasters; DC as the difference)
//             jpegdec_dc_kernel      DC prediction = prefix sum of the differences per component in MCU order
//           progressive files: the scans in dependency levels (rod_jpegdec_host.h scan_levels), one launch per level
//             jpegdec_prog_kernel    one thread per (image, scan, restart interval) of the level, sequentially through the
//                                    interval (rod_jpegdec.h decode_prog_segment: DC predictions and EOBRUN resolved in
//                                    place, refinements read the coefficients of the earlier levels); the Huffman tables
//                                    of the batch's scans are read through L1; refinement scans only decode (history
//                                    from jpegdec_mask_kernel's per-block masks, results as masks per block)
//             jpegdec_mask_kernel    before a level with AC refinement scans: one thread per coefficient block, its
//                                    nonzero coefficients as a 64-bit mask over zigzag positions
//             jpegdec_apply_kernel   after a level with refinement scans: one thread per block of each, the corrections
//                                    and new coefficients applied
//           jpegdec_idct_kernel      one thread per 8x8 block: dequantisation + islow IDCT in registers -> Y / Cb / Cr planes
//           jpegdec_color_kernel     one thread per four output pixels: fancy chroma upsampling + YCbCr -> BGR, written
//                                    straight into the caller's HWC batch (the layout of a rod_plan)
// Baseline and progressive files share one coefficient buffer and one IDCT / colour pass.  Files of another layout
// (progressive unless the caller asked for it, EXIF rotation, CMYK, 4:1:1 ...) are reported per image; the caller decodes
// those with the host codec.  No CPU decoding in here.
#include <algorithm>
#include <map>
#include <string>
#include <thread>
#include <vector>

#include "rod_internal.h"
#include "rod_jpegdec_host.h"

namespace rod {
using namespace jpegdec;

struct JpegDecParams {
    const ImageRec* images;
    const TableSet* tables;
    const uint8_t* streams;
    int16_t* coef;
    uint8_t* planes;
    uint8_t* pixels;
    int32_t* status;
    const uint32_t* block_start;   // [n + 1] prefix sums of the number of blocks (the kernels use the differences)
    const uint32_t* quad_start;    // [n + 1] prefix sums of h * ceil(w / 4)
    const SegRec* segs;            // restart intervals of all images (an image without restart markers: one)
    const uint32_t* sub_start;     // [n_segs + 1] prefix sums of the number of subsequences
    const uint2* ctas;             // Huffman kernels: CTA -> (segment, first subsequence of the segment it covers)
    int n_segs;
    uint64_t* end_state;           // E[subsequence]
    uint64_t* used_start;          // U[subsequence]: the start state E was computed from
    uint32_t* first_block;         // [subsequence] global block index its first symbol belongs to
    unsigned int* changed;         // one flag per sync launch
    int n_images;
    const ScanRec* scans;          // progressive files: their scans, restart intervals (grouped by level) and tables
    const ScanSeg* psegs;
    const HuffTab* huff;
    uint64_t* nzmask;              // [coefficient block] zigzag_nz_mask before a level with AC refinement scans
    RefineOut* refine;             // refinement scans' results (ScanRec::out_block), applied after their level
};

constexpr int kHuffThreads = 128;

__device__ __forceinline__ void load_tables(TableSet* ts, uint8_t* nat, const TableSet* src_set) {
    const uint32_t* src = reinterpret_cast<const uint32_t*>(src_set);
    uint32_t* dst = reinterpret_cast<uint32_t*>(ts);
    for (int i = threadIdx.x; i < (int)(sizeof(TableSet) / 4); i += kHuffThreads) dst[i] = __ldg(src + i);
    if (threadIdx.x < 64) nat[threadIdx.x] = (uint8_t)rod::jpeg::natural_order(threadIdx.x);
    __syncthreads();
}
__device__ __forceinline__ uint64_t ld_volatile64(const uint64_t* p) {
    uint64_t v;
    asm volatile("ld.volatile.global.u64 %0, [%1];" : "=l"(v) : "l"(p));
    return v;
}
__device__ __forceinline__ void st_volatile64(uint64_t* p, uint64_t v) {
    asm volatile("st.volatile.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}

__global__ void __launch_bounds__(kHuffThreads) jpegdec_guess_kernel(JpegDecParams p) {
    __shared__ TableSet ts;
    __shared__ uint8_t nat[64];
    const uint2 c = p.ctas[blockIdx.x];
    const SegRec sg = p.segs[c.x];
    const ImageRec im = p.images[sg.image];
    load_tables(&ts, nat, p.tables + im.table_set);
    const uint32_t s = c.y + threadIdx.x, n_sub = p.sub_start[c.x + 1] - p.sub_start[c.x];
    if (s >= n_sub) return;
    const uint32_t gs = p.sub_start[c.x] + s, bit0 = 8u * sg.byte0;
    const uint64_t u = span_state(bit0 + s * kSubBits, 0, 0, 0);
    p.used_start[gs] = u;
    p.end_state[gs] = decode_span<false>(layout_of(im), sg.stream_bytes, ts, nat, p.streams + sg.stream_off, u, bit0 + (s + 1) * kSubBits,
                                         nullptr, 0, 0, nullptr);
}

__global__ void __launch_bounds__(kHuffThreads) jpegdec_sync_kernel(JpegDecParams p, int flag_slot) {
    __shared__ TableSet ts;
    __shared__ uint8_t nat[64];
    const uint2 c = p.ctas[blockIdx.x];
    const uint32_t s = c.y + threadIdx.x, n_sub = p.sub_start[c.x + 1] - p.sub_start[c.x];
    const bool mine = s >= 1 && s < n_sub;
    const uint32_t gs = p.sub_start[c.x] + s;
    uint64_t u = 0, st = 0;
    if (mine) {
        u = p.used_start[gs];
        st = state_start(ld_volatile64(p.end_state + gs - 1));
    }
    if (!__syncthreads_or(mine && st != u)) return;   // nothing to do for this CTA: the tables are not even loaded
    const SegRec sg = p.segs[c.x];
    const ImageRec im = p.images[sg.image];
    load_tables(&ts, nat, p.tables + im.table_set);
    if (!mine) return;
    const Layout L = layout_of(im);
    const uint32_t bit0 = 8u * sg.byte0;
    bool changed = false;
    for (int it = 0; it < 8 && st != u; ++it) {
        u = st;
        st_volatile64(p.end_state + gs, decode_span<false>(L, sg.stream_bytes, ts, nat, p.streams + sg.stream_off, u, bit0 + (s + 1) * kSubBits,
                                                           nullptr, 0, 0, nullptr));
        changed = true;
        st = state_start(ld_volatile64(p.end_state + gs - 1));   // the predecessor may have moved on meanwhile
    }
    if (changed) {
        p.used_start[gs] = u;
        p.changed[flag_slot] = 1u;
    }
}

// exclusive prefix sum of the block counts of a segment's subsequences; too few blocks in total: truncated data
__global__ void __launch_bounds__(256) jpegdec_scan_kernel(JpegDecParams p) {
    __shared__ uint32_t warp_sum[8];
    __shared__ uint32_t carry_s;
    const int seg = blockIdx.x;
    const uint32_t s0 = p.sub_start[seg], n_sub = p.sub_start[seg + 1] - s0;
    if (threadIdx.x == 0) carry_s = 0;
    __syncthreads();
    for (uint32_t base = 0; base < n_sub; base += 256) {
        const uint32_t s = base + threadIdx.x;
        const uint32_t v = s < n_sub ? state_nblk(p.end_state[s0 + s]) : 0u;
        uint32_t x = v;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const uint32_t y = __shfl_up_sync(0xFFFFFFFFu, x, d);
            if ((threadIdx.x & 31) >= d) x += y;
        }
        if ((threadIdx.x & 31) == 31) warp_sum[threadIdx.x >> 5] = x;
        __syncthreads();
        uint32_t before = carry_s;
        for (int w = 0; w < (int)(threadIdx.x >> 5); ++w) before += warp_sum[w];
        if (s < n_sub) p.first_block[s0 + s] = before + x - v;
        __syncthreads();
        if (threadIdx.x == 255) carry_s = before + x;
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        const SegRec sg = p.segs[seg];
        if (carry_s < sg.n_blocks) atomicMax(p.status + sg.image, 2);
    }
}

__global__ void __launch_bounds__(kHuffThreads) jpegdec_write_kernel(JpegDecParams p) {
    __shared__ TableSet ts;
    __shared__ uint8_t nat[64];
    const uint2 c = p.ctas[blockIdx.x];
    const SegRec sg = p.segs[c.x];
    const ImageRec im = p.images[sg.image];
    load_tables(&ts, nat, p.tables + im.table_set);
    const uint32_t s = c.y + threadIdx.x, n_sub = p.sub_start[c.x + 1] - p.sub_start[c.x];
    if (s >= n_sub) return;
    const uint32_t gs = p.sub_start[c.x] + s, bit0 = 8u * sg.byte0;
    const uint32_t local = p.first_block[gs];
    if (local >= sg.n_blocks) return;   // behind the segment's last block: padding
    int err = 0;
    decode_span<true>(layout_of(im), sg.stream_bytes, ts, nat, p.streams + sg.stream_off,
                      s == 0 ? span_state(bit0, 0, 0, 0) : state_start(p.end_state[gs - 1]), bit0 + (s + 1) * kSubBits,
                      p.coef + im.coef_off, sg.first_block + local, sg.first_block + sg.n_blocks, &err);
    if (err) atomicMax(p.status + sg.image, 1);
}

// One thread per restart interval of a progressive scan, `lanes` threads per warp (the intervals are serial work with
// divergent control flow: a warp of its own for each while the level has few of them).  Segments [seg0, seg0 + n).
__global__ void __launch_bounds__(128) jpegdec_prog_kernel(JpegDecParams p, uint32_t seg0, uint32_t n, uint32_t lanes) {
    __shared__ uint8_t nat[64];
    if (threadIdx.x < 64) nat[threadIdx.x] = (uint8_t)rod::jpeg::natural_order(threadIdx.x);
    __syncthreads();
    const uint32_t lane = threadIdx.x & 31u;
    if (lane >= lanes) return;
    const uint32_t j = ((blockIdx.x * 128u + threadIdx.x) >> 5) * lanes + lane;
    if (j >= n) return;
    const ScanSeg sg = p.psegs[seg0 + j];
    const ScanRec sc = p.scans[sg.scan];
    if (p.status[sc.image] != 0) return;   // an earlier level found the image's data corrupt
    const ImageRec im = p.images[sc.image];
    const int rc = decode_prog_segment(im, sc, sg, p.huff, nat, p.streams, p.coef + im.coef_off, p.nzmask + im.coef_off / 64,
                                       sc.Ah != 0 ? p.refine + sc.out_block : nullptr);
    if (rc) atomicMax(p.status + sc.image, rc);
}

__global__ void __launch_bounds__(256) jpegdec_mask_kernel(JpegDecParams p, uint32_t n_blocks) {
    __shared__ uint8_t nat[64];
    if (threadIdx.x < 64) nat[threadIdx.x] = (uint8_t)rod::jpeg::natural_order(threadIdx.x);
    __syncthreads();
    const uint32_t b = blockIdx.x * 256u + threadIdx.x;
    if (b < n_blocks) p.nzmask[b] = zigzag_nz_mask(p.coef + 64ull * b, nat);
}

// grid (blocks of the level's largest refinement scan / 256, refinement scans of the level: scans[])
__global__ void __launch_bounds__(256) jpegdec_apply_kernel(JpegDecParams p, const uint32_t* scans) {
    __shared__ uint8_t nat[64];
    if (threadIdx.x < 64) nat[threadIdx.x] = (uint8_t)rod::jpeg::natural_order(threadIdx.x);
    __syncthreads();
    const ScanRec sc = p.scans[scans[blockIdx.y]];
    if (p.status[sc.image] != 0) return;
    const ImageRec im = p.images[sc.image];
    const uint32_t j = blockIdx.x * 256u + threadIdx.x;
    if (j >= scan_units(im, sc) * scan_blocks_per_unit(im, sc)) return;
    apply_refinement(scan_block(p.coef + im.coef_off, im, sc, j), sc, p.refine[sc.out_block + j], nat);
}

// DC prediction (jdhuff.c: last_dc_val[ci] += diff): inclusive prefix sum of the stored differences of one component, in
// the order the blocks were coded, from 0 in every restart interval.  grid (n_segs, 3), 256 threads.
__global__ void __launch_bounds__(256) jpegdec_dc_kernel(JpegDecParams p) {
    __shared__ int warp_sum[8];
    __shared__ int carry_s;
    const int comp = blockIdx.y;
    const SegRec sg = p.segs[blockIdx.x];
    const ImageRec im = p.images[sg.image];
    if (p.status[sg.image] != 0 || comp >= im.ncomp) return;
    const Layout L = layout_of(im);
    const uint32_t n = (uint32_t)(comp == 0 ? L.nl : 1) * (sg.n_blocks / (uint32_t)L.nb);
    int16_t* coef = p.coef + im.coef_off;
    if (threadIdx.x == 0) carry_s = 0;
    __syncthreads();
    for (uint32_t base = 0; base < n; base += 256) {
        const uint32_t j = base + threadIdx.x;
        int16_t* blk = nullptr;
        if (j < n)
            blk = block_of(coef, L, sg.first_block + (comp == 0 ? (uint32_t)L.nb * (j / (uint32_t)L.nl) + j % (uint32_t)L.nl
                                                                : (uint32_t)L.nb * j + (uint32_t)(L.nl + comp - 1)));
        const int v = blk ? (int)blk[0] : 0;
        int x = v;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const int y = __shfl_up_sync(0xFFFFFFFFu, x, d);
            if ((threadIdx.x & 31) >= d) x += y;
        }
        if ((threadIdx.x & 31) == 31) warp_sum[threadIdx.x >> 5] = x;
        __syncthreads();
        int before = carry_s;
        for (int w = 0; w < (int)(threadIdx.x >> 5); ++w) before += warp_sum[w];
        if (blk) blk[0] = (int16_t)(before + x);
        __syncthreads();
        if (threadIdx.x == 255) carry_s = before + x;
        __syncthreads();
    }
}

__global__ void __launch_bounds__(128) jpegdec_idct_kernel(JpegDecParams p) {   // grid (blocks of the largest image / 128, image)
    const int img = blockIdx.y;
    const ImageRec im = p.images[img];
    if (im.h == 0 || __ldg(p.status + img) != 0) return;
    const uint32_t b = blockIdx.x * 128u + threadIdx.x;
    if (b >= __ldg(p.block_start + img + 1) - __ldg(p.block_start + img)) return;
    const Layout L = layout_of(im);
    const uint32_t yblocks = (uint32_t)(L.nl * L.mcus), cblocks = (uint32_t)L.mcus;
    int comp;
    uint32_t bi;
    long pitch;
    uint8_t* plane = p.planes + im.plane_off;
    if (b < yblocks) { comp = 0; bi = b; pitch = 8L * L.hs * L.mcu_w; }
    else if (b < yblocks + cblocks) { comp = 1; bi = b - yblocks; pitch = 8L * L.mcu_w; plane += 64L * yblocks; }
    else { comp = 2; bi = b - yblocks - cblocks; pitch = 8L * L.mcu_w; plane += 64L * (yblocks + cblocks); }
    const uint32_t bpr = (uint32_t)(pitch >> 3);
    const uint32_t by = bi / bpr, bx = bi - by * bpr;
    __align__(16) int16_t c[64];
    {
        const uint4* src = reinterpret_cast<const uint4*>(p.coef + im.coef_off + 64ull * b);
        uint4* dst = reinterpret_cast<uint4*>(c);
#pragma unroll
        for (int i = 0; i < 8; ++i) dst[i] = src[i];
    }
    __align__(16) uint16_t q[64];
    {
        const uint4* src = reinterpret_cast<const uint4*>(p.tables[im.table_set].quant[comp]);
        uint4* dst = reinterpret_cast<uint4*>(q);
#pragma unroll
        for (int i = 0; i < 8; ++i) dst[i] = __ldg(src + i);
    }
    __align__(8) uint8_t o[64];
    idct_islow(c, q, o, 8);
    uint8_t* dst = plane + (8L * by) * pitch + 8 * bx;
#pragma unroll
    for (int r = 0; r < 8; ++r) *reinterpret_cast<uint2*>(dst + r * pitch) = *reinterpret_cast<const uint2*>(o + 8 * r);
}

__global__ void __launch_bounds__(256) jpegdec_color_kernel(JpegDecParams p) {   // grid (quads of the largest image / 256, image)
    const int img = blockIdx.y;
    const ImageRec im = p.images[img];
    if (im.h == 0 || __ldg(p.status + img) != 0) return;
    const uint32_t k = blockIdx.x * 256u + threadIdx.x;
    if (k >= __ldg(p.quad_start + img + 1) - __ldg(p.quad_start + img)) return;
    const Layout L = layout_of(im);
    const int qw = (im.w + 3) >> 2;   // groups of four pixels per row
    const int cw = (im.w + L.hs - 1) / L.hs, ch = (im.h + L.vs - 1) / L.vs;
    const int y = (int)(k / (uint32_t)qw), x0 = 4 * (int)(k - (uint32_t)y * (uint32_t)qw);
    const long ypitch = 8L * L.hs * L.mcu_w, cpitch = 8L * L.mcu_w;
    const uint8_t* yp = p.planes + im.plane_off;
    const uint8_t* cbp = yp + 64L * L.nl * L.mcus;
    const uint8_t* crp = cbp + 64L * L.mcus;
    uint8_t* out = p.pixels + im.dst_off + (int64_t)y * im.dst_pitch + 3 * x0;
    const int nv = min(4, im.w - x0);
    const uint32_t y4 = *reinterpret_cast<const uint32_t*>(yp + y * ypitch + x0);   // (the plane is padded to whole blocks)
    uint32_t w[3] = {0u, 0u, 0u};   // the twelve output bytes
    int cb[4] = {128, 128, 128, 128}, cr[4] = {128, 128, 128, 128};
    if (im.ncomp == 3) {
        chroma_quad(cbp, cpitch, L.hs, L.vs, cw, ch, x0, y, cb);
        chroma_quad(crp, cpitch, L.hs, L.vs, cw, ch, x0, y, cr);
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const int yy = (int)((y4 >> (8 * i)) & 0xFFu);
        uint8_t t[3];
        if (im.ncomp == 1) t[0] = t[1] = t[2] = (uint8_t)yy;
        else ycc_to_bgr(yy, cb[i], cr[i], t);
#pragma unroll
        for (int c = 0; c < 3; ++c) w[(3 * i + c) >> 2] |= (uint32_t)t[c] << (8 * ((3 * i + c) & 3));
    }
    const uint32_t w0 = w[0], w1 = w[1], w2 = w[2];
    if (nv < 4) {
        for (int i = 0; i < 3 * nv; ++i) out[i] = (uint8_t)((i < 4 ? w0 : (i < 8 ? w1 : w2)) >> (8 * (i & 3)));
        return;
    }
    const uint32_t a = (uint32_t)((uintptr_t)out & 3u);
    if (a == 0) {   // twelve bytes as aligned words, whatever the row's byte phase is
        uint32_t* o = reinterpret_cast<uint32_t*>(out);
        o[0] = w0; o[1] = w1; o[2] = w2;
    } else if (a == 2) {
        *reinterpret_cast<uint16_t*>(out) = (uint16_t)w0;
        uint32_t* o = reinterpret_cast<uint32_t*>(out + 2);
        o[0] = __funnelshift_r(w0, w1, 16); o[1] = __funnelshift_r(w1, w2, 16);
        *reinterpret_cast<uint16_t*>(out + 10) = (uint16_t)(w2 >> 16);
    } else if (a == 1) {
        out[0] = (uint8_t)w0;
        *reinterpret_cast<uint16_t*>(out + 1) = (uint16_t)(w0 >> 8);
        uint32_t* o = reinterpret_cast<uint32_t*>(out + 3);
        o[0] = __funnelshift_r(w0, w1, 24); o[1] = __funnelshift_r(w1, w2, 24);
        out[11] = (uint8_t)(w2 >> 24);
    } else {
        out[0] = (uint8_t)w0;
        uint32_t* o = reinterpret_cast<uint32_t*>(out + 1);
        o[0] = __funnelshift_r(w0, w1, 8); o[1] = __funnelshift_r(w1, w2, 8);
        *reinterpret_cast<uint16_t*>(out + 9) = (uint16_t)(w2 >> 8);
        out[11] = (uint8_t)(w2 >> 24);
    }
}

}  // namespace rod

using namespace rod;

// Page-locked staging blocks are recycled like the device blocks (pinning costs ~0.3 ms per MB, more than the decoding).
#include <mutex>
namespace {
std::mutex g_host_mutex;
std::multimap<size_t, void*> g_host_cache;   // rounded size -> free page-locked block
size_t g_host_cache_bytes = 0;
constexpr size_t kHostCacheLimit = (size_t)4 << 30;   // page-locked memory parked here at most
size_t round_host(size_t n) {
    size_t r = 1 << 20;
    while (r < n) r <<= 1;
    return r;
}
cudaError_t host_cache_alloc(void** p, size_t n) {
    const size_t r = round_host(n);
    {
        std::lock_guard<std::mutex> lock(g_host_mutex);
        auto it = g_host_cache.find(r);
        if (it != g_host_cache.end()) { *p = it->second; g_host_cache.erase(it); g_host_cache_bytes -= r; return cudaSuccess; }
    }
    return cudaHostAlloc(p, r, cudaHostAllocDefault);
}
void host_cache_free(void* p, size_t n) {
    if (p == nullptr) return;
    const size_t r = round_host(n);
    {
        std::lock_guard<std::mutex> lock(g_host_mutex);
        if (g_host_cache_bytes + r <= kHostCacheLimit) {
            g_host_cache.insert({r, p});
            g_host_cache_bytes += r;
            return;
        }
    }
    cudaFreeHost(p);
}
}  // namespace

extern "C" void rod_jpegdec_trim(void) {
    std::lock_guard<std::mutex> lock(g_host_mutex);
    for (auto& kv : g_host_cache) cudaFreeHost(kv.second);
    g_host_cache.clear();
    g_host_cache_bytes = 0;
}

struct rod_jpeg_decoder {
    int device = 0;
    int n_images = 0;
    std::vector<ImageRec> h_images;
    std::vector<int32_t> h_status;       // host verdict per image: 0 decodable, else 10 + ParseStatus / 13 (no EOI)
    std::vector<TableSet> h_tables;
    std::vector<uint32_t> h_block_start, h_quad_start, h_sub_start;
    std::vector<uint2> h_ctas;
    std::vector<SegRec> h_segs;
    std::vector<ScanRec> h_scans;        // progressive files
    std::vector<ScanSeg> h_psegs;        // ... their restart intervals, level by level
    std::vector<uint32_t> h_level_start; // [levels + 1] into h_psegs
    std::vector<HuffTab> h_huff;         // ... the Huffman tables of their scans (equal tables shared)
    std::vector<uint32_t> h_refine_scans, h_refine_start;   // ... their refinement scans by level: [levels + 1] into the list
    std::vector<uint32_t> h_refine_max;  // ... blocks of the level's largest refinement scan
    std::vector<char> h_level_ac_refine; // ... the level has an AC refinement scan (it needs the history masks)
    size_t refine_blocks = 0;
    int n_sm = 148;
    uint8_t* h_streams = nullptr;        // page-locked
    size_t stream_bytes = 0, coef_elems = 0, plane_bytes = 0;
    ImageRec* d_images = nullptr;
    TableSet* d_tables = nullptr;
    uint32_t* d_block_start = nullptr;
    uint32_t* d_quad_start = nullptr;
    uint32_t* d_sub_start = nullptr;
    uint2* d_ctas = nullptr;
    SegRec* d_segs = nullptr;
    ScanRec* d_scans = nullptr;
    ScanSeg* d_psegs = nullptr;
    HuffTab* d_huff = nullptr;
    uint32_t* d_refine_scans = nullptr;
    uint64_t* d_nzmask = nullptr;
    RefineOut* d_refine = nullptr;
    unsigned int* d_changed = nullptr;
    uint64_t* d_end_state = nullptr;
    uint64_t* d_used_start = nullptr;
    uint32_t* d_first_block = nullptr;
    size_t n_sub = 0;
    uint8_t* d_small = nullptr;
    size_t small_bytes = 0;
    int sync_rounds = 0;                 // launches of the last decode (diagnostics)
    bool in_flight = false;              // decode() issued, status() not yet waited for
    int32_t* d_status = nullptr;
    uint8_t* d_streams = nullptr;
    int16_t* d_coef = nullptr;
    uint8_t* d_planes = nullptr;
};

extern "C" int rod_jpegdec_probe_ex(const uint8_t* file, uint64_t n, int formats, int* height, int* width) {
    if (file == nullptr || height == nullptr || width == nullptr || formats < 1 || formats > (kBaseline | kProgressive))
        return ROD_ERR_INVALID_ARG;
    FileInfo info;
    std::vector<TableSet> ts(1);
    const ParseStatus st = parse_file(file, (size_t)n, &info, &ts[0], formats);   // (a progressive file: every scan checked)
    if (st != PARSE_OK || (info.progressive ? !(formats & kProgressive) : !(formats & kBaseline))) return ROD_ERR_UNSUPPORTED;
    *height = info.height;
    *width = info.width;
    return ROD_OK;
}

extern "C" int rod_jpegdec_probe(const uint8_t* file, uint64_t n, int* height, int* width) {
    return rod_jpegdec_probe_ex(file, n, kBaseline, height, width);
}

extern "C" void rod_jpegdec_destroy(rod_jpeg_decoder* d) {
    if (d == nullptr) return;
    if (d->in_flight) cudaDeviceSynchronize();   // the buffers go to caches and may be reused at once
    block_cache_free(d->device, d->d_small, d->small_bytes);   // the descriptor arrays are carved out of one block
    block_cache_free(d->device, d->d_streams, d->stream_bytes);
    block_cache_free(d->device, d->d_coef, d->coef_elems * sizeof(int16_t));
    block_cache_free(d->device, d->d_planes, d->plane_bytes);
    block_cache_free(d->device, d->d_end_state, d->n_sub * sizeof(uint64_t));
    block_cache_free(d->device, d->d_used_start, d->n_sub * sizeof(uint64_t));
    block_cache_free(d->device, d->d_first_block, d->n_sub * sizeof(uint32_t));
    block_cache_free(d->device, d->d_nzmask, d->coef_elems / 64 * sizeof(uint64_t));
    block_cache_free(d->device, d->d_refine, d->refine_blocks * sizeof(RefineOut));
    host_cache_free(d->h_streams, d->stream_bytes);
    delete d;
}

extern "C" int rod_jpegdec_create_ex(const uint8_t* const* files, const uint64_t* lens, int n_images, const uint64_t* dst_offsets,
                                     const int64_t* dst_pitches, int host_threads, int formats, rod_jpeg_decoder** out_dec) {
    if (files == nullptr || lens == nullptr || dst_offsets == nullptr || n_images < 1 || out_dec == nullptr || formats < 1 ||
        formats > (kBaseline | kProgressive))
        return ROD_ERR_INVALID_ARG;
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) { cudaGetLastError(); return ROD_ERR_NO_DEVICE; }
    rod_jpeg_decoder* d = new (std::nothrow) rod_jpeg_decoder();
    if (d == nullptr) return ROD_ERR_OOM;
    if (cudaGetDevice(&d->device) != cudaSuccess) { delete d; cudaGetLastError(); return ROD_ERR_NO_DEVICE; }
    d->n_images = n_images;
    d->h_images.assign(n_images, ImageRec{});
    d->h_status.assign(n_images, 0);
    // stream slots: a file's unstuffed scans are never longer than the file
    std::vector<uint64_t> slot(n_images + 1, 0);
    for (int i = 0; i < n_images; ++i) slot[i + 1] = slot[i] + ((lens[i] + 32 + 15) & ~(uint64_t)15);
    d->stream_bytes = (size_t)slot[n_images] + 64;
    if (host_cache_alloc((void**)&d->h_streams, d->stream_bytes) != cudaSuccess) {
        cudaGetLastError();
        rod_jpegdec_destroy(d);
        return ROD_ERR_OOM;
    }
    std::vector<TableSet> per_image(n_images);
    std::vector<std::vector<SegRec>> per_image_segs(n_images);
    std::vector<FileInfo> per_image_prog(n_images);   // progressive files: scans and tables
    std::vector<std::vector<ScanSeg>> per_image_psegs(n_images);
    auto work = [&](int lo, int hi) {
        for (int i = lo; i < hi; ++i) {
            ImageRec& im = d->h_images[i];
            FileInfo info;
            ParseStatus st = files[i] ? parse_file(files[i], (size_t)lens[i], &info, &per_image[i], formats, d->h_streams + slot[i])
                                      : PARSE_NOT_JPEG;
            if (st == PARSE_OK && !(formats & (info.progressive ? kProgressive : kBaseline))) st = PARSE_UNSUPPORTED;
            if (st != PARSE_OK) { d->h_status[i] = 10 + (int)st; continue; }
            if (info.progressive) {
                ImageRec r{};
                r.h = info.height; r.w = info.width;
                r.hs = (uint8_t)info.hs; r.vs = (uint8_t)info.vs; r.ncomp = (uint8_t)info.ncomp;
                r.stream_bytes = (uint32_t)info.stream_bytes;
                r.stream_off = slot[i];
                r.dst_off = dst_offsets[i];
                r.dst_pitch = (dst_pitches && dst_pitches[i]) ? dst_pitches[i] : 3LL * info.width;
                bool ok = true;
                for (size_t s = 0; s < info.scans.size() && ok; ++s)   // (scan: index within the file until the batch is laid out)
                    ok = make_scan_segments(r, info.scans[s], (uint32_t)s, slot[i], &per_image_psegs[i]);
                if (!ok) { d->h_status[i] = 13; continue; }
                per_image_prog[i] = std::move(info);
                im = r;
                continue;
            }
            std::vector<uint32_t> rst;
            const size_t sb = unstuff_scan(files[i], (size_t)lens[i], info.scan_begin, d->h_streams + slot[i], &rst);
            if (sb == (size_t)-1) { d->h_status[i] = 13; continue; }
            ImageRec r{};
            r.h = info.height; r.w = info.width;
            r.hs = (uint8_t)info.hs; r.vs = (uint8_t)info.vs; r.ncomp = (uint8_t)info.ncomp;
            r.stream_bytes = (uint32_t)sb;
            r.stream_off = slot[i];
            r.dst_off = dst_offsets[i];
            r.dst_pitch = (dst_pitches && dst_pitches[i]) ? dst_pitches[i] : 3LL * info.width;
            // the restart markers found must be the ones the DRI segment announces
            if (!make_segments(r, (uint32_t)i, info.restart_interval, slot[i], sb, rst, &per_image_segs[i])) { d->h_status[i] = 13; continue; }
            im = r;
        }
    };
    {
        int nt = host_threads < 1 ? 1 : (host_threads > 64 ? 64 : host_threads);
        if (nt > n_images) nt = n_images;
        // a thread is worth starting for about a megabyte of file data (unstuffing runs at memory speed)
        const uint64_t by_bytes = 1 + (slot[n_images] >> 20);
        if ((uint64_t)nt > by_bytes) nt = (int)by_bytes;
        std::vector<std::thread> th;
        for (int t = 1; t < nt; ++t) th.emplace_back(work, (int)((long)n_images * t / nt), (int)((long)n_images * (t + 1) / nt));
        work(0, (int)((long)n_images / nt));
        for (auto& t : th) t.join();
    }
    // shared table sets, buffer layout
    std::map<std::string, int> seen, seen_huff;
    std::vector<std::vector<ScanSeg>> by_level;
    std::vector<std::vector<uint32_t>> refine_by_level;
    d->h_block_start.assign(n_images + 1, 0);
    d->h_quad_start.assign(n_images + 1, 0);
    d->h_sub_start.assign(1, 0);
    uint64_t blocks = 0, quads = 0, subs = 0;
    for (int i = 0; i < n_images; ++i) {
        ImageRec& im = d->h_images[i];
        if (d->h_status[i] == 0) {
            std::string key(reinterpret_cast<const char*>(&per_image[i]), sizeof(TableSet));
            auto it = seen.find(key);
            if (it == seen.end()) {
                it = seen.emplace(std::move(key), (int)d->h_tables.size()).first;
                d->h_tables.push_back(per_image[i]);
            }
            im.table_set = it->second;
            const Layout L = layout_of(im);
            const uint64_t nblocks = (uint64_t)L.mcus * (uint64_t)L.nb;
            im.coef_off = d->coef_elems;
            im.plane_off = d->plane_bytes;
            d->coef_elems += nblocks * 64;
            d->plane_bytes += nblocks * 64;
            blocks += nblocks;
            quads += (uint64_t)im.h * (uint64_t)((im.w + 3) >> 2);
            if (per_image_prog[i].progressive) {   // scans, tables, restart intervals by level
                FileInfo& pf = per_image_prog[i];
                std::vector<int32_t> tab(pf.huff.size());
                for (size_t t = 0; t < pf.huff.size(); ++t) {
                    std::string hk(reinterpret_cast<const char*>(&pf.huff[t]), sizeof(HuffTab));
                    auto ht = seen_huff.find(hk);
                    if (ht == seen_huff.end()) {
                        ht = seen_huff.emplace(std::move(hk), (int)d->h_huff.size()).first;
                        d->h_huff.push_back(pf.huff[t]);
                    }
                    tab[t] = ht->second;
                }
                std::vector<int> level;
                const int n_levels = scan_levels(pf.scans, &level);
                if ((int)by_level.size() < n_levels) by_level.resize(n_levels);
                if (refine_by_level.size() < (size_t)n_levels) {
                    refine_by_level.resize(n_levels);
                    d->h_refine_max.resize(n_levels, 0);
                    d->h_level_ac_refine.resize(n_levels, 0);
                }
                const uint32_t scan0 = (uint32_t)d->h_scans.size();
                for (size_t s = 0; s < pf.scans.size(); ++s) {
                    const ScanInfo& si = pf.scans[s];
                    ScanRec r = si.rec;
                    r.image = (uint32_t)i;
                    for (int j = 0; j < 3; ++j) r.dc_tab[j] = si.dc_slot[j] >= 0 ? tab[si.dc_slot[j]] : -1;
                    r.ac_tab = si.ac_slot >= 0 ? tab[si.ac_slot] : -1;
                    if (r.Ah != 0) {   // a refinement scan: room for its results, applied after its level
                        const uint32_t nb = scan_units(im, r) * scan_blocks_per_unit(im, r);
                        r.out_block = (uint32_t)d->refine_blocks;
                        d->refine_blocks += nb;
                        refine_by_level[level[s]].push_back(scan0 + (uint32_t)s);
                        d->h_refine_max[level[s]] = std::max(d->h_refine_max[level[s]], nb);
                        if (r.Ss != 0) d->h_level_ac_refine[level[s]] = 1;
                    }
                    d->h_scans.push_back(r);
                }
                for (ScanSeg sg : per_image_psegs[i]) {
                    const int lv = level[sg.scan];
                    sg.scan += scan0;
                    by_level[lv].push_back(sg);
                }
            }
            for (const SegRec& sg : per_image_segs[i]) {
                const uint32_t bits = 8u * (sg.stream_bytes - sg.byte0);
                const uint32_t n_sub = bits ? (bits + kSubBits - 1) / kSubBits : 1u;
                const unsigned seg = (unsigned)d->h_segs.size();
                for (uint32_t s0 = 0; s0 < n_sub; s0 += kHuffThreads) d->h_ctas.push_back(make_uint2(seg, s0));
                subs += n_sub;
                d->h_segs.push_back(sg);
                d->h_sub_start.push_back((uint32_t)subs);
            }
        }
        d->h_block_start[i + 1] = (uint32_t)blocks;
        d->h_quad_start[i + 1] = (uint32_t)quads;
    }
    d->n_sub = (size_t)subs;
    d->h_level_start.assign(1, 0);
    for (std::vector<ScanSeg>& lv : by_level) {   // the longest intervals first: they start in the first wave of the launch
        std::stable_sort(lv.begin(), lv.end(), [](const ScanSeg& a, const ScanSeg& b) { return a.stream_bytes > b.stream_bytes; });
        d->h_psegs.insert(d->h_psegs.end(), lv.begin(), lv.end());
        d->h_level_start.push_back((uint32_t)d->h_psegs.size());
    }
    d->h_refine_start.assign(1, 0);
    for (const std::vector<uint32_t>& lv : refine_by_level) {
        d->h_refine_scans.insert(d->h_refine_scans.end(), lv.begin(), lv.end());
        d->h_refine_start.push_back((uint32_t)d->h_refine_scans.size());
    }
    if (d->refine_blocks >= (1ull << 32)) { rod_jpegdec_destroy(d); return ROD_ERR_UNSUPPORTED; }
    if (!d->h_psegs.empty() && cudaDeviceGetAttribute(&d->n_sm, cudaDevAttrMultiProcessorCount, d->device) != cudaSuccess) {
        rod_jpegdec_destroy(d);
        return cuda_fail(cudaGetLastError());
    }
    if (blocks >= (1ull << 32) || quads >= (1ull << 32) || subs >= (1ull << 32)) { rod_jpegdec_destroy(d); return ROD_ERR_UNSUPPORTED; }
    if (d->h_tables.empty()) d->h_tables.push_back(TableSet{});
    cudaError_t err = cudaSuccess;
    auto calloc_ = [&](void** p, size_t n) { if (err == cudaSuccess) err = block_cache_alloc(d->device, p, n ? n : 16); };
    // descriptor arrays: one cached block (cudaMalloc / cudaFree per decoder would synchronise the device every batch)
    size_t sizes[13] = {sizeof(ImageRec) * n_images, sizeof(TableSet) * d->h_tables.size(), sizeof(uint32_t) * (n_images + 1),
                        sizeof(uint32_t) * (n_images + 1), sizeof(int32_t) * n_images, sizeof(uint32_t) * d->h_sub_start.size(),
                        sizeof(SegRec) * d->h_segs.size(), sizeof(uint2) * d->h_ctas.size(), sizeof(unsigned int) * 4,
                        sizeof(ScanRec) * d->h_scans.size(), sizeof(ScanSeg) * d->h_psegs.size(), sizeof(HuffTab) * d->h_huff.size(),
                        sizeof(uint32_t) * d->h_refine_scans.size()};
    size_t offs[13];
    for (int q = 0; q < 13; ++q) { offs[q] = d->small_bytes; d->small_bytes += (sizes[q] + 255) & ~(size_t)255; }
    calloc_((void**)&d->d_small, d->small_bytes);
    if (err == cudaSuccess) {
        d->d_images = reinterpret_cast<ImageRec*>(d->d_small + offs[0]);
        d->d_tables = reinterpret_cast<TableSet*>(d->d_small + offs[1]);
        d->d_block_start = reinterpret_cast<uint32_t*>(d->d_small + offs[2]);
        d->d_quad_start = reinterpret_cast<uint32_t*>(d->d_small + offs[3]);
        d->d_status = reinterpret_cast<int32_t*>(d->d_small + offs[4]);
        d->d_sub_start = reinterpret_cast<uint32_t*>(d->d_small + offs[5]);
        d->d_segs = reinterpret_cast<SegRec*>(d->d_small + offs[6]);
        d->d_ctas = reinterpret_cast<uint2*>(d->d_small + offs[7]);
        d->d_changed = reinterpret_cast<unsigned int*>(d->d_small + offs[8]);
        d->d_scans = reinterpret_cast<ScanRec*>(d->d_small + offs[9]);
        d->d_psegs = reinterpret_cast<ScanSeg*>(d->d_small + offs[10]);
        d->d_huff = reinterpret_cast<HuffTab*>(d->d_small + offs[11]);
        d->d_refine_scans = reinterpret_cast<uint32_t*>(d->d_small + offs[12]);
    }
    calloc_((void**)&d->d_end_state, d->n_sub * sizeof(uint64_t));
    calloc_((void**)&d->d_used_start, d->n_sub * sizeof(uint64_t));
    calloc_((void**)&d->d_first_block, d->n_sub * sizeof(uint32_t));
    calloc_((void**)&d->d_streams, d->stream_bytes);
    calloc_((void**)&d->d_coef, d->coef_elems * sizeof(int16_t));
    calloc_((void**)&d->d_planes, d->plane_bytes);
    if (d->refine_blocks) {
        calloc_((void**)&d->d_nzmask, d->coef_elems / 64 * sizeof(uint64_t));
        calloc_((void**)&d->d_refine, d->refine_blocks * sizeof(RefineOut));
    }
    if (err != cudaSuccess) {
        rod_jpegdec_destroy(d);
        return cuda_fail(err);
    }
    *out_dec = d;
    return ROD_OK;
}

extern "C" int rod_jpegdec_create(const uint8_t* const* files, const uint64_t* lens, int n_images, const uint64_t* dst_offsets,
                                  const int64_t* dst_pitches, int host_threads, rod_jpeg_decoder** out_dec) {
    return rod_jpegdec_create_ex(files, lens, n_images, dst_offsets, dst_pitches, host_threads, kBaseline, out_dec);
}

extern "C" int rod_jpegdec_host_status(const rod_jpeg_decoder* d, int32_t* status, int32_t* heights, int32_t* widths) {
    if (d == nullptr || status == nullptr) return ROD_ERR_INVALID_ARG;
    for (int i = 0; i < d->n_images; ++i) {
        status[i] = d->h_status[i];
        if (heights) heights[i] = d->h_images[i].h;
        if (widths) widths[i] = d->h_images[i].w;
    }
    return ROD_OK;
}

extern "C" int rod_jpegdec_decode(rod_jpeg_decoder* d, uint8_t* pixels, void* stream) {
    if (d == nullptr || pixels == nullptr) return ROD_ERR_INVALID_ARG;
    cudaStream_t st = (cudaStream_t)stream;
    const int n = d->n_images;
    ROD_CUDA(cudaMemcpyAsync(d->d_images, d->h_images.data(), sizeof(ImageRec) * n, cudaMemcpyHostToDevice, st));
    ROD_CUDA(cudaMemcpyAsync(d->d_tables, d->h_tables.data(), sizeof(TableSet) * d->h_tables.size(), cudaMemcpyHostToDevice, st));
    ROD_CUDA(cudaMemcpyAsync(d->d_block_start, d->h_block_start.data(), sizeof(uint32_t) * (n + 1), cudaMemcpyHostToDevice, st));
    ROD_CUDA(cudaMemcpyAsync(d->d_quad_start, d->h_quad_start.data(), sizeof(uint32_t) * (n + 1), cudaMemcpyHostToDevice, st));
    ROD_CUDA(cudaMemcpyAsync(d->d_status, d->h_status.data(), sizeof(int32_t) * n, cudaMemcpyHostToDevice, st));
    ROD_CUDA(cudaMemcpyAsync(d->d_sub_start, d->h_sub_start.data(), sizeof(uint32_t) * d->h_sub_start.size(), cudaMemcpyHostToDevice, st));
    if (!d->h_segs.empty())
        ROD_CUDA(cudaMemcpyAsync(d->d_segs, d->h_segs.data(), sizeof(SegRec) * d->h_segs.size(), cudaMemcpyHostToDevice, st));
    if (!d->h_ctas.empty())
        ROD_CUDA(cudaMemcpyAsync(d->d_ctas, d->h_ctas.data(), sizeof(uint2) * d->h_ctas.size(), cudaMemcpyHostToDevice, st));
    if (!d->h_psegs.empty()) {
        ROD_CUDA(cudaMemcpyAsync(d->d_scans, d->h_scans.data(), sizeof(ScanRec) * d->h_scans.size(), cudaMemcpyHostToDevice, st));
        ROD_CUDA(cudaMemcpyAsync(d->d_psegs, d->h_psegs.data(), sizeof(ScanSeg) * d->h_psegs.size(), cudaMemcpyHostToDevice, st));
        ROD_CUDA(cudaMemcpyAsync(d->d_huff, d->h_huff.data(), sizeof(HuffTab) * d->h_huff.size(), cudaMemcpyHostToDevice, st));
        if (!d->h_refine_scans.empty())
            ROD_CUDA(cudaMemcpyAsync(d->d_refine_scans, d->h_refine_scans.data(), sizeof(uint32_t) * d->h_refine_scans.size(),
                                     cudaMemcpyHostToDevice, st));
    }
    ROD_CUDA(cudaMemcpyAsync(d->d_streams, d->h_streams, d->stream_bytes, cudaMemcpyHostToDevice, st));
    d->in_flight = true;
    if (d->coef_elems == 0 || (d->h_ctas.empty() && d->h_psegs.empty())) return ROD_OK;
    ROD_CUDA(cudaMemsetAsync(d->d_coef, 0, d->coef_elems * sizeof(int16_t), st));
    JpegDecParams p;
    p.images = d->d_images; p.tables = d->d_tables; p.streams = d->d_streams; p.coef = d->d_coef; p.planes = d->d_planes;
    p.pixels = pixels; p.status = d->d_status; p.block_start = d->d_block_start; p.quad_start = d->d_quad_start;
    p.segs = d->d_segs; p.n_segs = (int)d->h_segs.size();
    p.sub_start = d->d_sub_start; p.ctas = d->d_ctas; p.end_state = d->d_end_state; p.used_start = d->d_used_start;
    p.first_block = d->d_first_block; p.changed = d->d_changed;
    p.n_images = n;
    p.scans = d->d_scans; p.psegs = d->d_psegs; p.huff = d->d_huff; p.nzmask = d->d_nzmask; p.refine = d->d_refine;
    if (!d->h_psegs.empty()) {   // progressive scans, level by level
        const uint32_t n_sm = (uint32_t)d->n_sm;
        for (size_t lv = 0; lv + 1 < d->h_level_start.size(); ++lv) {
            if (d->h_level_ac_refine[lv]) {
                const uint32_t nb = (uint32_t)(d->coef_elems / 64);
                jpegdec_mask_kernel<<<(nb + 255) / 256, 256, 0, st>>>(p, nb);
            }
            const uint32_t s0 = d->h_level_start[lv], ns = d->h_level_start[lv + 1] - s0;
            // a warp per interval while every SM gets at most 32 warps of them, more lanes per warp beyond
            const uint32_t lanes = std::min<uint32_t>(32u, (ns + 32u * n_sm - 1) / (32u * n_sm));
            const uint32_t warps = (ns + lanes - 1) / lanes;
            jpegdec_prog_kernel<<<(warps + 3) / 4, 128, 0, st>>>(p, s0, ns, lanes);
            for (uint32_t r0 = d->h_refine_start[lv]; r0 < d->h_refine_start[lv + 1]; r0 += 65535) {   // (grid.y <= 65535)
                const uint32_t nr = std::min<uint32_t>(d->h_refine_start[lv + 1] - r0, 65535u);
                jpegdec_apply_kernel<<<dim3((d->h_refine_max[lv] + 255) / 256, nr), 256, 0, st>>>(p, d->d_refine_scans + r0);
            }
        }
    }
    const unsigned n_ctas = (unsigned)d->h_ctas.size();
    d->sync_rounds = 0;
    if (n_ctas > 0) {   // baseline scans
        jpegdec_guess_kernel<<<n_ctas, kHuffThreads, 0, st>>>(p);
        // synchronisation rounds, four launches per host round trip, until a launch changes no end state
        for (;;) {
            unsigned int flags[4];
            ROD_CUDA(cudaMemsetAsync(d->d_changed, 0, sizeof(flags), st));
            for (int q = 0; q < 4; ++q) jpegdec_sync_kernel<<<n_ctas, kHuffThreads, 0, st>>>(p, q);
            ROD_CUDA(cudaMemcpyAsync(flags, d->d_changed, sizeof(flags), cudaMemcpyDeviceToHost, st));
            ROD_CUDA(cudaStreamSynchronize(st));
            d->sync_rounds += 4;
            if (!(flags[0] && flags[1] && flags[2] && flags[3])) break;
        }
        jpegdec_scan_kernel<<<p.n_segs, 256, 0, st>>>(p);
        jpegdec_write_kernel<<<n_ctas, kHuffThreads, 0, st>>>(p);
        jpegdec_dc_kernel<<<dim3(p.n_segs, 3), 256, 0, st>>>(p);
    }
    uint32_t max_blocks = 0, max_quads = 0;
    for (int i = 0; i < n; ++i) {
        max_blocks = std::max(max_blocks, d->h_block_start[i + 1] - d->h_block_start[i]);
        max_quads = std::max(max_quads, d->h_quad_start[i + 1] - d->h_quad_start[i]);
    }
    for (int i0 = 0; i0 < n; i0 += 65535) {   // (grid.y is limited to 65535)
        JpegDecParams q = p;
        q.images += i0; q.status += i0; q.block_start += i0; q.quad_start += i0;
        const int ny = std::min(n - i0, 65535);
        jpegdec_idct_kernel<<<dim3((max_blocks + 127) / 128, ny), 128, 0, st>>>(q);
        jpegdec_color_kernel<<<dim3((max_quads + 255) / 256, ny), 256, 0, st>>>(q);
    }
    ROD_CUDA(cudaGetLastError());
    return ROD_OK;
}

// per-image result after the work on `stream` is complete: 0 decoded; 1 / 2 corrupt / short stream (pixels undefined);
// >= 10 not decodable on the device (the verdict of rod_jpegdec_create)
extern "C" int rod_jpegdec_status(rod_jpeg_decoder* d, int32_t* status, void* stream) {
    if (d == nullptr || status == nullptr) return ROD_ERR_INVALID_ARG;
    cudaStream_t st = (cudaStream_t)stream;
    ROD_CUDA(cudaMemcpyAsync(status, d->d_status, sizeof(int32_t) * d->n_images, cudaMemcpyDeviceToHost, st));
    ROD_CUDA(cudaStreamSynchronize(st));
    d->in_flight = false;
    return ROD_OK;
}
