// letterbox.cu -- training-path output stage (BASELINE config 5): uint8 HWC BGR -> fp16 NCHW RGB
// with Ultralytics' LetterBox (INTER_LINEAR resize-to-fit + constant pad) and /255 normalise.
//
// Not part of /root/reference (it lives in Ultralytics 8.3.x, which the reference's
// train_*_augmented.py scripts call through model.train(...)); the resize arithmetic is the same
// 8-bit fixed-point INTER_LINEAR of SURVEY 8a/a5, the rest is pad(114) + channel swap +
// half(float(u8) / 255.f).  In letterbox_kernel one thread produces one output pixel and writes
// it as three scalar halves, one per colour plane.
#include <cuda_fp16.h>

#include "rod_internal.h"

namespace rod {

struct LbParams {
    const DevImage* images;
    const DevLetterbox* lb;
    const uint32_t* tab;
    const Tile* tiles;
    int n_tiles;
    const uint8_t* img;   // corrupted images, laid out by the plan's dst descriptors
    const uint8_t* src;   // original images (src descriptors): read directly when opcodes[i] == ROD_OP_NONE
    const uint8_t* opcodes;
    __half* out;
    int out_h, out_w;
    int pad;
};

constexpr int kLbRowsPerThread = kLbTH / 4;  // 256 threads = 64 columns x 4 row groups

// Six consecutive bytes (two BGR pixels) starting at an arbitrary address, as byte0..3 / byte4..5 of (lo, hi).
// Aligned 32-bit loads; a word is read only if at least one of its bytes lies below `safe_end` (the end of the
// image), so the over-read is at most 3 bytes inside an aligned word that is partly valid (never a new page).
__device__ __forceinline__ void load6(const uint8_t* p, const uint8_t* safe_end, uint32_t& lo, uint32_t& hi) {
    const uint8_t* a = reinterpret_cast<const uint8_t*>(reinterpret_cast<uintptr_t>(p) & ~(uintptr_t)3);
    const int sh = (int)(reinterpret_cast<uintptr_t>(p) & 3) * 8;
    const uint32_t w0 = __ldg(reinterpret_cast<const uint32_t*>(a));
    const uint32_t w1 = (a + 4 < safe_end) ? __ldg(reinterpret_cast<const uint32_t*>(a + 4)) : 0u;
    const uint32_t w2 = (sh != 0 && a + 8 < safe_end) ? __ldg(reinterpret_cast<const uint32_t*>(a + 8)) : 0u;
    lo = __funnelshift_r(w0, w1, sh);
    hi = __funnelshift_r(w1, w2, sh);
}

__global__ void __launch_bounds__(256) letterbox_kernel(LbParams p) {
    __shared__ __half lut[256];  // half(float(v) / 255.f): the normalisation of preprocess_batch, one division per value
    lut[threadIdx.x] = __float2half_rn(__fdiv_rn((float)threadIdx.x, 255.0f));
    __syncthreads();
    const size_t plane = (size_t)p.out_h * p.out_w;
    const int cx_l = threadIdx.x & (kLbTW - 1), rgrp = threadIdx.x / kLbTW;
    const __half padh = lut[p.pad];
    for (int ti = blockIdx.x; ti < p.n_tiles; ti += gridDim.x) {
        const Tile t = p.tiles[ti];
        const DevImage im = p.images[t.img];
        const DevLetterbox g = p.lb[im.shape_id];
        const bool from_src = (p.opcodes != nullptr && p.opcodes[t.img] == ROD_OP_NONE);
        const uint8_t* base = from_src ? p.src + im.src_off : p.img + im.dst_off;
        const int64_t pitch = from_src ? im.src_pitch : im.dst_pitch;
        const uint8_t* safe_end = base + (int64_t)(g.h - 1) * pitch + 3 * g.w;
        __half* o = p.out + (size_t)t.img * 3 * plane;
        const int X = t.b + cx_l;
        if (X >= p.out_w) continue;
        const int cx = X - g.left;
        const bool col_in = cx >= 0 && cx < g.new_w;
        int s0 = 0;
        uint32_t a = 0;
        bool one_tap = false;
        if (col_in && !g.identity && !g.area2) {
            s0 = reinterpret_cast<const int32_t*>(p.tab + g.lx_s0)[cx];
            a = p.tab[g.lx_a + cx];
            one_tap = (s0 + 1 > g.w - 1);  // right border: both taps are the last pixel
        }
        const int Ya = t.a + rgrp * kLbRowsPerThread;
#pragma unroll 2
        for (int rr = 0; rr < kLbRowsPerThread; ++rr) {
            const int Y = Ya + rr;
            if (Y >= p.out_h) break;
            const int cy = Y - g.top;
            uint32_t v[3];
            bool content = col_in && cy >= 0 && cy < g.new_h;
            if (content) {
                if (g.identity) {
                    const uint8_t* sp = base + (int64_t)cy * pitch + cx * 3;
                    v[0] = sp[0]; v[1] = sp[1]; v[2] = sp[2];
                } else if (g.area2) {
                    const uint8_t* sp = base + (int64_t)(2 * cy) * pitch + (2 * cx) * 3;
#pragma unroll
                    for (int c = 0; c < 3; ++c) v[c] = ((uint32_t)sp[c] + sp[3 + c] + sp[pitch + c] + sp[pitch + 3 + c] + 2u) >> 2;
                } else {
                    const uint32_t ys = p.tab[g.ly_s + cy], yb = p.tab[g.ly_b + cy];
                    const uint8_t* r0 = base + (int64_t)(ys & 0xFFFFu) * pitch + 3 * s0;
                    const uint8_t* r1 = base + (int64_t)(ys >> 16) * pitch + 3 * s0;
                    uint32_t lo0, hi0, lo1, hi1;
                    load6(r0, safe_end, lo0, hi0);
                    load6(r1, safe_end, lo1, hi1);
                    if (one_tap) {  // pixel 1 := pixel 0
                        hi0 = __byte_perm(lo0, 0u, 0x4421); lo0 = __byte_perm(lo0, 0u, 0x0210);
                        hi1 = __byte_perm(lo1, 0u, 0x4421); lo1 = __byte_perm(lo1, 0u, 0x0210);
                    }
                    // channel c: taps are bytes c and c + 3 of the six
                    const uint32_t g0[3] = {__byte_perm(lo0, hi0, 0x4430), __byte_perm(lo0, hi0, 0x4441), __byte_perm(lo0, hi0, 0x4452)};
                    const uint32_t g1[3] = {__byte_perm(lo1, hi1, 0x4430), __byte_perm(lo1, hi1, 0x4441), __byte_perm(lo1, hi1, 0x4452)};
#pragma unroll
                    for (int c = 0; c < 3; ++c) {
                        const uint32_t h0 = dot2_lo(a, g0[c], 0u) >> 4;
                        const uint32_t h1 = dot2_lo(a, g1[c], 0u) >> 4;
                        v[c] = linear_v(h0, h1, yb);
                    }
                }
            }
            __half* dstp = o + (size_t)Y * p.out_w + X;
            // BGR -> RGB: source channel c lands in plane 2 - c
            dstp[2 * plane] = content ? lut[v[0]] : padh;
            dstp[plane] = content ? lut[v[1]] : padh;
            dstp[0] = content ? lut[v[2]] : padh;
        }
    }
}

// =====================================================================================
// Fused training path: corruption + letterbox + normalise in ONE pass over the source (BASELINE config 5).
// A warp owns one output row.  It produces the (at most two) full-resolution CORRUPTED source rows that row blends
// into its private shared-memory buffers -- clean rows are copied, noise rows get the Philox (or supplied) field,
// blur rows are filtered from a staged raw row with reflected halo (same arithmetic as noise.cu / blur.cu) -- and
// then resamples them.  With a down-scaling letterbox every source row is produced exactly once, so the corrupted
// full-resolution image never exists in HBM.  Images whose op is LowRes are the exception: the resize kernels
// write them to the scratch first and this kernel reads them from there like clean rows.
// =====================================================================================
struct FusedLbParams {
    const DevImage* images;
    const DevLetterbox* lb;
    const uint32_t* tab;
    int n_images;
    const uint8_t* src;      // original images (src descriptors)
    const uint8_t* scratch;  // LowRes-corrupted images (dst descriptors)
    const uint8_t* opcodes;
    const float* noise;      // supplied field (compat mode) or NULL (Philox)
    __half* out;
    int out_h, out_w, pad;
    float K;                 // sigma * sqrt(2 ln 2)
    uint32_t key0, key1, offset;
    PhiloxKeys keys;  // the ten round keys of (key0, key1): constant-bank / uniform operands, no per-round key additions
    uint64_t first_image;
    int k;                   // blur taps (odd)
    const DevShape* shapes;  // lowres tables (plan->d_shapes / d_tab), used when lowres_in_kernel
    const uint32_t* ltab;
    int lowres_in_kernel;    // 1: LowRes rows are produced in shared memory too (every LowRes-able shape is exact-2x)
    int buf_bytes;           // bytes of one row buffer (16-byte multiple)
};

constexpr int kFusedLeft = 64;  // bytes in front of pixel 0 in every row buffer (halo of up to 15 pixels + window)

__device__ __forceinline__ void fused_cp_async16(uint32_t smem_addr, const void* g) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(smem_addr), "l"(g) : "memory");
}

// start copying source row `srow` (n bytes) to row[0 .. n): 16-byte cp.async when the row is 16-byte aligned (whole
// chunks; the last one may read up to 15 bytes past the row, inside the same 16-byte granule of the allocation),
// plain 32-bit / byte loads otherwise.  Completion: cp.async.wait_group + __syncwarp by the caller.
__device__ __forceinline__ void fused_stage_row(const uint8_t* srow, int n, uint8_t* row, int lane) {
    if ((((uintptr_t)srow) & 15) == 0) {
        const uint32_t d = (uint32_t)__cvta_generic_to_shared(row);
        for (int j = lane; j < ((n + 15) >> 4); j += 32) fused_cp_async16(d + 16 * j, srow + 16 * j);
    } else if (((((uintptr_t)srow) | (uintptr_t)n) & 3) == 0) {
        for (int i = lane; i < (n >> 2); i += 32) reinterpret_cast<uint32_t*>(row)[i] = __ldg(reinterpret_cast<const uint32_t*>(srow) + i);
    } else {
        for (int i = lane; i < n; i += 32) row[i] = srow[i];
    }
}

// in place: row := noise(row) for image row y (flat element index e0 = y * n of its first byte)
__device__ __forceinline__ void fused_noise_row(const FusedLbParams& p, const DevImage& im, int img_index, int y, uint8_t* row,
                                                int lane) {
    const int n = 3 * im.w;
    const uint32_t e0 = (uint32_t)y * (uint32_t)n;
    if (p.noise != nullptr) {
        const float* nz = p.noise + im.elem_base + e0;
        for (int i = lane; i < n; i += 32) row[i] = (uint8_t)noise_px(__uint_as_float(0x4B000000u | row[i]) - 8388608.0f, nz[i]);
        return;
    }
    const uint64_t ig = p.first_image + (uint64_t)img_index;
    const uint32_t g_first = e0 >> 3, g_last = (e0 + (uint32_t)n - 1u) >> 3;
    const bool words = ((e0 | (uint32_t)n) & 7u) == 0;  // the row is made of whole Philox groups (row buffers are 16-byte aligned)
#pragma unroll 2
    for (uint32_t g = g_first + lane; g <= g_last; g += 32) {
        uint32_t r[4];
        float sf[8];
        philox4x32_10_rk(g, (uint32_t)ig, (uint32_t)(ig >> 32), p.offset, p.keys, r);
        if (philox_needs_tail(r)) {
            uint32_t t[4];
            philox4x32_10(g, (uint32_t)ig, (uint32_t)(ig >> 32) ^ ROD_PHILOX_TAIL_FLIP, p.offset, p.key0, p.key1, t);
            gauss8(r, t, sf);
        } else {
            gauss8(r, nullptr, sf);
        }
        if (words) {
            uint2* q = reinterpret_cast<uint2*>(row + (int)(8u * g - e0));
            const uint2 v = *q;
            *q = make_uint2(philox_word(v.x, sf, p.K), philox_word(v.y, sf + 4, p.K));
            continue;
        }
#pragma unroll
        for (int q = 0; q < 8; ++q) {
            const int x = (int)(8u * g + q - e0);
            if (x >= 0 && x < n) row[x] = (uint8_t)noise_philox_px(row[x], sf[q], p.K);
        }
    }
}

// dst[0 .. n) := blur(row) where row (with kFusedLeft bytes of room in front and 64 behind) holds the raw image row
__device__ __forceinline__ void fused_blur_row(const FusedLbParams& p, const DevImage& im, uint8_t* row, uint8_t* dst, int lane) {
    const int n = 3 * im.w, halo = 3 * (p.k >> 1);
    for (int q = lane; q < 2 * halo; q += 32) {
        const int i = (q < halo) ? (q - halo) : (n + q - halo);
        const int px = (i >= 0) ? i / 3 : -((-i + 2) / 3);
        const int c = i - 3 * px;
        row[i] = row[3 * reflect101(px, im.w) + c];
    }
    __syncwarp();
    if (p.k == 9) {
        for (int j = lane; j < ((n + 15) >> 4); j += 32) {
            const uint4* wp = reinterpret_cast<const uint4*>(row + 16 * j - 16);
            const uint4 a = wp[0], b = wp[1], c = wp[2];
            const uint32_t w[12] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w, c.x, c.y, c.z, c.w};
            uint32_t o[4];
            blur9_chunk16(w, o);
            *reinterpret_cast<uint4*>(dst + 16 * j) = make_uint4(o[0], o[1], o[2], o[3]);  // the tail beyond n is padding
        }
    } else {
        for (int i = lane; i < n; i += 32) dst[i] = (uint8_t)blur_byte_generic(row, i, p.k);
    }
}

// ---- LowRes rows in shared memory (exact-2x shapes, w % 4 == 0): same arithmetic as lowres.cu ----
// low-res row j of the image -> prow (layout of the strip kernel: [1..3] = pixel 0 replicated, [4 + 3i + c], pixel nw-1 replicated)
__device__ __forceinline__ void fused_lowres_prow(const DevImage& im, const DevShape& sh, const uint32_t* ltab,
                                                  const uint8_t* simg, int j, uint8_t* prow, int lane) {
    const int nw = sh.nw, n_units = nw >> 1;
    const bool fast2 = (sh.area_mode == AREA_FAST2);
    int sy0 = 2 * j;
    float b0 = 0.f, b1 = 0.f, b2 = 0.f;
    if (!fast2) {
        const uint4 pk = reinterpret_cast<const uint4*>(ltab + sh.ay_pack)[j];
        sy0 = (int)pk.x; b0 = __uint_as_float(pk.y); b1 = __uint_as_float(pk.z); b2 = __uint_as_float(pk.w);
    }
    const uint8_t* r0 = simg + (int64_t)sy0 * im.src_pitch;
    const uint8_t* r1 = r0 + im.src_pitch;
    const uint8_t* r2 = simg + (int64_t)min(sy0 + 2, im.h - 1) * im.src_pitch;
    for (int u = lane; u < n_units; u += 32) {
        const uint32_t* w0 = reinterpret_cast<const uint32_t*>(r0 + 12 * u);
        const uint32_t* w1 = reinterpret_cast<const uint32_t*>(r1 + 12 * u);
        const uint32_t ra[3] = {__ldg(w0), __ldg(w0 + 1), __ldg(w0 + 2)}, rb[3] = {__ldg(w1), __ldg(w1 + 1), __ldg(w1 + 2)};
        uint32_t o6[6];
        if (fast2) {
            area_fast2_unit(ra, rb, o6);
        } else {
            const uint32_t* w2 = reinterpret_cast<const uint32_t*>(r2 + 12 * u);
            const uint32_t rc[3] = {__ldg(w2), __ldg(w2 + 1), __ldg(w2 + 2)};
            float acc[6];
            area_x2f_accumulate(ra, b0, true, acc);
            area_x2f_accumulate(rb, b1, false, acc);
            area_x2f_accumulate(rc, b2, false, acc);
            area_x2f_finish(acc, o6);
        }
        uint16_t* o16 = reinterpret_cast<uint16_t*>(prow + 4 + 6 * u);
        o16[0] = (uint16_t)__byte_perm(o6[0], o6[1], 0x0040);
        o16[1] = (uint16_t)__byte_perm(o6[2], o6[3], 0x0040);
        o16[2] = (uint16_t)__byte_perm(o6[4], o6[5], 0x0040);
        if (u == 0) { prow[1] = (uint8_t)o6[0]; prow[2] = (uint8_t)o6[1]; prow[3] = (uint8_t)o6[2]; }
        if (u == n_units - 1) {
            uint8_t* e = prow + 4 + 3 * nw;
            e[0] = (uint8_t)o6[3]; e[1] = (uint8_t)o6[4]; e[2] = (uint8_t)o6[5];
        }
    }
}

// full-resolution row y of lowres(image) from the two resident low-res rows -> dst[0 .. 3w)
__device__ __forceinline__ void fused_lowres_fullrow(const DevImage& im, const DevShape& sh, const uint32_t* ltab, int y,
                                                     const uint8_t* pslots, int p_pitch, uint8_t* dst, int lane) {
    const uint32_t ys = ltab[sh.ly_s + y];
    const int s0 = (int)(ys & 0xFFFFu), s1 = (int)(ys >> 16);
    const float4 rf = reinterpret_cast<const float4*>(ltab + sh.ly_rc)[y];
    X2Row rc;
    rc.c0s = rf.x; rc.c1s = rf.y; rc.k0 = rf.z; rc.k2 = rf.w;
    const uint8_t* p0 = pslots + (s0 & 1) * p_pitch;
    const uint8_t* p1 = pslots + (s1 & 1) * p_pitch;
    const int n = 3 * im.w, nchunks = (im.w + 7) >> 3;
    for (int ch = lane; ch < nchunks; ch += 32) {
        float x0[24], x1[24];
#pragma unroll
        for (int q = 0; q < 2; ++q) {
            const uint32_t* w = reinterpret_cast<const uint32_t*>(q ? p1 : p0) + 3 * ch;
            const uint32_t w0 = w[0], w1 = w[1], w2 = w[2], w3 = w[3], w4 = w[4], w5 = w[5];
            const uint32_t win[5] = {funnel_r(w0, w1, 8), funnel_r(w1, w2, 8), funnel_r(w2, w3, 8), funnel_r(w3, w4, 8),
                                     funnel_r(w4, w5, 8)};
            x2_expand24(win, q ? x1 : x0);
        }
        uint32_t o[24];
#pragma unroll
        for (int t = 0; t < 24; ++t) o[t] = x2_vertical(x0[t], x1[t], rc);
        uint32_t wds[6];
#pragma unroll
        for (int g = 0; g < 6; ++g) {
            const uint32_t lo = __byte_perm(o[4 * g], o[4 * g + 1], 0x0040);
            const uint32_t hi = __byte_perm(o[4 * g + 2], o[4 * g + 3], 0x0040);
            wds[g] = __byte_perm(lo, hi, 0x5410);
        }
        const int nvalid = min(24, n - 24 * ch);
        uint2* d8 = reinterpret_cast<uint2*>(dst + 24 * ch);
        if (nvalid == 24) {
            d8[0] = make_uint2(wds[0], wds[1]); d8[1] = make_uint2(wds[2], wds[3]); d8[2] = make_uint2(wds[4], wds[5]);
        } else {
            for (int b = 0; b < nvalid; ++b) dst[24 * ch + b] = (uint8_t)(wds[b >> 2] >> (8 * (b & 3)));
        }
    }
}

// six consecutive bytes of a shared-memory row buffer starting at byte offset `o` (buffers are padded: no bound check)
__device__ __forceinline__ void load6_smem(const uint8_t* buf, int o, uint32_t& lo, uint32_t& hi) {
    const uint32_t* a = reinterpret_cast<const uint32_t*>(buf + (o & ~3));
    const int sh = (o & 3) * 8;
    const uint32_t w0 = a[0], w1 = a[1], w2 = a[2];
    lo = __funnelshift_r(w0, w1, sh);
    hi = __funnelshift_r(w1, w2, sh);
}

// =====================================================================================
// The fused kernel.  It needs an even out_w (rod_corrupt_letterbox_f16 sends odd widths to the unfused path):
//   * every WARP works on single output rows on its own (no block barrier).  Rows are ordered by op class (noise, LowRes,
//     blur, clean), centre-out and image-minor, and dealt round-robin to the resident warps: the expensive rows of all
//     images run first, spread evenly, and the cheap padding rows fill the tail;
//   * the resampling loop makes two adjacent output columns per lane and step: x taps from a per-shape table in global
//     memory (one 16-byte load through L1), the horizontal stage as dp2a onto the 2^23 float grid, the vertical stage as the
//     three round-toward-zero FMAs of the resize kernels, half(v / 255) as one more FMA and a packed half2 conversion;
//     three 4-byte stores per step (~50 instructions per output column);
//   * padding rows leave as 16-byte stores.
// half(fl(v * fl(1/255))) must equal the 256-entry half(float(v) / 255.f) table of letterbox_kernel for every byte value
// v (it does, checked exhaustively): the unfused fallback has to produce the same bytes.
// =====================================================================================
__device__ __forceinline__ void fused_column(const uint8_t* bufA, const uint8_t* rowB, uint32_t o3, uint32_t a, const X2Row& rc,
                                             float c255, float nc255, float out[3]) {
    uint32_t lo0, hi0, lo1, hi1;
    load6_smem(bufA, (int)o3, lo0, hi0);
    load6_smem(rowB, (int)o3, lo1, hi1);
    // at the right border both taps are the last pixel: OpenCV's coefficients there are (2048, 0), so whatever the second
    // tap reads (row padding) is multiplied by zero
    const uint32_t g0[3] = {__byte_perm(lo0, hi0, 0x4430), __byte_perm(lo0, hi0, 0x4441), __byte_perm(lo0, hi0, 0x4452)};
    const uint32_t g1[3] = {__byte_perm(lo1, hi1, 0x4430), __byte_perm(lo1, hi1, 0x4441), __byte_perm(lo1, hi1, 0x4452)};
#pragma unroll
    for (int c = 0; c < 3; ++c) {
        // 2^23 + H (H = tap0 * a0 + tap1 * a1 < 2^23) -> 2^23 + (H >> 4): one multiply-add rounded toward zero
        const float x0 = __fmaf_rz(__uint_as_float(dot2_lo(a, g0[c], 0x4B000000u)), 0.0625f, 7864320.0f);
        const float x1 = __fmaf_rz(__uint_as_float(dot2_lo(a, g1[c], 0x4B000000u)), 0.0625f, 7864320.0f);
        const float y = __uint_as_float(x2_vertical(x0, x1, rc));   // 2^23 + v
        out[c] = __fmaf_rn(y, c255, nc255);                          // fl(v * fl(1 / 255)); its half is half(float(v) / 255.f)
    }
}

constexpr int kFusedMaxSorted = 256;   // batches up to this size are walked most-expensive-op first

template <int NW>
__global__ void __launch_bounds__(32 * NW, 16 / NW) fused_letterbox2_kernel(FusedLbParams p) {
    extern __shared__ __align__(16) uint8_t smem[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    // image order: by op class, the most expensive rows first (noise, LowRes, blur, clean), so that the cheap rows fill
    // the tail of the launch; every CTA derives the same permutation from the op-codes
    uint16_t* perm = reinterpret_cast<uint16_t*>(smem);   // [kFusedMaxSorted] + class starts
    int* cls = reinterpret_cast<int*>(smem + 2 * kFusedMaxSorted);   // cls[c] = first sorted position of class c, cls[4] = n
    const bool sorted = p.n_images <= kFusedMaxSorted;
    if (sorted) {
        auto rank_of = [](int op) { return op == ROD_OP_NOISE ? 0 : op == ROD_OP_LOWRES ? 1 : op == ROD_OP_BLUR ? 2 : 3; };
        for (int i = threadIdx.x; i < p.n_images; i += 32 * NW) {
            const int r = rank_of(p.opcodes[i]);
            int pos = 0;
            for (int j = 0; j < p.n_images; ++j) {
                const int rj = rank_of(p.opcodes[j]);
                pos += (rj < r || (rj == r && j < i)) ? 1 : 0;
            }
            perm[pos] = (uint16_t)i;
        }
        if (threadIdx.x < 5) {
            int c = 0;
            for (int j = 0; j < p.n_images; ++j) c += rank_of(p.opcodes[j]) < (int)threadIdx.x ? 1 : 0;
            cls[threadIdx.x] = c;
        }
    }
    __syncthreads();
    const size_t buf0 = 2 * kFusedMaxSorted + 32;
    uint8_t* X0 = smem + buf0 + (size_t)warp * (3 * p.buf_bytes) + kFusedLeft;   // three identical row buffers per warp: [kFusedLeft | row | 64]
    uint8_t* X1 = X0 + p.buf_bytes;
    uint8_t* X2 = X1 + p.buf_bytes;
    const size_t plane = (size_t)p.out_h * p.out_w;
    const float c255 = __fdiv_rn(1.0f, 255.0f), nc255 = -8388608.0f * c255;
    const float padf = __fmul_rn((float)p.pad, c255);
    const __half2 pad2 = __floats2half2_rn(padf, padf);
    const int total = p.n_images * p.out_h, mid = p.out_h >> 1;
    const int half_w = p.out_w >> 1;
    // rows are dealt round-robin to the resident warps, in the cost-sorted order above: consecutive indices cost about the
    // same, so every warp gets the same mix.  (A dynamic counter does not pay here: ptxas turns a single-lane atomicAdd
    // into its warp-aggregated form, whose broadcast shuffle waits for the atomic on the spot -- 0.45 us per row.)
    const int stride = (int)gridDim.x * NW;
    for (int ti = (int)blockIdx.x * NW + warp; ti < total; ti += stride) {
        // row order inside a class block: centre-out (mid, mid-1, mid+1, ...: a bijection onto [0, out_h)), image-minor
        int img, kk;
        if (sorted) {
            const int c1 = cls[1] * p.out_h, c2 = cls[2] * p.out_h, c3 = cls[3] * p.out_h;
            const int c = (ti >= c1) + (ti >= c2) + (ti >= c3);
            const int first = cls[c], cnt = cls[c + 1] - first;
            const int local = ti - first * p.out_h;
            kk = local / cnt;
            img = perm[first + (local - kk * cnt)];
        } else {
            kk = ti / p.n_images;
            img = ti - kk * p.n_images;
        }
        const int d = (kk + 1) >> 1;
        const int Y = (kk & 1) ? mid - d : mid + d;
        const DevImage im = p.images[img];
        const DevLetterbox g = p.lb[im.shape_id];
        __half* orow = p.out + (size_t)img * 3 * plane + (size_t)Y * p.out_w;
        const int cy = Y - g.top;
        if (cy < 0 || cy >= g.new_h) {
            if ((p.out_w & 7) == 0 && (((uintptr_t)p.out) & 15) == 0) {
                const uint32_t pw = *reinterpret_cast<const uint32_t*>(&pad2);
                const uint4 v = make_uint4(pw, pw, pw, pw);
                for (int q = lane; q < (p.out_w >> 3); q += 32) {
                    reinterpret_cast<uint4*>(orow)[q] = v;
                    reinterpret_cast<uint4*>(orow + plane)[q] = v;
                    reinterpret_cast<uint4*>(orow + 2 * plane)[q] = v;
                }
            } else {
                for (int q = lane; q < half_w; q += 32) {
                    reinterpret_cast<__half2*>(orow)[q] = pad2;
                    reinterpret_cast<__half2*>(orow + plane)[q] = pad2;
                    reinterpret_cast<__half2*>(orow + 2 * plane)[q] = pad2;
                }
            }
            continue;
        }
        const int op = p.opcodes[img];
        const bool lowres_here = (op == ROD_OP_LOWRES) && p.lowres_in_kernel != 0 && p.shapes[im.shape_id].lin_identity == 0;
        const bool pre = (op == ROD_OP_LOWRES) && p.lowres_in_kernel == 0;
        const uint8_t* base = pre ? p.scratch + im.dst_off : p.src + im.src_off;
        const int64_t pitch = pre ? im.dst_pitch : im.src_pitch;
        const uint32_t ys = p.tab[g.ly_s + cy], yb = p.tab[g.ly_b + cy];
        const int r0 = (int)(ys & 0xFFFFu), r1 = (int)(ys >> 16);
        const int n = 3 * im.w;
        const bool two = (r1 != r0);
        const bool blur = (op == ROD_OP_BLUR);
        const uint4* xt = reinterpret_cast<const uint4*>(p.tab + g.lx_pack);
        // step order of this lane: groups of lane_group lanes start one step apart (their windows would otherwise fall into
        // the same shared-memory bank, see plan.cu); every lane still visits all steps
        const int n_it = (half_w + 31) >> 5;
        int itt = (g.lane_group > 0 ? lane / g.lane_group : 0) % n_it;
        uint4 e = __ldg(xt + min(lane + 32 * itt, half_w - 1));   // x taps of this lane's first column pair: needed after the row producers
        __syncwarp();  // the previous row's reads of the buffers are done
        if (lowres_here) {
            const DevShape sh = p.shapes[im.shape_id];
            const int p_pitch = (3 * sh.nw + 24 + 15) & ~15;
            const uint32_t ya = p.ltab[sh.ly_s + r0];
            const int a0 = (int)(ya & 0xFFFFu), a1 = (int)(ya >> 16);
            fused_lowres_prow(im, sh, p.ltab, base, a0, X2 + (a0 & 1) * p_pitch, lane);
            if (a1 != a0) fused_lowres_prow(im, sh, p.ltab, base, a1, X2 + (a1 & 1) * p_pitch, lane);
            __syncwarp();
            fused_lowres_fullrow(im, sh, p.ltab, r0, X2, p_pitch, X0, lane);
            __syncwarp();
            if (two) {
                const uint32_t yb2 = p.ltab[sh.ly_s + r1];
                const int b0 = (int)(yb2 & 0xFFFFu), b1 = (int)(yb2 >> 16);
                if (b0 != a0 && b0 != a1) fused_lowres_prow(im, sh, p.ltab, base, b0, X2 + (b0 & 1) * p_pitch, lane);
                if (b1 != a0 && b1 != a1 && b1 != b0) fused_lowres_prow(im, sh, p.ltab, base, b1, X2 + (b1 & 1) * p_pitch, lane);
                __syncwarp();
                fused_lowres_fullrow(im, sh, p.ltab, r1, X2, p_pitch, X1, lane);
            }
        } else {
            fused_stage_row(base + (int64_t)r0 * pitch, n, blur ? X1 : X0, lane);
            if (two) fused_stage_row(base + (int64_t)r1 * pitch, n, blur ? X2 : X1, lane);
            asm volatile("cp.async.commit_group;\ncp.async.wait_group 0;" ::: "memory");
            __syncwarp();
            if (op == ROD_OP_NOISE) {
                fused_noise_row(p, im, img, r0, X0, lane);
                if (two) fused_noise_row(p, im, img, r1, X1, lane);
            } else if (blur) {
                fused_blur_row(p, im, X1, X0, lane);
                __syncwarp();
                if (two) fused_blur_row(p, im, X2, X1, lane);
            }
        }
        const uint8_t* bufA = X0;
        const uint8_t* rowB = two ? X1 : X0;
        const X2Row rc = x2g_row_consts(yb);
        __half2* o0 = reinterpret_cast<__half2*>(orow);
        __half2* o1 = reinterpret_cast<__half2*>(orow + plane);
        __half2* o2 = reinterpret_cast<__half2*>(orow + 2 * plane);
        __syncwarp();
#pragma unroll 1
        for (int it = 0; it < n_it; ++it) {
            const int q = lane + 32 * itt;
            itt = (itt + 1 == n_it) ? 0 : itt + 1;
            const uint4 en = __ldg(xt + min(lane + 32 * itt, half_w - 1));   // next step's x taps, in flight during this step
            if (q < half_w) {
                float fa[3] = {padf, padf, padf}, fb[3] = {padf, padf, padf};
                if (e.x != 0xFFFFFFFFu) fused_column(bufA, rowB, e.x, e.y, rc, c255, nc255, fa);
                if (e.z != 0xFFFFFFFFu) fused_column(bufA, rowB, e.z, e.w, rc, c255, nc255, fb);
                o0[q] = __floats2half2_rn(fa[2], fb[2]);   // BGR -> RGB planes
                o1[q] = __floats2half2_rn(fa[1], fb[1]);
                o2[q] = __floats2half2_rn(fa[0], fb[0]);
            }
            e = en;
        }
    }
}

// 4 warps per CTA: smaller CTAs balance the expensive noise / blur / LowRes rows (measured 6 % faster than 8 at batch 64,
// equal at batch 16).  Measured on a B200 (1360x765 sources, seed-42 mix): batch 64 152 us, batch 16 43.5 us.
// (Tried and dropped: keeping the NEXT row's source rows in flight during the resampling loop -- four row buffers per
// warp, 12 warps per SM: 171 us at batch 64.  The loop is bound by its shared-memory reads, not by the source-row
// latency: at scale 2.125 the six-byte windows of every fifth column pair fall into the same bank.)
constexpr int kFusedWarps = 4;

// bytes of one row buffer: also holds two low-res rows (3 * max_w / 2 + 39 each)
static int fused_buf_bytes(const rod_plan* plan) { return kFusedLeft + ((3 * plan->max_w + 15) & ~15) + 128; }

size_t fused_letterbox_smem(const rod_plan* plan) {
    return (size_t)(2 * kFusedMaxSorted + 32) + (size_t)kFusedWarps * (size_t)(3 * fused_buf_bytes(plan));
}

int launch_fused_letterbox(const rod_plan* plan, const uint8_t* src, const uint8_t* scratch, const uint8_t* opcodes,
                           const float* noise, void* out_f16, int pad_value, float sigma, int k, uint64_t seed,
                           uint64_t first_image, uint32_t offset, bool lowres_in_kernel, cudaStream_t stream) {
    FusedLbParams p;
    p.shapes = plan->d_shapes; p.ltab = plan->d_tab; p.lowres_in_kernel = lowres_in_kernel ? 1 : 0;
    p.images = plan->d_images; p.lb = plan->d_lb; p.tab = plan->d_lb_tab; p.n_images = plan->n_images;
    p.src = src; p.scratch = scratch; p.opcodes = opcodes; p.noise = noise;
    p.out = reinterpret_cast<__half*>(out_f16);
    p.out_h = plan->lb_out_h; p.out_w = plan->lb_out_w; p.pad = pad_value;
    p.K = sigma * ROD_NOISE_K_PER_SIGMA;
    p.key0 = (uint32_t)seed; p.key1 = (uint32_t)(seed >> 32); p.offset = offset; p.first_image = first_image;
    p.keys = philox_round_keys(p.key0, p.key1);
    p.k = k;
    p.buf_bytes = fused_buf_bytes(plan);
    constexpr int nw = kFusedWarps;
    const size_t smem = fused_letterbox_smem(plan);
    if (smem > kFusedMaxSmem) return ROD_ERR_UNSUPPORTED;
    int per_sm = (int)((227 * 1024) / (smem + 1024));
    per_sm = per_sm < 1 ? 1 : per_sm;
    // one output row per warp, dealt round-robin (no work counter: one launch, nothing else on the stream)
    const int ctas = (plan->n_images * p.out_h + nw - 1) / nw;
    ROD_CUDA(cudaFuncSetAttribute(fused_letterbox2_kernel<nw>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    fused_letterbox2_kernel<nw><<<grid_for(plan, ctas, per_sm), 32 * nw, smem, stream>>>(p);
    ROD_CUDA(cudaGetLastError());
    return ROD_OK;
}

int launch_letterbox(const rod_plan* plan, const uint8_t* img, const uint8_t* src, const uint8_t* opcodes, void* out_f16,
                     int pad_value, cudaStream_t stream) {
    if (plan->lb_tiles.n == 0) return ROD_OK;
    LbParams p;
    p.images = plan->d_images;
    p.lb = plan->d_lb;
    p.tab = plan->d_lb_tab;
    p.tiles = plan->lb_tiles.d;
    p.n_tiles = plan->lb_tiles.n;
    p.img = img;
    p.src = src;
    p.opcodes = opcodes;
    p.out = reinterpret_cast<__half*>(out_f16);
    p.out_h = plan->lb_out_h;
    p.out_w = plan->lb_out_w;
    p.pad = pad_value;
    const int grid = grid_for(plan, plan->lb_tiles.n, 8);
    letterbox_kernel<<<grid, 256, 0, stream>>>(p);
    ROD_CUDA(cudaGetLastError());
    return ROD_OK;
}

}  // namespace rod
