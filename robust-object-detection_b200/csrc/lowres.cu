// lowres.cu -- a4+a5: fused INTER_AREA downscale + 8-bit INTER_LINEAR upscale (sm_100a).
//
// Reference: scripts/augmentations.py:41-45 (apply_lowres): cv2.resize(img,(nw,nh),INTER_AREA) followed by
// cv2.resize(small,(w,h),INTER_LINEAR).  The low-resolution intermediate never exists in HBM.
//
// Every image goes to one tile list (ensure_lowres_tables in plan.cu); a call launches one kernel per non-empty list
// (launch_lowres_lists below).  Shapes are at factor 0.5 unless noted; "rows aligned to n" means the image's pitch and
// offset are multiples of n.  tests/test_kernel_paths.py asserts this table.
//   kernel                       list          layouts that select it
//   lowres_x2i_kernel<true>      X2I_CARRY     odd w = 2 nw + 1 with three x taps, regular y axis, odd h
//   lowres_x2i_kernel<false>     X2I_EVEN      ... even h
//   lowres_x2g_kernel            X2G           odd w with three x taps, other y axes (no alignment requirement)
//   lowres_x2p_kernel<16|8|4>    X2P16|8|4     exact 2x in both axes, w % 4 == 0; source and destination rows aligned to 4;
//                                              copy unit 16 / 8 / 4: w and every pitch and offset a multiple of it
//   lowres_x2h_kernel<16|8|4>    X2H16|8|4     exact-2x width, w % 4 == 0, odd h whose low-res row j reads source rows
//                                              2j..2j+2 (h up to ~2000); alignment and copy unit as X2P
//   lowres_x2f_kernel<16|8|4>    X2F16|8|4     exact-2x width, w % 4 == 0, other packed y axes (odd h from ~2001); as X2P
//   lowres_x2w_kernel<true>      X2W8          the X2P / X2H / X2F shapes whose source rows are aligned to 8 (w % 8 == 0)
//                                              but whose destination rows are not aligned to 4 (odd pitch, offset 2 mod 4)
//   lowres_x2w_kernel<false>     X2W4          ... source rows aligned to 4 only; and X2W8 when the source base is not
//                                              8-aligned
//   lowres_x2_kernel<128>        X2_REST       other exact-2x widths (w % 4 != 0 or a FASTN y axis), and the X2P / X2H /
//                                              X2F shapes whose source rows are not aligned to 4
//                                X2_STRIP      every exact-2x image, in place of all of the above but X2I / X2G, when the
//                                              source base is not 4-aligned, or the destination base is not 4-aligned
//                                              while an X2P / X2H / X2F list is not empty
//   lowres_kernel                GENERIC       anything else (other factors, widths that are not 2 nw or 2 nw + 1)
// The base pointers may also be less aligned than a staged list's copy unit: the list then runs the kernel of the unit
// that src | dst allows (lowres_x2p_kernel<8> for X2P16 at a base 8 mod 16).
//
// lowres_kernel: tiles of kLowresTH rows x kLowresTWB output BYTES (cut in byte columns: every stage is per byte,
// channel = byte % 3)
//     phase B1/B2: separable INTER_AREA in OpenCV's operation order (resizeArea_ / resizeAreaFast_), horizontal pass
//                  per source row into a float buffer, then the y taps -> low-res tile P (u8, shared)
//     phase C1   : horizontal fixed-point pass  hx = (P[s0]*a0 + P[s1]*a1) >> 4   (u16, shared)
//     phase C2   : vertical pass + pack; each thread owns 8 byte columns and marches down 8 rows
// lowres_x2_kernel: full-width strips, low-res rows in shared memory.  The band kernels (x2w, x2p, x2h, x2f, x2g, x2i):
// a warp owns a band of rows x a strip of 30 chunks of 8 output pixels (see the banner above lowres_x2w_kernel).

#include <algorithm>
#include <mutex>

#include "rod_internal.h"

namespace rod {

struct LowresParams {
    const DevImage* images;
    const Tile* tiles;
    int n_tiles;
    const DevShape* shapes;
    const uint32_t* tab;
    const uint8_t* src;
    uint8_t* dst;
    const uint8_t* opcodes;
    int half_rows;  // allocation (worst case over the plan): low-res rows one tile touches
    int p_pitch;    // bytes per low-res row in shared memory
    int hb_pitch;   // floats per source row of the horizontal INTER_AREA buffer
    int union_bytes;  // size of the hbuf / hx union
};

constexpr int kHxPitch = kLowresTWB + 8;


__device__ __forceinline__ uint32_t ldg32(const void* p) { return __ldg(reinterpret_cast<const uint32_t*>(p)); }
// exact float of a byte: 0x4B0000bb is 2^23 + bb
__device__ __forceinline__ float u8f(uint32_t b) { return __uint_as_float(0x4B000000u | b) - 8388608.0f; }

__device__ __forceinline__ void store_chunk8(uint8_t* p, uint32_t lo, uint32_t hi, int nvalid) {
    // p is the address of the chunk's first byte; alignment depends on the row (warp-uniform)
    if (nvalid == 8) {
        const uintptr_t a = (uintptr_t)p;
        if ((a & 7) == 0) {
            asm volatile("st.global.L1::no_allocate.v2.u32 [%0], {%1,%2};" ::"l"(p), "r"(lo), "r"(hi) : "memory");
        } else if ((a & 3) == 0) {
            reinterpret_cast<uint32_t*>(p)[0] = lo;
            reinterpret_cast<uint32_t*>(p)[1] = hi;
        } else if ((a & 1) == 0) {
            uint16_t* q = reinterpret_cast<uint16_t*>(p);
            q[0] = (uint16_t)lo; q[1] = (uint16_t)(lo >> 16); q[2] = (uint16_t)hi; q[3] = (uint16_t)(hi >> 16);
        } else {
#pragma unroll
            for (int b = 0; b < 4; ++b) { p[b] = (uint8_t)(lo >> (8 * b)); p[4 + b] = (uint8_t)(hi >> (8 * b)); }
        }
    } else {
        for (int b = 0; b < nvalid; ++b) p[b] = (uint8_t)((b < 4 ? lo : hi) >> (8 * (b & 3)));
    }
}

__global__ void __launch_bounds__(256, 3) lowres_kernel(LowresParams p) {
    extern __shared__ __align__(16) uint8_t smem[];
    uint8_t* P = smem;
    uint8_t* un = smem + (((size_t)p.half_rows * p.p_pitch + 15) & ~(size_t)15);
    float* hbuf = reinterpret_cast<float*>(un);       // phase B: horizontal INTER_AREA pass, [source row][low-res byte col]
    uint16_t* hx = reinterpret_cast<uint16_t*>(un);   // phase C: horizontal INTER_LINEAR pass (same bytes, later)
    // per low-res row of the tile: {hbuf row offset of its first tap, tap count, weights[kMaxAreaTaps]}
    uint32_t* ytab = reinterpret_cast<uint32_t*>(un + p.union_bytes);

    for (int ti = blockIdx.x; ti < p.n_tiles; ti += gridDim.x) {
        const Tile t = p.tiles[ti];
        if (p.opcodes != nullptr && p.opcodes[t.img] != ROD_OP_LOWRES) continue;
        const DevImage im = p.images[t.img];
        const DevShape sh = p.shapes[im.shape_id];
        const uint8_t* simg = p.src + im.src_off;
        uint8_t* dimg = p.dst + im.dst_off;
        const int y0 = t.a, b0 = t.b;
        const int n = 3 * im.w;
        const int th = min(kLowresTH, im.h - y0), twb = min(kLowresTWB, n - b0);

        if (sh.lin_identity) {  // factor maps (h, w) onto itself: both resizes are copies
            for (int idx = threadIdx.x; idx < th * twb; idx += 256) {
                const int r = idx / twb, o = idx - r * twb;
                dimg[(int64_t)(y0 + r) * im.dst_pitch + b0 + o] = simg[(int64_t)(y0 + r) * im.src_pitch + b0 + o];
            }
            continue;
        }
        const uint32_t* ly_s = p.tab + sh.ly_s;
        const uint32_t* ly_b = p.tab + sh.ly_b;
        const int32_t* lx_s0 = reinterpret_cast<const int32_t*>(p.tab + sh.lx_s0);
        const uint32_t* lx_a = p.tab + sh.lx_a;
        const int x_first = b0 / 3, x_last = (b0 + twb - 1) / 3;
        const int j_lo = (int)(ly_s[y0] & 0xFFFFu), j_hi = (int)(ly_s[y0 + th - 1] >> 16);
        const int nj = j_hi - j_lo + 1;
        const int i_lo = lx_s0[x_first], i_hi = min(lx_s0[x_last] + 1, sh.nw - 1);  // low-res pixel columns held in P
        const int ncol = 3 * (i_hi - i_lo + 1);
        const bool general = (sh.area_mode == AREA_GENERAL);
        const int32_t* xfirst = reinterpret_cast<const int32_t*>(p.tab + sh.ax_first);
        const int32_t* xcount = reinterpret_cast<const int32_t*>(p.tab + sh.ax_count);
        const float* xalpha = reinterpret_cast<const float*>(p.tab + sh.ax_alpha);
        const int32_t* yfirst = reinterpret_cast<const int32_t*>(p.tab + sh.ay_first);
        const int32_t* ycount = reinterpret_cast<const int32_t*>(p.tab + sh.ay_count);
        const float* yalpha = reinterpret_cast<const float*>(p.tab + sh.ay_alpha);
        // source rows the tile's low-res rows read
        const int sy_lo = general ? yfirst[j_lo] : j_lo * sh.iy;
        const int sy_hi = general ? yfirst[j_hi] + ycount[j_hi] - 1 : j_hi * sh.iy + sh.iy - 1;
        const int nsr = sy_hi - sy_lo + 1;

        if (general) {
            for (int jr = threadIdx.x; jr < nj; jr += 256) {
                uint32_t* e = ytab + jr * (2 + kMaxAreaTaps);
                const int j = j_lo + jr;
                e[0] = (uint32_t)((yfirst[j] - sy_lo) * p.hb_pitch);
                e[1] = (uint32_t)ycount[j];
                for (int q = 0; q < sh.yt; ++q) e[2 + q] = __float_as_uint(yalpha[j * sh.yt + q]);
            }
        }
        // ---- phase B1: horizontal INTER_AREA pass (OpenCV's resizeArea_ / resizeAreaFast_ row buffer), one thread
        //      per low-res byte column walking down the source rows: hbuf[sr][o]
        for (int o = threadIdx.x; o < ncol; o += 256) {
            const int ir = o / 3, cch = o - 3 * ir, dx = i_lo + ir;
            const int sx0 = general ? xfirst[dx] : dx * sh.ix;
            const int nx = general ? xcount[dx] : sh.ix;
            const uint8_t* sp = simg + (int64_t)sy_lo * im.src_pitch + 3 * sx0 + cch;
            float* hb = hbuf + o;
            if (general && nx <= 4) {
                // taps beyond nx carry weight 0 (adding +0 is exact) and re-read the last valid tap
                float al[4];
#pragma unroll
                for (int q = 0; q < 4; ++q) al[q] = (q < nx) ? xalpha[dx * sh.xt + q] : 0.f;
                const int o1 = 3 * min(1, nx - 1), o2 = 3 * min(2, nx - 1), o3 = 3 * min(3, nx - 1);
                for (int sr = 0; sr < nsr; ++sr, sp += im.src_pitch, hb += p.hb_pitch) {
                    // byte -> float through the 2^23 mantissa trick (LOP3 + FADD) instead of I2F on the quarter-rate XU pipe
                    float buf = fmul(u8f(sp[0]), al[0]);
                    buf = fadd(buf, fmul(u8f(sp[o1]), al[1]));
                    buf = fadd(buf, fmul(u8f(sp[o2]), al[2]));
                    buf = fadd(buf, fmul(u8f(sp[o3]), al[3]));
                    *hb = buf;
                }
            } else if (general) {
                const float* al = xalpha + dx * sh.xt;
                for (int sr = 0; sr < nsr; ++sr, sp += im.src_pitch, hb += p.hb_pitch) {
                    float buf = 0.f;
                    for (int q = 0; q < nx; ++q) buf = fadd(buf, fmul((float)sp[3 * q], al[q]));
                    *hb = buf;
                }
            } else {  // integer scale: exact sums
                for (int sr = 0; sr < nsr; ++sr, sp += im.src_pitch, hb += p.hb_pitch) {
                    uint32_t sum = 0;
                    for (int q = 0; q < nx; ++q) sum += sp[3 * q];
                    *hb = (float)sum;
                }
            }
        }
        __syncthreads();
        // ---- phase B2: vertical INTER_AREA pass -> low-res tile P[jr][o] (u8)
        for (int o = threadIdx.x; o < ncol; o += 256) {
            for (int jr = 0; jr < nj; ++jr) {
                const int j = j_lo + jr;
                uint32_t v;
                if (general) {
                    const uint32_t* e = ytab + jr * (2 + kMaxAreaTaps);
                    const int ny = (int)e[1];
                    const float* hp = hbuf + e[0] + o;
                    float sum = fmul(__uint_as_float(e[2]), hp[0]);
                    for (int q = 1; q < ny; ++q) sum = fadd(sum, fmul(__uint_as_float(e[2 + q]), hp[q * p.hb_pitch]));
                    float r = frint(sum);
                    r = r < 0.f ? 0.f : (r > 255.f ? 255.f : r);
                    v = (uint32_t)(int)r;
                } else {
                    const float* hp = hbuf + (j * sh.iy - sy_lo) * p.hb_pitch + o;
                    float sum = 0.f;
                    for (int q = 0; q < sh.iy; ++q) sum += hp[q * p.hb_pitch];  // exact (integers < 2^24)
                    if (sh.area_mode == AREA_FAST2) {
                        v = ((uint32_t)sum + 2u) >> 2;
                    } else {
                        float r = frint(fmul(sum, sh.inv_area));
                        r = r < 0.f ? 0.f : (r > 255.f ? 255.f : r);
                        v = (uint32_t)(int)r;
                    }
                }
                P[jr * p.p_pitch + o] = (uint8_t)v;
            }
        }
        __syncthreads();

        // ---- phase C1: horizontal INTER_LINEAR pass -> hx[jr][ob] (u16), one thread per output byte column
        for (int ob = threadIdx.x; ob < twb; ob += 256) {
            const int o = b0 + ob;
            const int x = o / 3, cch = o - 3 * x;
            const int s0 = lx_s0[x];
            const int s1 = min(s0 + 1, sh.nw - 1);
            const uint32_t a = lx_a[x];
            const uint8_t* pa = P + (s0 - i_lo) * 3 + cch;
            const uint8_t* pb = P + (s1 - i_lo) * 3 + cch;
            uint16_t* hrow = hx + ob;
            for (int jr = 0; jr < nj; ++jr, pa += p.p_pitch, pb += p.p_pitch, hrow += kHxPitch)
                *hrow = (uint16_t)linear_h4(*pa, *pb, a);
        }
        __syncthreads();

        // ---- phase C2: vertical pass; thread = (row group of 8 rows, 8 byte columns)
        {
            const int rg = threadIdx.x >> 6, cc = threadIdx.x & 63;
            const int col = 8 * cc;
            const int nvalid = min(8, twb - col);
            if (nvalid > 0) {
                uint32_t ha[8], hb[8];  // hx rows ja / jb of this thread's 8 columns
                int ja = -1, jb = -1;
                const int r_end = min(th, 8 * rg + 8);
                for (int r = 8 * rg; r < r_end; ++r) {
                    const uint32_t ys = ly_s[y0 + r], yb = ly_b[y0 + r];
                    const int s0 = (int)(ys & 0xFFFFu), s1 = (int)(ys >> 16);
                    if (s0 != ja) {
                        if (s0 == jb) {
#pragma unroll
                            for (int q = 0; q < 8; ++q) ha[q] = hb[q];
                        } else {
                            const uint4 v = *reinterpret_cast<const uint4*>(hx + (s0 - j_lo) * kHxPitch + col);
                            ha[0] = v.x & 0xFFFFu; ha[1] = v.x >> 16; ha[2] = v.y & 0xFFFFu; ha[3] = v.y >> 16;
                            ha[4] = v.z & 0xFFFFu; ha[5] = v.z >> 16; ha[6] = v.w & 0xFFFFu; ha[7] = v.w >> 16;
                        }
                        ja = s0;
                    }
                    if (s1 != jb) {
                        if (s1 == ja) {
#pragma unroll
                            for (int q = 0; q < 8; ++q) hb[q] = ha[q];
                        } else {
                            const uint4 v = *reinterpret_cast<const uint4*>(hx + (s1 - j_lo) * kHxPitch + col);
                            hb[0] = v.x & 0xFFFFu; hb[1] = v.x >> 16; hb[2] = v.y & 0xFFFFu; hb[3] = v.y >> 16;
                            hb[4] = v.z & 0xFFFFu; hb[5] = v.z >> 16; hb[6] = v.w & 0xFFFFu; hb[7] = v.w >> 16;
                        }
                        jb = s1;
                    }
                    const uint32_t c0 = yb & 0xFFFFu, c1 = yb >> 16;
                    uint32_t o8[8];
#pragma unroll
                    for (int q = 0; q < 8; ++q) o8[q] = (((c0 * ha[q]) >> 16) + ((c1 * hb[q]) >> 16) + 2u) >> 2;
                    const uint32_t lo = o8[0] | (o8[1] << 8) | (o8[2] << 16) | (o8[3] << 24);
                    const uint32_t hi = o8[4] | (o8[5] << 8) | (o8[6] << 16) | (o8[7] << 24);
                    store_chunk8(dimg + (int64_t)(y0 + r) * im.dst_pitch + b0 + col, lo, hi, nvalid);
                }
            }
        }
        __syncthreads();  // smem is rewritten by the next tile
    }
}

// =====================================================================================
// Fast kernel for exact-2x widths (w == 2 * nw: every even-width image, e.g. 1360 x 765).
// Work item of a CTA = one full-width strip of `strip_rows` output rows of one image.
//   phase B: low-res rows of the strip -> shared memory P (u8), one thread per 12 source bytes x taps
//            P row layout: [0] unused, [1..3] = pixel 0 replicated, [4 + 3i + c] = pixel i, then pixel nw-1 replicated
//   phase C: item = (8 output rows, 8 output pixels = 24 bytes).  The horizontal stage runs in registers
//            (dp2a on gathered byte pairs -> 24 floats per low-res row, kept in two parity slots while the
//            thread walks down its 8 rows); the vertical stage is four fp32 ops per byte (x2_vertical).
// =====================================================================================
struct LowresX2Params {
    const DevImage* images;
    const Tile* tiles;   // a = first output row of the strip
    int n_tiles;
    const DevShape* shapes;
    const uint32_t* tab;
    const uint8_t* src;
    uint8_t* dst;
    const uint8_t* opcodes;
};

__device__ __forceinline__ void x2_load_row(const uint8_t* prow, int chunk, float x[24]) {
    // window bytes [12*chunk + 1, +20) of the P row: six aligned words, funnel-shifted by one byte
    const uint32_t* w = reinterpret_cast<const uint32_t*>(prow) + 3 * chunk;
    const uint32_t w0 = w[0], w1 = w[1], w2 = w[2], w3 = w[3], w4 = w[4], w5 = w[5];
    const uint32_t win[5] = {funnel_r(w0, w1, 8), funnel_r(w1, w2, 8), funnel_r(w2, w3, 8), funnel_r(w3, w4, 8),
                             funnel_r(w4, w5, 8)};
    x2_expand24(win, x);
}

__device__ __forceinline__ void stg8(void* p, uint32_t lo, uint32_t hi) {
    asm volatile("st.global.L1::no_allocate.v2.u32 [%0], {%1,%2};" ::"l"(p), "r"(lo), "r"(hi) : "memory");
}
// HINT: the caller knows (uniformly) whether every row start is 8-byte aligned (`al8`)
template <bool HINT = false>
__device__ __forceinline__ void x2_emit_row(const float* xlo, const float* xhi, const X2Row& rc, uint8_t* dptr,
                                            int nvalid, bool al8 = false) {
    uint32_t o[24];
#pragma unroll
    for (int t = 0; t < 24; ++t) o[t] = x2_vertical(xlo[t], xhi[t], rc);
    uint32_t wds[6];
#pragma unroll
    for (int g = 0; g < 6; ++g) {
        const uint32_t lo = __byte_perm(o[4 * g], o[4 * g + 1], 0x0040);
        const uint32_t hi = __byte_perm(o[4 * g + 2], o[4 * g + 3], 0x0040);
        wds[g] = __byte_perm(lo, hi, 0x5410);
    }
    if (HINT && al8 && nvalid == 24) {
        stg8(dptr, wds[0], wds[1]);
        stg8(dptr + 8, wds[2], wds[3]);
        stg8(dptr + 16, wds[4], wds[5]);
    } else if (nvalid == 24) {
        store_chunk8(dptr, wds[0], wds[1], 8);
        store_chunk8(dptr + 8, wds[2], wds[3], 8);
        store_chunk8(dptr + 16, wds[4], wds[5], 8);
    } else {
        for (int b = 0; b < nvalid; ++b) dptr[b] = (uint8_t)(wds[b >> 2] >> (8 * (b & 3)));
    }
}

template <int NT>
__global__ void __launch_bounds__(NT, 4) lowres_x2_kernel(LowresX2Params p) {
    extern __shared__ __align__(16) uint8_t smem[];
    for (int ti = blockIdx.x; ti < p.n_tiles; ti += gridDim.x) {
        const Tile t = p.tiles[ti];
        if (p.opcodes != nullptr && p.opcodes[t.img] != ROD_OP_LOWRES) continue;
        const DevImage im = p.images[t.img];
        const DevShape sh = p.shapes[im.shape_id];
        const uint8_t* simg = p.src + im.src_off;
        uint8_t* dimg = p.dst + im.dst_off;
        const int y0 = t.a;
        const int th = min(sh.strip_rows, im.h - y0);
        const int n = 3 * im.w, nw = sh.nw;
        const int p_pitch = (3 * nw + 24 + 15) & ~15;
        const uint32_t* ly_s = p.tab + sh.ly_s;
        const uint32_t* ly_b = p.tab + sh.ly_b;
        const int j_lo = (int)(ly_s[y0] & 0xFFFFu), j_hi = (int)(ly_s[y0 + th - 1] >> 16);
        const int nj = j_hi - j_lo + 1;

        // ---- phase B: two (low-res row, 12-byte unit) items per thread per step, all loads issued first
        const bool vec = (im.w & 3) == 0 && ((((uintptr_t)simg) | (uintptr_t)im.src_pitch) & 3) == 0 &&
                         (sh.area_mode == AREA_FAST2 || (sh.area_mode == AREA_GENERAL && sh.ay_packed));
        if (vec) {
            const int n_units = nw >> 1;
            const uint32_t magic_div = 0xFFFFFFFFu / (uint32_t)n_units + 1u;  // floor(idx / n_units) = umulhi(idx, magic)
            const int total = nj * n_units;
            const bool fast2 = (sh.area_mode == AREA_FAST2);
            const uint4* ypack = reinterpret_cast<const uint4*>(p.tab + sh.ay_pack);
            for (int base = threadIdx.x; base < total; base += 2 * NT) {
                uint32_t rw[2][3][3];
                float beta[2][3];
                int jrs[2], us[2];
#pragma unroll
                for (int it = 0; it < 2; ++it) {
                    const int idx = (base + NT * it < total) ? base + NT * it : base;  // tail: redo item 0, dropped below
                    const int jr = (n_units == 1) ? idx : (int)__umulhi((uint32_t)idx, magic_div);
                    const int u = idx - jr * n_units;
                    const int dy = j_lo + jr;
                    jrs[it] = jr; us[it] = u;
                    int sy0 = 2 * dy;
                    beta[it][0] = beta[it][1] = beta[it][2] = 0.f;
                    if (!fast2) {
                        const uint4 pk = __ldg(ypack + dy);
                        sy0 = (int)pk.x;
                        beta[it][0] = __uint_as_float(pk.y); beta[it][1] = __uint_as_float(pk.z); beta[it][2] = __uint_as_float(pk.w);
                    }
                    const uint8_t* r0 = simg + (int64_t)sy0 * im.src_pitch + 12 * u;
                    const uint8_t* r1 = r0 + im.src_pitch;
                    rw[it][0][0] = ldg32(r0); rw[it][0][1] = ldg32(r0 + 4); rw[it][0][2] = ldg32(r0 + 8);
                    rw[it][1][0] = ldg32(r1); rw[it][1][1] = ldg32(r1 + 4); rw[it][1][2] = ldg32(r1 + 8);
                    if (!fast2) {  // third tap: weight 0 (and a clamped row) when this low-res row has two taps only
                        const uint8_t* r2 = simg + (int64_t)min(sy0 + 2, im.h - 1) * im.src_pitch + 12 * u;
                        rw[it][2][0] = ldg32(r2); rw[it][2][1] = ldg32(r2 + 4); rw[it][2][2] = ldg32(r2 + 8);
                    }
                }
#pragma unroll
                for (int it = 0; it < 2; ++it) {
                    if (it == 1 && base + NT >= total) break;
                    uint32_t o6[6];
                    if (fast2) {
                        area_fast2_unit(rw[it][0], rw[it][1], o6);
                    } else {
                        float acc[6];
                        area_x2f_accumulate(rw[it][0], beta[it][0], true, acc);
                        area_x2f_accumulate(rw[it][1], beta[it][1], false, acc);
                        area_x2f_accumulate(rw[it][2], beta[it][2], false, acc);
                        area_x2f_finish(acc, o6);
                    }
                    uint16_t* o16 = reinterpret_cast<uint16_t*>(smem + jrs[it] * p_pitch + 4 + 6 * us[it]);
                    o16[0] = (uint16_t)__byte_perm(o6[0], o6[1], 0x0040);
                    o16[1] = (uint16_t)__byte_perm(o6[2], o6[3], 0x0040);
                    o16[2] = (uint16_t)__byte_perm(o6[4], o6[5], 0x0040);
                }
            }
        } else {
            const int total = nj * 3 * nw;
            for (int idx = threadIdx.x; idx < total; idx += NT) {
                const int jr = idx / (3 * nw), o = idx - jr * 3 * nw;
                const int i = o / 3, c = o - 3 * i;
                smem[jr * p_pitch + 4 + o] = (uint8_t)area_value(simg, im.src_pitch, sh, p.tab, j_lo + jr, i, c);
            }
        }
        __syncthreads();
        // replicate the border pixels: P[-1] := P[0], P[nw] := P[nw-1] (OpenCV's clamped x taps)
        for (int q = threadIdx.x; q < nj * 6; q += NT) {
            const int jr = q / 6, kk = q - 6 * jr;
            uint8_t* prow = smem + jr * p_pitch;
            if (kk < 3) prow[1 + kk] = prow[4 + kk];
            else prow[4 + 3 * nw + (kk - 3)] = prow[4 + 3 * (nw - 1) + (kk - 3)];
        }
        __syncthreads();

        // ---- phase C
        {
            const int nchunks = (im.w + 7) >> 3;
            const int ngroups = (th + 7) >> 3;
            const uint32_t magic_div = 0xFFFFFFFFu / (uint32_t)nchunks + 1u;
            const int total = ngroups * nchunks;
            for (int idx = threadIdx.x; idx < total; idx += NT) {
                const int rg = (nchunks == 1) ? idx : (int)__umulhi((uint32_t)idx, magic_div);
                const int ch = idx - rg * nchunks;
                const int nvalid = min(24, n - 24 * ch);
                float xe[24], xo[24];  // horizontal stage of the even / odd low-res row currently held
                int je = -1, jo = -1;
                const int r_end = min(th, 8 * rg + 8);
                uint32_t ys = ly_s[y0 + 8 * rg], yb = ly_b[y0 + 8 * rg];
                for (int r = 8 * rg; r < r_end; ++r) {
                    const int s0 = (int)(ys & 0xFFFFu), s1 = (int)(ys >> 16);
                    const X2Row rc = x2_row_consts(yb);
                    if (r + 1 < r_end) { ys = ly_s[y0 + r + 1]; yb = ly_b[y0 + r + 1]; }  // prefetch the next row's table entries
                    // slot (s0 & 1) must hold row s0 and the other slot row s1 (s1 == s0 only on the first / last image rows)
                    const int want_e = (s0 & 1) ? s1 : s0, want_o = (s0 & 1) ? s0 : s1;
                    if (je != want_e) { x2_load_row(smem + (want_e - j_lo) * p_pitch, ch, xe); je = want_e; }
                    if (jo != want_o) { x2_load_row(smem + (want_o - j_lo) * p_pitch, ch, xo); jo = want_o; }
                    uint8_t* dptr = dimg + (int64_t)(y0 + r) * im.dst_pitch + 24 * ch;
                    if (s0 & 1) x2_emit_row(xo, xe, rc, dptr, nvalid);
                    else x2_emit_row(xe, xo, rc, dptr, nvalid);
                }
            }
        }
        __syncthreads();  // P is rewritten by the next strip
    }
}

// =====================================================================================
// Warp-marching kernel for exact-2x widths (w % 4 == 0, 4-byte aligned rows): no shared memory, no block barrier.
// A work item is a column strip of 30 output chunks (8 pixels = 24 bytes each) x a band of output rows of one
// image; one warp owns it and walks down the rows.  Lane l holds chunk 30*strip - 1 + l, so lanes 0 and 31 are
// halo lanes: they compute low-res pixels like everybody else but store nothing.
//   * a low-res row is produced ONCE per lane, in registers: the lane loads its own 24 source bytes of each tap
//     row (coalesced 768 B per warp and row), forms its four low-res pixels (same arithmetic as the strip kernel),
//     and gets the neighbouring low-res pixel on either side by warp shuffle;
//   * the source words of the NEXT low-res row are already in flight while the current one is processed
//     (register prefetch), so global-load latency is off the critical path;
//   * the horizontal 2x stage of each low-res row is expanded once into 24 floats (parity slots xe / xo) and
//     reused by the two or three output rows that blend it; the vertical stage is x2_vertical (3 FFMA.RZ / byte).
// The low-resolution intermediate never leaves the register file.
// =====================================================================================
struct LowresX2wParams {
    const DevImage* images;
    const Tile* tiles;   // a = first output row of the band, b = end row (exclusive), c = column strip
    int n_tiles;
    const DevShape* shapes;
    const uint32_t* tab;
    const uint8_t* src;
    uint8_t* dst;
    const uint8_t* opcodes;
    unsigned int* counter;  // zeroed before the launch: next tile to hand out
};

constexpr int kX2wChunksPerStrip = 30;

__device__ __forceinline__ uint32_t ldg_stream4(const void* p) {
    uint32_t r;
    asm volatile("ld.global.nc.L1::no_allocate.u32 %0, [%1];" : "=r"(r) : "l"(p));
    return r;
}
__device__ __forceinline__ void ldg_stream8(const void* p, uint32_t& a, uint32_t& b) {
    asm volatile("ld.global.nc.L1::no_allocate.v2.u32 {%0,%1}, [%2];" : "=r"(a), "=r"(b) : "l"(p));
}

struct X2wCtx {
    const uint8_t* scol;     // this lane's source column: simg + 24 * chunk
    int64_t pitch;
    const uint4* ypack;      // this warp's shared copy of the packed y table, entry 0 = low-res row j_first
    int j_first;
    int h;
    bool fast2, second_unit;  // second_unit: the chunk has four low-res pixels (else two: last chunk, w % 8 == 4)
    bool first_chunk, last_chunk;
};

// issue the loads of the source words low-res row j needs (3 tap rows x 24 bytes; tap 2 unused for fast2) and of
// its packed y table entry {first source row, beta0, beta1, beta2}
template <bool AL8>
__device__ __forceinline__ void x2w_prefetch(const X2wCtx& c, int j, uint32_t rw[3][6], uint4& pk) {
    int sy0 = 2 * j;
    if (!c.fast2) {
        pk = c.ypack[j - c.j_first];
        sy0 = (int)pk.x;
    }
    const uint8_t* r0 = c.scol + (int64_t)sy0 * c.pitch;
    const uint8_t* r1 = r0 + c.pitch;
    const uint8_t* r2 = c.scol + (int64_t)min(sy0 + 2, c.h - 1) * c.pitch;
    const int o2 = c.second_unit ? 12 : 0;  // a two-pixel chunk re-reads its first unit (the result is discarded)
#pragma unroll
    for (int t = 0; t < 3; ++t) {
        if (t == 2 && c.fast2) break;
        const uint8_t* r = (t == 0) ? r0 : (t == 1) ? r1 : r2;
        // streaming loads that do not allocate in L1: the small per-row tables stay resident there
        if (AL8) {  // rows are 8-byte aligned (and then every chunk has both units: w % 8 == 0)
            ldg_stream8(r, rw[t][0], rw[t][1]);
            ldg_stream8(r + 8, rw[t][2], rw[t][3]);
            ldg_stream8(r + 16, rw[t][4], rw[t][5]);
        } else {
            rw[t][0] = ldg_stream4(r); rw[t][1] = ldg_stream4(r + 4); rw[t][2] = ldg_stream4(r + 8);
            rw[t][3] = ldg_stream4(r + o2); rw[t][4] = ldg_stream4(r + o2 + 4); rw[t][5] = ldg_stream4(r + o2 + 8);
        }
    }
}

// the lane's four low-res pixels of a row (12 bytes in own[3]) from the prefetched words and table entry
__device__ __forceinline__ void x2w_reduce(const X2wCtx& c, const uint4 pk, const uint32_t rw[3][6], uint32_t own[3]) {
    uint32_t o6[2][6];
    if (c.fast2) {
#pragma unroll
        for (int hf = 0; hf < 2; ++hf) area_fast2_unit(&rw[0][3 * hf], &rw[1][3 * hf], o6[hf]);
    } else {
        const float b0 = __uint_as_float(pk.y), b1 = __uint_as_float(pk.z), b2 = __uint_as_float(pk.w);
#pragma unroll
        for (int hf = 0; hf < 2; ++hf) {
            float acc[6];
            area_x2f_accumulate(&rw[0][3 * hf], b0, true, acc);
            area_x2f_accumulate(&rw[1][3 * hf], b1, false, acc);
            area_x2f_accumulate(&rw[2][3 * hf], b2, false, acc);
            area_x2f_finish(acc, o6[hf]);
        }
    }
    const uint32_t a01 = __byte_perm(o6[0][0], o6[0][1], 0x0040), a23 = __byte_perm(o6[0][2], o6[0][3], 0x0040);
    const uint32_t a45 = __byte_perm(o6[0][4], o6[0][5], 0x0040);
    const uint32_t c01 = __byte_perm(o6[1][0], o6[1][1], 0x0040), c23 = __byte_perm(o6[1][2], o6[1][3], 0x0040);
    const uint32_t c45 = __byte_perm(o6[1][4], o6[1][5], 0x0040);
    own[0] = __byte_perm(a01, a23, 0x5410);
    own[1] = __byte_perm(a45, c01, 0x5410);
    own[2] = __byte_perm(c23, c45, 0x5410);
    if (!c.second_unit) {  // two-pixel last chunk: pixel 2 := pixel 1 (OpenCV's clamped right tap P[nw] = P[nw-1])
        own[2] = __byte_perm(own[1], 0u, 0x4441);             // byte 8 = byte 5
        own[1] = __byte_perm(own[0], own[1], 0x4354);         // bytes 4,5 kept; bytes 6,7 = bytes 3,4
    }
}

// own 12 bytes + the neighbouring pixels (by shuffle, or replicated at the image border) -> 24 horizontal-stage floats
__device__ __forceinline__ void x2w_expand(const X2wCtx& c, const uint32_t own[3], float x[24]) {
    const uint32_t from_left = __shfl_up_sync(0xFFFFFFFFu, own[2], 1);     // left lane's last pixel = its bytes 9..11
    const uint32_t from_right = __shfl_down_sync(0xFFFFFFFFu, own[0], 1);  // right lane's first pixel = its bytes 0..2
    const uint32_t w0 = c.first_chunk ? (own[0] << 8) : (from_left & 0xFFFFFF00u);
    const uint32_t w4 = c.last_chunk ? (own[2] >> 8) : (from_right & 0x00FFFFFFu);
    const uint32_t win[5] = {funnel_r(w0, own[0], 8), funnel_r(own[0], own[1], 8), funnel_r(own[1], own[2], 8),
                             funnel_r(own[2], w4, 8), w4 >> 8};
    x2_expand24(win, x);
}

// per-warp shared tables of one band (loads from shared memory use the short scoreboard, so waiting for a table
// entry never waits for the source prefetch that is in flight on the long scoreboard)
constexpr int kX2wMaxBandRows = 256;
constexpr int kX2wMaxLowRows = kX2wMaxBandRows / 2 + 8;
struct X2wWarpTables {
    float4 rc[kX2wMaxBandRows];   // vertical-stage constants per output row
    uint4 pk[kX2wMaxLowRows];     // {first source row, beta0, beta1, beta2} per low-res row
    uint32_t ys[kX2wMaxBandRows]; // s0 | s1 << 16 per output row
};

// Resident CTAs per SM of the band kernels: their __launch_bounds__ minimum and the grid of their launches.
// Measured on a B200 (128 x 1920x1080): lowres_x2p_kernel 3 CTAs/SM 5.88 TB/s, 4: 5.79, 2: 5.17.  The float-tap kernels
// are issue-bound and gain from more warps: lowres_x2f_kernel 4: 3.69, 3: 3.34, 2: 2.74 TB/s.  lowres_x2i_kernel at 4
// (128 registers): -5...+1 % (DESIGN section 4).  lowres_x2w_kernel: see below.
constexpr int kX2wCtasPerSm = 4, kX2pCtasPerSm = 3, kX2fCtasPerSm = 4, kX2hCtasPerSm = 4, kX2gCtasPerSm = 3, kX2iCtasPerSm = 3;

template <bool AL8>  // 128 registers, 4 CTAs per SM.  Measured alternatives: 96 registers / 5 CTAs (spills) -35 %;
                     // a 4-pixel-chunk variant with 80 registers / 6 CTAs -14 %: the kernel is issue-bound, not latency-bound
__global__ void __launch_bounds__(128, kX2wCtasPerSm) lowres_x2w_kernel(LowresX2wParams p) {
    extern __shared__ __align__(16) uint8_t smem[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, wpb = blockDim.x >> 5;
    X2wWarpTables& tb = reinterpret_cast<X2wWarpTables*>(smem)[warp];
    // tiles are handed out dynamically (one atomic per warp and tile): bands and strips differ in size, and a static
    // round-robin leaves a tail
    (void)wpb;
    for (;;) {
        int ti = 0;
        if (lane == 0) ti = (int)atomicAdd(p.counter, 1u);
        ti = __shfl_sync(0xFFFFFFFFu, ti, 0);
        if (ti >= p.n_tiles) break;
        const Tile t = p.tiles[ti];
        if (p.opcodes != nullptr && p.opcodes[t.img] != ROD_OP_LOWRES) continue;
        const DevImage im = p.images[t.img];
        const DevShape sh = p.shapes[im.shape_id];
        const uint8_t* simg = p.src + im.src_off;
        uint8_t* dimg = p.dst + im.dst_off;
        const int n = 3 * im.w, nw = sh.nw;
        const int nchunks = (im.w + 7) >> 3;
        const int ch = kX2wChunksPerStrip * t.c - 1 + lane;
        const bool cvalid = ch >= 0 && ch < nchunks;
        const int cc = min(max(ch, 0), nchunks - 1);
        const uint32_t* ly_s = p.tab + sh.ly_s;
        const float4* ly_rc = reinterpret_cast<const float4*>(p.tab + sh.ly_rc);
        const int Y0 = t.a, Y1 = t.b;
        const int j_first = (int)(ly_s[Y0] & 0xFFFFu), j_last = (int)(ly_s[Y1 - 1] >> 16);
        X2wCtx c;
        c.scol = simg + 24 * cc;
        c.pitch = im.src_pitch;
        c.ypack = tb.pk;
        c.j_first = j_first;
        c.h = im.h;
        c.fast2 = (sh.area_mode == AREA_FAST2);
        c.second_unit = (nw - 4 * cc) >= 4;
        c.first_chunk = (cc == 0);
        c.last_chunk = (cc == nchunks - 1);
        const int nvalid = (cvalid && lane >= 1 && lane <= kX2wChunksPerStrip) ? min(24, n - 24 * cc) : 0;
        const bool dst_al8 = ((((uintptr_t)dimg) | (uintptr_t)im.dst_pitch) & 7) == 0;

        __syncwarp();  // the previous band's tables are dead
        for (int i = lane; i < Y1 - Y0; i += 32) {
            tb.ys[i] = ly_s[Y0 + i];
            tb.rc[i] = ly_rc[Y0 + i];
        }
        if (!c.fast2) {
            const uint4* ypack = reinterpret_cast<const uint4*>(p.tab + sh.ay_pack);
            for (int i = lane; i <= j_last - j_first; i += 32) tb.pk[i] = ypack[j_first + i];
        }
        __syncwarp();

        uint32_t rw[3][6];
        uint4 pk = make_uint4(0u, 0u, 0u, 0u);
        float xe[24], xo[24];  // horizontal stage of the even / odd low-res row currently held
        int have = j_first - 1;  // highest low-res row produced so far
        x2w_prefetch<AL8>(c, j_first, rw, pk);
        uint8_t* dptr = dimg + (int64_t)Y0 * im.dst_pitch + 24 * cc;
        for (int r = Y0; r < Y1; ++r, dptr += im.dst_pitch) {
            const uint32_t ys = tb.ys[r - Y0];
            const float4 rf = tb.rc[r - Y0];
            const int s0 = (int)(ys & 0xFFFFu), s1 = (int)(ys >> 16);
            X2Row rc;
            rc.c0s = rf.x; rc.c1s = rf.y; rc.k0 = rf.z; rc.k2 = rf.w;
            while (have < s1) {
                ++have;
                uint32_t own[3];
                x2w_reduce(c, pk, rw, own);
                if (have < j_last) x2w_prefetch<AL8>(c, have + 1, rw, pk);
                if (have & 1) x2w_expand(c, own, xo);
                else x2w_expand(c, own, xe);
            }
            if (s0 & 1) {
                if (s1 & 1) x2_emit_row<true>(xo, xo, rc, dptr, nvalid, dst_al8);
                else x2_emit_row<true>(xo, xe, rc, dptr, nvalid, dst_al8);
            } else {
                if (s1 & 1) x2_emit_row<true>(xe, xo, rc, dptr, nvalid, dst_al8);
                else x2_emit_row<true>(xe, xe, rc, dptr, nvalid, dst_al8);
            }
        }
    }
}

// =====================================================================================
// Packed-integer kernel for shapes that are exact 2x in BOTH axes (even w and h at factor 0.5, w % 4 == 0, 4-byte aligned
// source and destination rows): 7 of the 8 VisDrone frame sizes.  Same work split as lowres_x2w_kernel (a warp owns a
// band of output rows x a strip of 30 chunks of 8 output pixels, lanes 0 and 31 are halo lanes), but
//   * the whole pipeline is integer arithmetic on packed 16-bit halves (rod_core.h x2p_*): per low-res row a lane forms
//     its twelve low-res values (resizeAreaFast_), the horizontal 2x stage and the two vertical-stage terms A / B' of
//     its 24 output byte columns; an output row is then ONE packed add per two bytes plus one byte permute per four.
//     No tables (the row pairs and the (1536, 512) y coefficients follow from the row parity), no floating point:
//     ~4.5 instructions per output byte where the float kernel needs 13.7;
//   * global memory is only touched by fully coalesced warp-wide copies: the two source rows of a low-res row are
//     staged in the warp's shared-memory ring by 16-byte cp.async copies (three stages in flight: the copies of low-res
//     rows j+1 and j+2 overlap the arithmetic of row j), and finished output rows leave through a shared staging
//     buffer as 16-byte stores.  (The first version had every lane load and store its own 24-byte chunk: 8 bytes of
//     every 32-byte sector per instruction, 3.6x / 3.0x the ideal sector count at L1 / L2 and 4.0 TB/s at 33 % issue
//     utilisation.)  Only __syncwarp() is used: warps never share data.
// =====================================================================================
constexpr int kX2pStages = 3;
constexpr int kX2pRowBytes = 32 * 24 + 32;  // staged source bytes of one row: 32 chunks + 16-byte phase + slack
constexpr int kX2pOutBytes = 30 * 24 + 32;  // one output row of the strip
struct alignas(16) X2pWarpSmem {
    uint8_t in[kX2pStages][2][kX2pRowBytes];
    uint8_t out[2][kX2pOutBytes];
};

__device__ __forceinline__ void cp_async16(uint32_t smem_addr, const void* gptr) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(smem_addr), "l"(gptr) : "memory");
}
__device__ __forceinline__ void cp_async4(uint32_t smem_addr, const void* gptr) {
    asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(smem_addr), "l"(gptr) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }
__device__ __forceinline__ void stg4s(void* p, uint32_t v) {
    asm volatile("st.global.L1::no_allocate.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ void stg16s(void* p, uint4 v) {
    asm volatile("st.global.L1::no_allocate.v4.u32 [%0], {%1,%2,%3,%4};" ::"l"(p), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
}

// Warp-cooperative copies between a global row segment and the warp's shared buffer.  Every lane moves the units
// lane, lane + 32, lane + 64, ... of the segment (unit = 16 bytes when the image qualifies: width a multiple of 16
// pixels and 16-byte aligned rows, so that every strip segment starts on a 16-byte boundary; else 4 bytes), so a lane's
// addresses are ONE running pointer (global base + unit * lane, advanced by the pitch per row) plus compile-time
// offsets, and a row costs two address instructions plus one copy per unit.
template <int U>
__device__ __forceinline__ void cp_async_u(uint32_t sm, const void* g) {
    if (U == 16) asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(sm), "l"(g) : "memory");
    else if (U == 8) asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(sm), "l"(g) : "memory");
    else asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(sm), "l"(g) : "memory");
}
template <int U>
__device__ __forceinline__ void x2p_copy_in(uint32_t sm_lane, const uint8_t* g_lane, int lane, int nunits) {
    constexpr int K = (kX2pRowBytes / U + 31) / 32;
#pragma unroll
    for (int k = 0; k < K; ++k)
        if (lane + 32 * k < nunits) cp_async_u<U>(sm_lane + 32 * U * k, g_lane + 32 * U * k);
}
template <int U>
__device__ __forceinline__ void x2p_copy_out(const uint8_t* sm_lane, uint8_t* g_lane, int lane, int nunits) {
    constexpr int K = (kX2wChunksPerStrip * 24 / U + 31) / 32;
#pragma unroll
    for (int k = 0; k < K; ++k) {
        if (lane + 32 * k < nunits) {
            if (U == 16) stg16s(g_lane + 32 * U * k, *reinterpret_cast<const uint4*>(sm_lane + 32 * U * k));
            else if (U == 8) { const uint2 v = *reinterpret_cast<const uint2*>(sm_lane + 32 * U * k); stg8(g_lane + 32 * U * k, v.x, v.y); }
            else stg4s(g_lane + 32 * U * k, *reinterpret_cast<const uint32_t*>(sm_lane + 32 * U * k));
        }
    }
}

struct X2pLane {
    int soff;             // byte offset of this lane's chunk inside a staged source row
    bool second;          // the chunk has four low-res pixels (else two: last chunk when w % 8 == 4)
    bool first, last;     // the chunk touches the left / right image border
};

// the lane's 24 source bytes of both rows of a ring slot (the staged chunk is 8-byte aligned)
__device__ __forceinline__ void x2p_read_stage(const uint8_t* st, int off, uint32_t rw[2][6]) {
#pragma unroll
    for (int t = 0; t < 2; ++t) {
        const uint2* r = reinterpret_cast<const uint2*>(st + t * kX2pRowBytes + off);
        const uint2 a = r[0], b = r[1], c = r[2];
        rw[t][0] = a.x; rw[t][1] = a.y; rw[t][2] = b.x; rw[t][3] = b.y; rw[t][4] = c.x; rw[t][5] = c.y;
    }
}

// the lane's low-res row from its source words: A / B' of its 24 output byte columns
__device__ __forceinline__ void x2p_finish(const X2pLane& c, uint32_t b[6], uint32_t A[12], uint32_t Bp[12]) {
    if (!c.second) x2p_patch_two_pixel(b);
    const uint32_t left_n9 = __shfl_up_sync(0xFFFFFFFFu, b[3], 1), left_n10 = __shfl_up_sync(0xFFFFFFFFu, x2p_n10(b), 1);
    const uint32_t right_b4 = __shfl_down_sync(0xFFFFFFFFu, b[4], 1), right_b0 = __shfl_down_sync(0xFFFFFFFFu, b[0], 1);
    x2p_build(b, left_n9, left_n10, right_b4, right_b0, c.first, c.last, A, Bp);
}

// one output row of the strip: every storing lane puts its 24 bytes into the staging buffer (8-byte aligned there), then
// the warp copies the row segment out with coalesced stores.  ooff < 0: this lane stores nothing.
template <int U>
__device__ __forceinline__ void x2p_store_row(uint8_t* ob, int ooff, const uint32_t* near_bp, const uint32_t* far_a,
                                              uint8_t* g_lane, int lane, int nunits) {
    if (ooff >= 0) {
        uint32_t w[6];
        x2p_emit(near_bp, far_a, w);
        uint2* o = reinterpret_cast<uint2*>(ob + ooff);
        o[0] = make_uint2(w[0], w[1]);
        o[1] = make_uint2(w[2], w[3]);
        o[2] = make_uint2(w[4], w[5]);
    }
    __syncwarp();
    x2p_copy_out<U>(ob + U * lane, g_lane, lane, nunits);
}

template <int U>
__device__ __forceinline__ void x2p_tile(const LowresX2wParams& p, const Tile& t, const DevImage& im, X2pWarpSmem& ws, int lane) {
    constexpr bool M16 = (U == 16);
    const uint32_t in_s = (uint32_t)__cvta_generic_to_shared(&ws.in[0][0][0]) + U * lane;
    const uint8_t* simg = p.src + im.src_off;
    uint8_t* dimg = p.dst + im.dst_off;
    const int n = 3 * im.w, nw = im.w >> 1, H = im.h, nh = H >> 1;
    const int nchunks = (im.w + 7) >> 3;
    const int c0 = kX2wChunksPerStrip * t.c;                     // first chunk this strip stores
    const int ch = c0 - 1 + lane;
    const int cc = min(max(ch, 0), nchunks - 1);
    // staged source segment: chunks [cs, ce]: the strip and one halo chunk either side, clipped to the row (16-byte
    // mode starts one chunk earlier so that 24 * cs is a multiple of 16)
    const int cs = max(c0 - (M16 ? 2 : 1), 0), ce = min(c0 + kX2wChunksPerStrip, nchunks - 1);
    const int in_units = (min(24 * (ce + 1), n) - 24 * cs + U - 1) / U;
    const int out_units = (min(24 * (c0 + kX2wChunksPerStrip), n) - 24 * c0) / U;   // chunks [c0, c0 + 30): a multiple of U
    X2pLane c;
    c.soff = 24 * (cc - cs);
    c.second = (nw - 4 * cc) >= 4;
    c.first = (cc == 0);
    c.last = (cc == nchunks - 1);
    const bool stores = ch >= 0 && ch < nchunks && lane >= 1 && lane <= kX2wChunksPerStrip;
    const int ooff = stores ? 24 * (lane - 1) : -1;
    const int Y0 = t.a, Y1 = t.b;                 // Y0 is even; Y1 is even or H (H is even)
    const int j0 = Y0 >> 1;
    const int jfirst = max(j0 - 1, 0), jlast = min(Y1 >> 1, nh - 1);
    const int64_t sp = im.src_pitch, dp = im.dst_pitch;
    const uint8_t* gin = simg + 24 * cs + U * lane + (int64_t)(2 * jfirst) * sp;   // this lane's unit 0 of the next row to stage
    uint8_t* gout = dimg + 24 * c0 + U * lane;                                     // ... of output row 0

    __syncwarp();  // the previous tile's reads of the ring are done
    // prologue: low-res rows jfirst .. jfirst + stages - 2 in flight
    int jn = jfirst;       // next low-res row to stage
    uint32_t sn = 0;       // its ring slot
#pragma unroll
    for (int q = 0; q < kX2pStages - 1; ++q) {
        if (jn <= jlast) {
            x2p_copy_in<U>(in_s + sn * (2 * kX2pRowBytes), gin, lane, in_units);
            x2p_copy_in<U>(in_s + sn * (2 * kX2pRowBytes) + kX2pRowBytes, gin + sp, lane, in_units);
            gin += 2 * sp;
        }
        cp_async_commit();
        ++jn;
        sn = (sn + 1 == kX2pStages) ? 0 : sn + 1;
    }
    uint32_t Ae[12], Be[12], Ao[12], Bo[12];      // A / B' of the latest even / odd low-res row
    int obuf = 0;
    uint32_t sc = 0;       // ring slot of low-res row j
    // low-res row j completes output rows 2j-1 (near row j-1, far row j) and 2j (near row j, far row j-1)
    for (int j = jfirst; j <= jlast; ++j) {
        if (jn <= jlast) {  // refill the slot that row j-1 used
            x2p_copy_in<U>(in_s + sn * (2 * kX2pRowBytes), gin, lane, in_units);
            x2p_copy_in<U>(in_s + sn * (2 * kX2pRowBytes) + kX2pRowBytes, gin + sp, lane, in_units);
            gin += 2 * sp;
        }
        cp_async_commit();
        ++jn;
        sn = (sn + 1 == kX2pStages) ? 0 : sn + 1;
        cp_async_wait<kX2pStages - 1>();  // this lane's copies of row j have landed ...
        __syncwarp();                     // ... and so have everybody else's
        uint32_t rw[2][6], b[6];
        x2p_read_stage(&ws.in[sc][0][0], c.soff, rw);
        sc = (sc + 1 == kX2pStages) ? 0 : sc + 1;
        x2p_area(rw[0], rw[1], b);
        const bool up = j > j0, down = j >= j0 && 2 * j < Y1;
        uint8_t* g1 = gout + (int64_t)(2 * j - 1) * dp;
        if (j & 1) {
            x2p_finish(c, b, Ao, Bo);
            if (up) { x2p_store_row<U>(ws.out[obuf], ooff, Be, Ao, g1, lane, out_units); obuf ^= 1; }
            if (down) { x2p_store_row<U>(ws.out[obuf], ooff, Bo, Ae, g1 + dp, lane, out_units); obuf ^= 1; }
        } else {
            x2p_finish(c, b, Ae, Be);
            if (up) { x2p_store_row<U>(ws.out[obuf], ooff, Bo, Ae, g1, lane, out_units); obuf ^= 1; }
            if (down) {
                if (j == 0) x2p_store_row<U>(ws.out[obuf], ooff, Be, Ae, gout, lane, out_units);   // row 0 blends low-res row 0 with itself
                else x2p_store_row<U>(ws.out[obuf], ooff, Be, Ao, g1 + dp, lane, out_units);
                obuf ^= 1;
            }
        }
        __syncwarp();  // all lanes have read their slot before the next iteration refills the one before it
    }
    if (Y1 == H) {  // the last image row blends low-res row nh-1 with itself
        if ((nh - 1) & 1) x2p_store_row<U>(ws.out[obuf], ooff, Bo, Ao, gout + (int64_t)(H - 1) * dp, lane, out_units);
        else x2p_store_row<U>(ws.out[obuf], ooff, Be, Ae, gout + (int64_t)(H - 1) * dp, lane, out_units);
    }
    cp_async_wait<0>();
}

// U: copy unit in bytes (16: image width a multiple of 16 and 16-byte aligned rows; 8; 4)
template <int U>
__global__ void __launch_bounds__(128, kX2pCtasPerSm) lowres_x2p_kernel(LowresX2wParams p) {
    extern __shared__ __align__(16) uint8_t smem[];
    const int lane = threadIdx.x & 31;
    X2pWarpSmem& ws = reinterpret_cast<X2pWarpSmem*>(smem)[threadIdx.x >> 5];
    for (;;) {
        int ti = 0;
        if (lane == 0) ti = (int)atomicAdd(p.counter, 1u);
        ti = __shfl_sync(0xFFFFFFFFu, ti, 0);
        if (ti >= p.n_tiles) break;
        const Tile t = p.tiles[ti];
        if (p.opcodes != nullptr && p.opcodes[t.img] != ROD_OP_LOWRES) continue;
        const DevImage im = p.images[t.img];
        x2p_tile<U>(p, t, im, ws, lane);
    }
}

// =====================================================================================
// Float-tap kernel for exact-2x WIDTHS whose height is not exact 2x (odd h at factor 0.5, e.g. 1360 x 765 -- the
// BASELINE frame size): INTER_AREA runs OpenCV's general path (x taps (0.5, 0.5), two or three float y taps per low-res
// row) and the INTER_LINEAR y coefficients are general.  Same strips, bands, halo lanes and shared-memory staging as
// lowres_x2p_kernel (coalesced cp.async in, coalesced stores out); the arithmetic is lowres_x2w_kernel's, trimmed:
//   * every SOURCE ROW is staged once in a ring of 8 rows and its pair sums are formed once: the last tap row of
//     low-res row j is the first tap row of row j+1 and its sums are carried in registers (x2w loaded and reduced
//     three tap rows per low-res row);
//   * the vertical stage is 2 FFMA.RZ per byte + a packed integer finish (rod_core.h x2_vertical_pair) instead of
//     3 FFMA.RZ + a byte pack;
//   * per-row constants come from the global tables through L1 one row ahead (nothing else is in flight on the
//     long scoreboard, the pixels arrive by cp.async), so no per-warp shared tables.
// =====================================================================================
constexpr int kX2fRing = 8;  // staged source rows per warp (power of two); eligibility (plan.cu): h <= 8 or h / nh <= 2.25
struct alignas(16) X2fWarpSmem {
    uint8_t in[kX2fRing][kX2pRowBytes];
    uint8_t out[2][kX2pOutBytes];
};

// own 12 low-res bytes + the neighbouring pixels (by shuffle, or replicated at the image border) -> 24 horizontal-stage floats
__device__ __forceinline__ void x2f_expand(const X2pLane& c, const uint32_t own[3], float x[24]) {
    const uint32_t from_left = __shfl_up_sync(0xFFFFFFFFu, own[2], 1);     // left lane's last pixel = its bytes 9..11
    const uint32_t from_right = __shfl_down_sync(0xFFFFFFFFu, own[0], 1);  // right lane's first pixel = its bytes 0..2
    const uint32_t w0 = c.first ? (own[0] << 8) : (from_left & 0xFFFFFF00u);
    const uint32_t w4 = c.last ? (own[2] >> 8) : (from_right & 0x00FFFFFFu);
    const uint32_t win[5] = {funnel_r(w0, own[0], 8), funnel_r(own[0], own[1], 8), funnel_r(own[1], own[2], 8),
                             funnel_r(own[2], w4, 8), w4 >> 8};
    x2_expand24(win, x);
}

// one output row: 24 bytes per lane from the horizontal stages of the two low-res rows it blends
template <int U>
__device__ __forceinline__ void x2f_store_row(uint8_t* ob, int ooff, const float* xlo, const float* xhi, float c0s, float c1s,
                                              float k0p, uint32_t cfix, uint8_t* g_lane, int lane, int nunits) {
    if (ooff >= 0) {
        uint32_t pr[12];
#pragma unroll
        for (int t = 0; t < 12; ++t)
            pr[t] = x2_vertical_pair(xlo[2 * t], xhi[2 * t], xlo[2 * t + 1], xhi[2 * t + 1], c0s, c1s, k0p, cfix);
        uint2* o = reinterpret_cast<uint2*>(ob + ooff);
#pragma unroll
        for (int g = 0; g < 3; ++g)
            o[g] = make_uint2(perm<0x7531>(pr[4 * g], pr[4 * g + 1]), perm<0x7531>(pr[4 * g + 2], pr[4 * g + 3]));
    }
    __syncwarp();
    x2p_copy_out<U>(ob + U * lane, g_lane, lane, nunits);
}

template <int U>
__device__ __forceinline__ void x2f_tile(const LowresX2wParams& p, const Tile& t, const DevImage& im, const DevShape& sh,
                                         X2fWarpSmem& ws, int lane) {
    constexpr bool M16 = (U == 16);
    const uint32_t in_s = (uint32_t)__cvta_generic_to_shared(&ws.in[0][0]) + U * lane;
    const uint8_t* simg = p.src + im.src_off;
    uint8_t* dimg = p.dst + im.dst_off;
    const int n = 3 * im.w, nw = sh.nw, H = im.h;
    const int nchunks = (im.w + 7) >> 3;
    const int c0 = kX2wChunksPerStrip * t.c;
    const int ch = c0 - 1 + lane;
    const int cc = min(max(ch, 0), nchunks - 1);
    const int cs = max(c0 - (M16 ? 2 : 1), 0), ce = min(c0 + kX2wChunksPerStrip, nchunks - 1);
    const int in_units = (min(24 * (ce + 1), n) - 24 * cs + U - 1) / U;
    const int out_units = (min(24 * (c0 + kX2wChunksPerStrip), n) - 24 * c0) / U;
    X2pLane c;
    c.soff = 24 * (cc - cs);
    c.second = (nw - 4 * cc) >= 4;
    c.first = (cc == 0);
    c.last = (cc == nchunks - 1);
    const bool stores = ch >= 0 && ch < nchunks && lane >= 1 && lane <= kX2wChunksPerStrip;
    const int ooff = stores ? 24 * (lane - 1) : -1;
    const int64_t sp = im.src_pitch, dp = im.dst_pitch;
    const uint8_t* gin = simg + 24 * cs + U * lane;    // this lane's unit 0 of source row 0
    uint8_t* gout = dimg + 24 * c0 + U * lane;         // ... of output row 0
    const uint32_t* ly_s = p.tab + sh.ly_s;
    const uint4* ypack = reinterpret_cast<const uint4*>(p.tab + sh.ay_pack);
    const int Y0 = t.a, Y1 = t.b;
    const int j_first = (int)(__ldg(ly_s + Y0) & 0xFFFFu), j_last = (int)(__ldg(ly_s + Y1 - 1) >> 16);

    // ---- staging: source rows are issued in increasing order, each once; one commit group per low-res row
    int next_row = (int)__ldg(ypack + j_first).x;
    const uint8_t* gnext = gin + (int64_t)next_row * sp;                           // this lane's unit 0 of source row next_row
    uint32_t snext = in_s + (uint32_t)((next_row & (kX2fRing - 1)) * kX2pRowBytes);  // its ring slot
    const uint32_t ring_end = in_s + kX2fRing * kX2pRowBytes;
    auto stage_for = [&](int jt) {   // make sure the tap rows of low-res row jt are on their way
        __syncwarp();                // nobody still reads the ring slots that are about to be refilled
        if (jt <= j_last) {
            const int target = min((int)__ldg(&ypack[jt].x) + 2, H - 1);
            while (next_row <= target) {
                x2p_copy_in<U>(snext, gnext, lane, in_units);
                gnext += sp;
                snext = (snext + kX2pRowBytes == ring_end) ? in_s : snext + kX2pRowBytes;
                ++next_row;
            }
        }
        cp_async_commit();
    };
    stage_for(j_first);
    stage_for(j_first + 1);

    float xe[24], xo[24];        // horizontal stage of the even / odd low-res row currently held
    uint32_t carry[12];          // pair sums of source row carry_row (the last tap row of the previous low-res row)
    int carry_row = -1;
    int have = j_first - 1;      // highest low-res row produced so far
    uint8_t* ob0 = ws.out[0];
    uint8_t* ob1 = ws.out[1];
    const uint8_t* in0 = &ws.in[0][c.soff];
    // per-row constants {c0s, c1s, k0 + 2, cfix} and row pairs, fetched one output row ahead through L1
    const float4* p_rc = reinterpret_cast<const float4*>(p.tab + sh.ly_rc2) + Y0;
    const uint32_t* p_ys = ly_s + Y0;
    uint32_t ys = __ldg(p_ys);
    float4 rf = __ldg(p_rc);
    uint4 pk = __ldg(ypack + j_first);   // {first tap row, beta0, beta1, beta2} of the next low-res row to produce
    uint8_t* grow = gout + (int64_t)Y0 * dp;
    for (int r = Y0; r < Y1; ++r, grow += dp) {
        const int s0 = (int)(ys & 0xFFFFu), s1 = (int)(ys >> 16);
        const float c0s = rf.x, c1s = rf.y, k0p = rf.z;
        const uint32_t cfix = __float_as_uint(rf.w);
        if (r + 1 < Y1) { ys = __ldg(++p_ys); rf = __ldg(++p_rc); }
        while (have < s1) {
            ++have;
            stage_for(have + 2);
            cp_async_wait<2>();   // this lane's copies for low-res row `have` have landed ...
            __syncwarp();         // ... and so have everybody else's
            const int sy0 = (int)pk.x;
            const float b0 = __uint_as_float(pk.y), b1 = __uint_as_float(pk.z), b2 = __uint_as_float(pk.w);
            if (have < j_last) pk = __ldg(ypack + have + 1);
            float acc[12];
#pragma unroll
            for (int tp = 0; tp < 3; ++tp) {
                const int row = (tp == 2) ? min(sy0 + 2, H - 1) : sy0 + tp;
                if (!(tp == 0 && row == carry_row)) {   // (warp-uniform) the first tap row is usually the carried one
                    const uint2* rp = reinterpret_cast<const uint2*>(in0 + (row & (kX2fRing - 1)) * kX2pRowBytes);
                    const uint2 a = rp[0], b = rp[1], d = rp[2];
                    const uint32_t rw[6] = {a.x, a.y, b.x, b.y, d.x, d.y};
                    x2f_pairsums(rw, carry);
                }
                x2f_mac(carry, tp == 0 ? b0 : (tp == 1 ? b1 : b2), tp == 0, acc);
                carry_row = row;
            }
            uint32_t o6[2][6];
            area_x2f_finish(acc, o6[0]);
            area_x2f_finish(acc + 6, o6[1]);
            uint32_t own[3];
            {
                const uint32_t a01 = __byte_perm(o6[0][0], o6[0][1], 0x0040), a23 = __byte_perm(o6[0][2], o6[0][3], 0x0040);
                const uint32_t a45 = __byte_perm(o6[0][4], o6[0][5], 0x0040);
                const uint32_t c01 = __byte_perm(o6[1][0], o6[1][1], 0x0040), c23 = __byte_perm(o6[1][2], o6[1][3], 0x0040);
                const uint32_t c45 = __byte_perm(o6[1][4], o6[1][5], 0x0040);
                own[0] = __byte_perm(a01, a23, 0x5410);
                own[1] = __byte_perm(a45, c01, 0x5410);
                own[2] = __byte_perm(c23, c45, 0x5410);
                if (!c.second) {  // two-pixel last chunk: pixel 2 := pixel 1 (OpenCV's clamped right tap P[nw] = P[nw-1])
                    own[2] = __byte_perm(own[1], 0u, 0x4441);
                    own[1] = __byte_perm(own[0], own[1], 0x4354);
                }
            }
            if (have & 1) x2f_expand(c, own, xo);
            else x2f_expand(c, own, xe);
        }
        // s1 is s0 + 1 except on the first / last image rows (s1 == s0): the parity of s0 picks the slots
        if (s1 != s0) {
            if (s0 & 1) x2f_store_row<U>(ob0, ooff, xo, xe, c0s, c1s, k0p, cfix, grow, lane, out_units);
            else x2f_store_row<U>(ob0, ooff, xe, xo, c0s, c1s, k0p, cfix, grow, lane, out_units);
        } else {
            if (s0 & 1) x2f_store_row<U>(ob0, ooff, xo, xo, c0s, c1s, k0p, cfix, grow, lane, out_units);
            else x2f_store_row<U>(ob0, ooff, xe, xe, c0s, c1s, k0p, cfix, grow, lane, out_units);
        }
        uint8_t* tswap = ob0; ob0 = ob1; ob1 = tswap;
    }
    cp_async_wait<0>();
}

template <int U>
__global__ void __launch_bounds__(128, kX2fCtasPerSm) lowres_x2f_kernel(LowresX2wParams p) {
    extern __shared__ __align__(16) uint8_t smem[];
    const int lane = threadIdx.x & 31;
    X2fWarpSmem& ws = reinterpret_cast<X2fWarpSmem*>(smem)[threadIdx.x >> 5];
    for (;;) {
        int ti = 0;
        if (lane == 0) ti = (int)atomicAdd(p.counter, 1u);
        ti = __shfl_sync(0xFFFFFFFFu, ti, 0);
        if (ti >= p.n_tiles) break;
        const Tile t = p.tiles[ti];
        if (p.opcodes != nullptr && p.opcodes[t.img] != ROD_OP_LOWRES) continue;
        const DevImage im = p.images[t.img];
        const DevShape sh = p.shapes[im.shape_id];
        x2f_tile<U>(p, t, im, sh, ws, lane);
    }
}

// =====================================================================================
// Regular three-tap kernel for exact-2x widths with h = 2 nh + 1 (DevShape::x2h: low-res row j reads source rows 2j, 2j+1,
// 2j+2 -- 1360 x 765, the BASELINE frame size).  Same arithmetic, strips, bands, halo lanes and coalesced staging as
// lowres_x2f_kernel, but the control flow is static so that the instruction stream is (almost) only arithmetic:
//   * the loop runs over LOW-RES rows, unrolled by parity (the even row's horizontal stage lives in xe, the odd row's in
//     xo: no register moves, no parity dispatch); a per-low-res-row table entry {beta0, beta1, beta2, first output row, nA,
//     nB} says which output rows leave once the row exists;
//   * source rows are staged as fixed pairs (2j+1, 2j+2) in a ring of four stages, one commit group per stage and one
//     __syncwarp per low-res row; row 2j is the previous stage's second row, whose pair sums are carried in registers;
//   * the per-output-row constants run two rows ahead in registers.
// (lowres_x2f_kernel spends 40 % of its instructions on ring / row bookkeeping: 317 warp instructions per output row of a
// strip where the arithmetic needs ~190.)
// =====================================================================================
constexpr int kX2hStages = 4;
__device__ __forceinline__ float4 ldg_early16(const void* p) {   // a read-only 16-byte load that stays where it is written
    float4 v;
    asm volatile("ld.global.nc.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "l"(p));
    return v;
}
struct alignas(16) X2hWarpSmem {
    uint8_t in[kX2hStages][2][kX2pRowBytes];
    uint8_t out[2][kX2pOutBytes];
};

template <int U>
struct X2hState {
    // staging
    uint32_t in_s;            // shared address of this lane's copy unit 0 in stage 0, row 0
    const uint8_t* gnext;     // this lane's unit 0 of the next source row to stage
    int64_t sp, dp;
    int in_units, out_units;
    int next_stage, n_stages;
    // reading
    const uint8_t* in0;       // this lane's chunk in stage 0, row 0
    // emission
    uint8_t* grow;            // this lane's copy unit 0 of the next output row
    uint32_t ob_s, ob_flip;   // shared address of the current output staging buffer; xor mask to the other one
    int ooff, loff;           // byte offsets in the staging buffer: this lane's chunk (< 0: stores nothing), its copy unit 0
    const float4* rc_tab;
    int r, H;
    int lane;
};

template <int U>
__device__ __forceinline__ void x2h_issue(X2hState<U>& s) {   // stage `next_stage`: source rows 2 jj + 1, 2 jj + 2
    if (s.next_stage < s.n_stages) {
        const uint32_t slot = s.in_s + (uint32_t)((s.next_stage & (kX2hStages - 1)) * (2 * kX2pRowBytes));
        x2p_copy_in<U>(slot, s.gnext, s.lane, s.in_units);
        x2p_copy_in<U>(slot + kX2pRowBytes, s.gnext + s.sp, s.lane, s.in_units);
        s.gnext += 2 * s.sp;
    }
    cp_async_commit();
    ++s.next_stage;
}

// one output row: 24 bytes per lane into the staging buffer, then the warp copies the row segment out with coalesced stores
template <int U>
__device__ __forceinline__ void x2h_emit_row(X2hState<U>& s, const float* xlo, const float* xhi, const float4 rf) {
    if (s.ooff >= 0) {
        const uint32_t cfix = __float_as_uint(rf.w);
        uint32_t pr[12];
#pragma unroll
        for (int t = 0; t < 12; ++t)
            pr[t] = x2_vertical_pair(xlo[2 * t], xhi[2 * t], xlo[2 * t + 1], xhi[2 * t + 1], rf.x, rf.y, rf.z, cfix);
        const uint32_t a = s.ob_s + (uint32_t)s.ooff;
#pragma unroll
        for (int g = 0; g < 3; ++g)
            asm volatile("st.shared.v2.u32 [%0], {%1,%2};" ::"r"(a + 8 * g), "r"(perm<0x7531>(pr[4 * g], pr[4 * g + 1])),
                         "r"(perm<0x7531>(pr[4 * g + 2], pr[4 * g + 3])) : "memory");
    }
    __syncwarp();
    constexpr int K = (kX2wChunksPerStrip * 24 / U + 31) / 32;
    const uint32_t l = s.ob_s + (uint32_t)s.loff;
#pragma unroll
    for (int k = 0; k < K; ++k) {
        if (s.lane + 32 * k < s.out_units) {
            if (U == 16) {
                uint4 v;
                asm volatile("ld.shared.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(l + 32 * U * k));
                stg16s(s.grow + 32 * U * k, v);
            } else if (U == 8) {
                uint2 v;
                asm volatile("ld.shared.v2.u32 {%0,%1}, [%2];" : "=r"(v.x), "=r"(v.y) : "r"(l + 32 * U * k));
                stg8(s.grow + 32 * U * k, v.x, v.y);
            } else {
                uint32_t v;
                asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(l + 32 * U * k));
                stg4s(s.grow + 32 * U * k, v);
            }
        }
    }
    s.ob_s ^= s.ob_flip;
    s.grow += s.dp;
    ++s.r;
}

// low-res row j: stage index st = j - j_first + 1.  xnew receives its horizontal stage, xprev holds row j - 1's.
template <int U>
__device__ __forceinline__ void x2h_row(X2hState<U>& s, const X2pLane& c, int st, uint4& hp_next, const uint4* hp_fetch,
                                        uint32_t carry[12], float* xnew, const float* xprev, int Y1) {
    cp_async_wait<kX2hStages - 2>();   // this lane's copies of stage st have landed ...
    __syncwarp();                      // ... and everybody else's; all lanes are done with the stage before it
    uint32_t ra[6], rb[6];
    {
        const uint8_t* sl = s.in0 + (st & (kX2hStages - 1)) * (2 * kX2pRowBytes);
        const uint2* pa = reinterpret_cast<const uint2*>(sl);
        const uint2* pb = reinterpret_cast<const uint2*>(sl + kX2pRowBytes);
        const uint2 a0 = pa[0], a1 = pa[1], a2 = pa[2], b0 = pb[0], b1 = pb[1], b2 = pb[2];
        ra[0] = a0.x; ra[1] = a0.y; ra[2] = a1.x; ra[3] = a1.y; ra[4] = a2.x; ra[5] = a2.y;
        rb[0] = b0.x; rb[1] = b0.y; rb[2] = b1.x; rb[3] = b1.y; rb[4] = b2.x; rb[5] = b2.y;
    }
    x2h_issue<U>(s);                   // refills the slot that was read one row ago
    const uint4 hp = hp_next;
    {
        const float4 t = ldg_early16(hp_fetch);
        hp_next = make_uint4(__float_as_uint(t.x), __float_as_uint(t.y), __float_as_uint(t.z), __float_as_uint(t.w));
    }
    // output rows whose lower tap row is j: [r0, r0 + nA) blend (j - 1, j), [r0 + nA, r0 + nA + nB) blend (j, j); the rows
    // before s.r have left already (s.r >= r0 by construction).  Constants of the first two, fetched before the arithmetic.
    const int ra_end = (int)(hp.w & 0xFFFFu) + (int)((hp.w >> 16) & 0xFFu);
    const int na = min(ra_end, Y1) - s.r, b_end = min(ra_end + (int)(hp.w >> 24), Y1);
    // (volatile: the compiler would otherwise sink these loads to their first use, after ~200 instructions of arithmetic)
    const float4 rc0 = ldg_early16(s.rc_tab + min(s.r, s.H - 1)), rc1 = ldg_early16(s.rc_tab + min(s.r + 1, s.H - 1));
    float acc[12];
    x2f_mac(carry, __uint_as_float(hp.x), true, acc);
    {
        uint32_t sa[12];
        x2f_pairsums(ra, sa);
        x2f_mac(sa, __uint_as_float(hp.y), false, acc);
    }
    x2f_pairsums(rb, carry);           // source row 2j + 2: also the first tap row of low-res row j + 1
    x2f_mac(carry, __uint_as_float(hp.z), false, acc);
    uint32_t o6[2][6];
    area_x2f_finish(acc, o6[0]);
    area_x2f_finish(acc + 6, o6[1]);
    uint32_t own[3];
    {
        const uint32_t a01 = __byte_perm(o6[0][0], o6[0][1], 0x0040), a23 = __byte_perm(o6[0][2], o6[0][3], 0x0040);
        const uint32_t a45 = __byte_perm(o6[0][4], o6[0][5], 0x0040);
        const uint32_t c01 = __byte_perm(o6[1][0], o6[1][1], 0x0040), c23 = __byte_perm(o6[1][2], o6[1][3], 0x0040);
        const uint32_t c45 = __byte_perm(o6[1][4], o6[1][5], 0x0040);
        own[0] = __byte_perm(a01, a23, 0x5410);
        own[1] = __byte_perm(a45, c01, 0x5410);
        own[2] = __byte_perm(c23, c45, 0x5410);
        if (!c.second) {  // two-pixel last chunk: pixel 2 := pixel 1 (OpenCV's clamped right tap P[nw] = P[nw-1])
            own[2] = __byte_perm(own[1], 0u, 0x4441);
            own[1] = __byte_perm(own[0], own[1], 0x4354);
        }
    }
    x2f_expand(c, own, xnew);
    if (na >= 1) {
        x2h_emit_row<U>(s, xprev, xnew, rc0);
        if (na >= 2) {
            x2h_emit_row<U>(s, xprev, xnew, rc1);
#pragma unroll 1
            for (int k = 2; k < na; ++k) x2h_emit_row<U>(s, xprev, xnew, __ldg(s.rc_tab + s.r));
        }
    }
#pragma unroll 1
    while (s.r < b_end) x2h_emit_row<U>(s, xnew, xnew, __ldg(s.rc_tab + s.r));   // top / bottom rows of the image only
}

template <int U>
__device__ __forceinline__ void x2h_tile(const LowresX2wParams& p, const Tile& t, const DevImage& im, const DevShape& sh,
                                         X2hWarpSmem& ws, int lane) {
    constexpr bool M16 = (U == 16);
    const uint8_t* simg = p.src + im.src_off;
    uint8_t* dimg = p.dst + im.dst_off;
    const int n = 3 * im.w, nw = sh.nw, H = im.h;
    const int nchunks = (im.w + 7) >> 3;
    const int c0 = kX2wChunksPerStrip * t.c;
    const int ch = c0 - 1 + lane;
    const int cc = min(max(ch, 0), nchunks - 1);
    const int cs = max(c0 - (M16 ? 2 : 1), 0), ce = min(c0 + kX2wChunksPerStrip, nchunks - 1);
    X2pLane c;
    c.soff = 24 * (cc - cs);
    c.second = (nw - 4 * cc) >= 4;
    c.first = (cc == 0);
    c.last = (cc == nchunks - 1);
    const bool stores = ch >= 0 && ch < nchunks && lane >= 1 && lane <= kX2wChunksPerStrip;
    const uint32_t* ly_s = p.tab + sh.ly_s;
    const uint4* hyp = reinterpret_cast<const uint4*>(p.tab + sh.hy_pack);
    const int Y0 = t.a, Y1 = t.b;
    const int j_first = (int)(__ldg(ly_s + Y0) & 0xFFFFu), j_last = (int)(__ldg(ly_s + Y1 - 1) >> 16);

    X2hState<U> s;
    s.lane = lane;
    s.in_s = (uint32_t)__cvta_generic_to_shared(&ws.in[0][0][0]) + U * lane;
    s.sp = im.src_pitch; s.dp = im.dst_pitch;
    s.in_units = (min(24 * (ce + 1), n) - 24 * cs + U - 1) / U;
    s.out_units = (min(24 * (c0 + kX2wChunksPerStrip), n) - 24 * c0) / U;
    s.in0 = &ws.in[0][0][c.soff];
    s.ooff = stores ? 24 * (lane - 1) : -1;
    s.loff = U * lane;
    s.ob_s = (uint32_t)__cvta_generic_to_shared(ws.out[0]);
    s.ob_flip = s.ob_s ^ (uint32_t)__cvta_generic_to_shared(ws.out[1]);
    s.grow = dimg + 24 * c0 + U * lane + (int64_t)Y0 * s.dp;
    s.rc_tab = reinterpret_cast<const float4*>(p.tab + sh.ly_rc2);
    s.r = Y0; s.H = H;
    // stage 0 holds source row 2 j_first alone (in its second row slot); stage st >= 1 rows 2 j + 1, 2 j + 2, j = j_first + st - 1
    s.n_stages = j_last - j_first + 2;
    s.gnext = simg + 24 * cs + U * lane + (int64_t)(2 * j_first) * s.sp;
    __syncwarp();  // the previous tile's reads of the ring are done
    x2p_copy_in<U>(s.in_s + kX2pRowBytes, s.gnext, lane, s.in_units);
    s.gnext += s.sp;
    cp_async_commit();
    s.next_stage = 1;
#pragma unroll
    for (int q = 1; q < kX2hStages - 1; ++q) x2h_issue<U>(s);
    uint4 hp_next = __ldg(hyp + j_first);

    float xe[24], xo[24];
    uint32_t carry[12];
    {   // stage 0: the pair sums of source row 2 j_first
        cp_async_wait<kX2hStages - 2>();
        __syncwarp();
        const uint2* pb = reinterpret_cast<const uint2*>(s.in0 + kX2pRowBytes);
        const uint2 b0 = pb[0], b1 = pb[1], b2 = pb[2];
        const uint32_t rb[6] = {b0.x, b0.y, b1.x, b1.y, b2.x, b2.y};
        x2h_issue<U>(s);
        x2f_pairsums(rb, carry);
    }
#pragma unroll 1
    for (int jj = j_first & ~1; jj <= j_last; jj += 2) {
        if (jj >= j_first) x2h_row<U>(s, c, jj - j_first + 1, hp_next, hyp + min(jj + 1, j_last), carry, xe, xo, Y1);
        if (jj + 1 <= j_last) x2h_row<U>(s, c, jj - j_first + 2, hp_next, hyp + min(jj + 2, j_last), carry, xo, xe, Y1);
    }
    cp_async_wait<0>();
}

template <int U>
__global__ void __launch_bounds__(128, kX2hCtasPerSm) lowres_x2h_kernel(LowresX2wParams p) {
    extern __shared__ __align__(16) uint8_t smem[];
    const int lane = threadIdx.x & 31;
    X2hWarpSmem& ws = reinterpret_cast<X2hWarpSmem*>(smem)[threadIdx.x >> 5];
    for (;;) {
        int ti = 0;
        if (lane == 0) ti = (int)atomicAdd(p.counter, 1u);
        ti = __shfl_sync(0xFFFFFFFFu, ti, 0);
        if (ti >= p.n_tiles) break;
        const Tile t = p.tiles[ti];
        if (p.opcodes != nullptr && p.opcodes[t.img] != ROD_OP_LOWRES) continue;
        const DevImage im = p.images[t.img];
        const DevShape sh = p.shapes[im.shape_id];
        x2h_tile<U>(p, t, im, sh, ws, lane);
    }
}

// =====================================================================================
// Odd-width kernel (w = 2 nw + 1 at factor 0.5; any height; rows at ANY byte alignment -- 3 w is odd, so consecutive rows
// of a contiguous image cycle through all four 4-byte phases).  Same strips, bands, halo lanes, source-row ring and carried
// tap row as lowres_x2f_kernel; what differs (rod_core.h x2g_*):
//   * staging copies whole aligned 4-byte words (cp.async) from the word that holds the segment's first byte, so a staged
//     row sits at its global phase (0..3) in the ring slot; a lane reads 8 aligned words and funnel-shifts them by that
//     (warp-uniform) phase into its 27-byte window (9 source pixels);
//   * the horizontal INTER_AREA stage is OpenCV's float pass with three taps per low-res column (per-column weights in
//     registers), the vertical one works on those floats;
//   * the INTER_LINEAR x stage uses the per-pixel coefficients and the per-pixel slip flag, the y stage the general
//     3 x FFMA.RZ form;
//   * output rows are byte aligned too: every lane shifts its 24 bytes by the row's destination phase (taking the
//     spill-over of its left neighbour by shuffle), so the staging buffer mirrors the global 4-byte words; the row leaves
//     as aligned 32-bit stores plus at most three byte stores at either end.
// This replaces the tiled lowres_kernel for these shapes (it ran at 0.7 TB/s: scalar byte loads per tap, three block
// barriers per tile).
// =====================================================================================
struct X2gLane {
    int soff;          // byte offset of this lane's window inside a staged source row (without the phase)
    int valid;         // valid low-res pixels of the chunk: min(4, nw - 4 * chunk), possibly <= 0
    bool first, last;  // the chunk touches the left / right image border
    uint32_t slip;     // bit k: odd output pixel 2k+1 of the chunk blends (P[k-1], P[k])
};

__device__ __forceinline__ void x2g_expand(const X2gLane& c, uint32_t own[3], const uint32_t coef[8], float x[24]) {
    const uint32_t from_left = __shfl_up_sync(0xFFFFFFFFu, own[2], 1);     // left lane's last pixel = its bytes 9..11
    if (c.valid < 4) x2g_replicate(own, max(c.valid, 0), from_left);
    const uint32_t from_right = __shfl_down_sync(0xFFFFFFFFu, own[0], 1);  // right lane's first pixel = its bytes 0..2
    const uint32_t w0 = c.first ? (own[0] << 8) : (from_left & 0xFFFFFF00u);
    const uint32_t w4 = c.last ? (own[2] >> 8) : (from_right & 0x00FFFFFFu);
    const uint32_t win[5] = {funnel_r(w0, own[0], 8), funnel_r(own[0], own[1], 8), funnel_r(own[1], own[2], 8),
                             funnel_r(own[2], w4, 8), w4 >> 8};
    x2g_expand24(win, coef, c.slip, x);
}

// one output row: the lane's 24 bytes, shifted to the destination row's 4-byte phase `ph`, into the staging buffer; then
// the warp stores the row segment [grow, grow + olen): head bytes, aligned words, tail bytes
__device__ __forceinline__ void x2g_store_row(uint8_t* ob, bool stores, const float* xlo, const float* xhi, const X2Row& rc,
                                              uint8_t* grow, int olen, int lane) {
    uint32_t o[24];
#pragma unroll
    for (int t = 0; t < 24; ++t) o[t] = x2_vertical(xlo[t], xhi[t], rc);
    uint32_t w[6];
#pragma unroll
    for (int g = 0; g < 6; ++g)
        w[g] = __byte_perm(__byte_perm(o[4 * g], o[4 * g + 1], 0x0040), __byte_perm(o[4 * g + 2], o[4 * g + 3], 0x0040), 0x5410);
    const int ph = (int)((uintptr_t)grow & 3);
    // buffer word 6 (lane - 1) + k = bytes [24 (lane - 1) + 4k - ph, +4) of the strip's output row: the last `ph` bytes of
    // the left neighbour's chunk, then own bytes
    const uint32_t prev = __shfl_up_sync(0xFFFFFFFFu, w[5], 1);
    const int sh = 32 - 8 * ph;  // ph == 0: funnel by 32 = the high word, i.e. w[k] itself
    uint32_t v[6];
    v[0] = ph ? __funnelshift_r(prev, w[0], sh) : w[0];
#pragma unroll
    for (int k = 1; k < 6; ++k) v[k] = ph ? __funnelshift_r(w[k - 1], w[k], sh) : w[k];
    if (lane >= 1) {  // (lane 31's words carry the spill-over of lane 30)
        uint2* q = reinterpret_cast<uint2*>(ob + 24 * (lane - 1));
        q[0] = make_uint2(v[0], v[1]); q[1] = make_uint2(v[2], v[3]); q[2] = make_uint2(v[4], v[5]);
    }
    (void)stores;
    __syncwarp();
    // buffer byte ph + i = output byte i of the segment
    const int head = min((4 - ph) & 3, olen);          // bytes before the first aligned global word
    const int nbody = (olen - head) >> 2;
    const int tail = olen - head - 4 * nbody;
    if (lane < head) grow[lane] = ob[ph + lane];
    if (lane >= 8 && lane - 8 < tail) grow[head + 4 * nbody + lane - 8] = ob[ph + head + 4 * nbody + lane - 8];
    const uint32_t* sb = reinterpret_cast<const uint32_t*>(ob + ph + head);   // 4-byte aligned: ph + head is 0 or 4
    uint32_t* gb = reinterpret_cast<uint32_t*>(grow + head);
#pragma unroll
    for (int k = 0; k < 6; ++k)
        if (lane + 32 * k < nbody) stg4s(gb + lane + 32 * k, sb[lane + 32 * k]);
}

__global__ void __launch_bounds__(128, kX2gCtasPerSm) lowres_x2g_kernel(LowresX2wParams p) {
    extern __shared__ __align__(16) uint8_t smem[];
    const int lane = threadIdx.x & 31;
    X2fWarpSmem& ws = reinterpret_cast<X2fWarpSmem*>(smem)[threadIdx.x >> 5];
    const uint32_t in_s = (uint32_t)__cvta_generic_to_shared(&ws.in[0][0]) + 4 * lane;
    for (;;) {
        int ti = 0;
        if (lane == 0) ti = (int)atomicAdd(p.counter, 1u);
        ti = __shfl_sync(0xFFFFFFFFu, ti, 0);
        if (ti >= p.n_tiles) break;
        const Tile t = p.tiles[ti];
        if (p.opcodes != nullptr && p.opcodes[t.img] != ROD_OP_LOWRES) continue;
        const DevImage im = p.images[t.img];
        const DevShape sh = p.shapes[im.shape_id];
        const uint8_t* simg = p.src + im.src_off;
        uint8_t* dimg = p.dst + im.dst_off;
        const int n = 3 * im.w, nw = sh.nw, H = im.h, W = im.w;
        const int nchunks = (W + 7) >> 3;
        const int c0 = kX2wChunksPerStrip * t.c;
        const int ch = c0 - 1 + lane;
        const int cc = min(max(ch, 0), nchunks - 1);
        const int cs = max(c0 - 1, 0), ce = min(c0 + kX2wChunksPerStrip, nchunks - 1);
        const int slen = min(24 * (ce + 1) + 3, n) - 24 * cs;          // staged bytes of a row: + the ninth pixel of chunk ce
        const int olen = min(24 * (c0 + kX2wChunksPerStrip), n) - 24 * c0;
        X2gLane c;
        c.soff = 24 * (cc - cs);
        c.valid = nw - 4 * cc;
        c.first = (cc == 0);
        c.last = (cc == nchunks - 1);
        const bool stores = ch >= 0 && ch < nchunks && lane >= 1 && lane <= kX2wChunksPerStrip;
        const int64_t sp = im.src_pitch, dp = im.dst_pitch;
        const uint8_t* sseg = simg + 24 * cs;
        uint8_t* dseg = dimg + 24 * c0;
        // per-lane column constants: area weights of its four low-res pixels, linear coefficients and slip flags of its
        // eight output pixels
        float al[12];
        uint32_t coef[8];
        {
            const float* xalpha = reinterpret_cast<const float*>(p.tab + sh.ax_alpha);
            const int32_t* lx_s0 = reinterpret_cast<const int32_t*>(p.tab + sh.lx_s0);
            const uint32_t* lx_a = p.tab + sh.lx_a;
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                const int dx = min(4 * cc + q, nw - 1);
#pragma unroll
                for (int tp = 0; tp < 3; ++tp) al[3 * q + tp] = __ldg(xalpha + 3 * dx + tp);
            }
            c.slip = 0;
#pragma unroll
            for (int x = 0; x < 8; ++x) {
                const int xa = min(8 * cc + x, W - 1);
                coef[x] = __ldg(lx_a + xa);
                if ((x & 1) && __ldg(lx_s0 + xa) == ((xa - 1) >> 1) - 1) c.slip |= 1u << (x >> 1);
            }
        }
        const uint32_t* ly_s = p.tab + sh.ly_s;
        const uint4* ypack = reinterpret_cast<const uint4*>(p.tab + sh.ay_pack);
        const int Y0 = t.a, Y1 = t.b;
        const int j_first = (int)(__ldg(ly_s + Y0) & 0xFFFFu), j_last = (int)(__ldg(ly_s + Y1 - 1) >> 16);

        // ---- staging: whole aligned words from the word that holds the segment's first byte; a row's ring slot then
        // holds it at its global phase
        int next_row = (int)__ldg(ypack + j_first).x;
        const uint8_t* gnext = sseg + (int64_t)next_row * sp;
        uint32_t snext = in_s + (uint32_t)((next_row & (kX2fRing - 1)) * kX2pRowBytes);
        const uint32_t ring_end = in_s + kX2fRing * kX2pRowBytes;
        auto stage_for = [&](int jt) {
            __syncwarp();
            if (jt <= j_last) {
                const int target = min((int)__ldg(&ypack[jt].x) + 2, H - 1);
                while (next_row <= target) {
                    const int ph = (int)((uintptr_t)gnext & 3);
                    x2p_copy_in<4>(snext, gnext - ph + 4 * lane, lane, (slen + ph + 3) >> 2);
                    gnext += sp;
                    snext = (snext + kX2pRowBytes == ring_end) ? in_s : snext + kX2pRowBytes;
                    ++next_row;
                }
            }
            cp_async_commit();
        };
        stage_for(j_first);
        stage_for(j_first + 1);

        float xe[24], xo[24];
        float carry[12];             // horizontal INTER_AREA values of source row carry_row
        int carry_row = -1;
        int have = j_first - 1;
        uint8_t* ob0 = ws.out[0];
        uint8_t* ob1 = ws.out[1];
        const uint8_t* in0 = &ws.in[0][c.soff];
        const float4* p_rc = reinterpret_cast<const float4*>(p.tab + sh.ly_rc3) + Y0;
        const uint32_t* p_ys = ly_s + Y0;
        uint32_t ys = __ldg(p_ys);
        float4 rf = __ldg(p_rc);
        uint4 pk = __ldg(ypack + j_first);
        uint8_t* grow = dseg + (int64_t)Y0 * dp;
        for (int r = Y0; r < Y1; ++r, grow += dp) {
            const int s0 = (int)(ys & 0xFFFFu), s1 = (int)(ys >> 16);
            X2Row rc;
            rc.c0s = rf.x; rc.c1s = rf.y; rc.k0 = rf.z; rc.k2 = rf.w;
            if (r + 1 < Y1) { ys = __ldg(++p_ys); rf = __ldg(++p_rc); }
            while (have < s1) {
                ++have;
                stage_for(have + 2);
                cp_async_wait<2>();
                __syncwarp();
                const int sy0 = (int)pk.x;
                const float b0 = __uint_as_float(pk.y), b1 = __uint_as_float(pk.z), b2 = __uint_as_float(pk.w);
                if (have < j_last) pk = __ldg(ypack + have + 1);
                float acc[12];
#pragma unroll
                for (int tp = 0; tp < 3; ++tp) {
                    const int row = (tp == 2) ? min(sy0 + 2, H - 1) : sy0 + tp;
                    if (!(tp == 0 && row == carry_row)) {
                        const int ph = (int)((uintptr_t)(sseg + (int64_t)row * sp) & 3);   // the staged row's phase (warp-uniform)
                        const uint2* rp = reinterpret_cast<const uint2*>(in0 + (row & (kX2fRing - 1)) * kX2pRowBytes);
                        const uint2 a = rp[0], b = rp[1], d = rp[2], e = rp[3];
                        const uint32_t raw[8] = {a.x, a.y, b.x, b.y, d.x, d.y, e.x, e.y};
                        uint32_t wn[7];
#pragma unroll
                        for (int k = 0; k < 7; ++k) wn[k] = __funnelshift_r(raw[k], raw[k + 1], 8 * ph);
                        x2g_hrow(wn, al, carry);
                    }
                    x2g_vmac(carry, tp == 0 ? b0 : (tp == 1 ? b1 : b2), tp == 0, acc);
                    carry_row = row;
                }
                uint32_t own[3];
                x2g_round12(acc, own);
                if (have & 1) x2g_expand(c, own, coef, xo);
                else x2g_expand(c, own, coef, xe);
            }
            if (s1 != s0) {
                if (s0 & 1) x2g_store_row(ob0, stores, xo, xe, rc, grow, olen, lane);
                else x2g_store_row(ob0, stores, xe, xo, rc, grow, olen, lane);
            } else {
                if (s0 & 1) x2g_store_row(ob0, stores, xo, xo, rc, grow, olen, lane);
                else x2g_store_row(ob0, stores, xe, xe, rc, grow, olen, lane);
            }
            uint8_t* tswap = ob0; ob0 = ob1; ob1 = tswap;
        }
        cp_async_wait<0>();
    }
}

// =====================================================================================
// Odd widths with a regular y axis (DevShape::x2i): lowres_x2g_kernel's arithmetic and byte-phase staging inside
// lowres_x2h_kernel's control structure -- a loop over low-res rows unrolled by parity, source rows staged as fixed pairs
// (CARRY, odd h: rows 2j+1, 2j+2 with row 2j's horizontal pass carried; else even h: rows 2j, 2j+1), the emission schedule
// of DevShape::hy_pack.  (lowres_x2g_kernel: 473 warp instructions per output row of a strip, ~290 of them arithmetic.)
// =====================================================================================
struct alignas(16) X2iWarpSmem {
    uint8_t in[kX2hStages][2][kX2pRowBytes];
    uint8_t out[2][kX2pOutBytes];
    float4 lc[8][32];   // per-lane column constants of the tile: [0..2] area weights, [3..5] -2^23 * weights, [6..7] linear coefficients
};
struct X2iState {
    uint32_t in_s;            // shared address of this lane's 16-byte unit 0 in stage 0, row 0
    const uint8_t* gnext;     // first byte of the strip's segment in the next source row to stage
    const uint8_t* gread;     // ... in the next source row to read from the ring (its low four bits place the row in its slot)
    int64_t sp, dp;
    int slen, olen;
    int next_stage, n_stages;
    uint32_t in0;             // shared address of this lane's window in stage 0, row 0 (without the row's 16-byte phase)
    uint8_t* grow;            // first byte of the strip's segment in the next output row
    uint32_t ob_s, ob_flip;   // shared address of the current output staging buffer; xor mask to the other one
    uint32_t lc_s;            // shared address of this lane's first constant vector (the others follow at 512-byte steps)
    bool first_strip, last_strip;
    const float4* rc_tab;
    int r, H;
    int lane;
};

// A source row is staged with 16-byte copies from the 16-byte block that holds the segment's first byte, so it sits in its
// ring slot at its global phase (0..15); the last unit copies only the bytes up to the segment's end (the rest is zero-filled).
__device__ __forceinline__ void x2i_stage_row(X2iState& s, uint32_t slot) {
    const int ph = (int)((uintptr_t)s.gnext & 15);
    const uint8_t* g = s.gnext - ph + 16 * s.lane;
    const int total = ph + s.slen;                      // bytes from the aligned start to the segment's end
    constexpr int K = (kX2pRowBytes / 16 + 31) / 32;
#pragma unroll
    for (int k = 0; k < K; ++k) {
        const int left = total - 16 * (s.lane + 32 * k);
        if (left > 0)
            asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(slot + 512 * k), "l"(g + 512 * k), "r"(min(left, 16)) : "memory");
    }
    s.gnext += s.sp;
}
__device__ __forceinline__ void x2i_issue(X2iState& s) {
    if (s.next_stage < s.n_stages) {
        const uint32_t slot = s.in_s + (uint32_t)((s.next_stage & (kX2hStages - 1)) * (2 * kX2pRowBytes));
        x2i_stage_row(s, slot);
        x2i_stage_row(s, slot + kX2pRowBytes);
    }
    cp_async_commit();
    ++s.next_stage;
}
// the lane's 27-byte window of the next source row to read (ring row at shared address `rowp`), shifted by the row's phase
__device__ __forceinline__ void x2i_window(X2iState& s, uint32_t rowp, uint32_t wn[7]) {
    const uint32_t ph = (uint32_t)((uintptr_t)s.gread & 15);
    s.gread += s.sp;
    const uint32_t a = rowp + (ph & ~3u);
    uint32_t raw[8];
#pragma unroll
    for (int k = 0; k < 8; ++k) asm volatile("ld.shared.u32 %0, [%1];" : "=r"(raw[k]) : "r"(a + 4 * k));
#pragma unroll
    for (int k = 0; k < 7; ++k) wn[k] = __funnelshift_r(raw[k], raw[k + 1], 8 * (ph & 3u));
}
// One output row.  Every lane shifts its 24 bytes by the destination row's 4-byte phase (taking the spill-over of its left
// neighbour by shuffle), so that the staging buffer mirrors the global 4-byte words: buffer word 0 = the aligned word that
// holds the segment's first byte.  The halo lanes' bytes are valid output too, so a segment that is not at the image border
// leaves as WHOLE aligned words (the two words it shares with the neighbouring strips are written by both, with the same
// bytes); only the first / last strip of a row finish with byte stores.
__device__ __forceinline__ void x2i_emit_row(X2iState& s, const float* xlo, const float* xhi, const float4 rf) {
    X2Row rc;
    rc.c0s = rf.x; rc.c1s = rf.y; rc.k0 = rf.z; rc.k2 = rf.w;
    uint32_t o[24];
#pragma unroll
    for (int t = 0; t < 24; ++t) o[t] = x2_vertical(xlo[t], xhi[t], rc);
    uint32_t w[6];
#pragma unroll
    for (int g = 0; g < 6; ++g)
        w[g] = __byte_perm(__byte_perm(o[4 * g], o[4 * g + 1], 0x0040), __byte_perm(o[4 * g + 2], o[4 * g + 3], 0x0040), 0x5410);
    const int ph = (int)((uintptr_t)s.grow & 3);
    const uint32_t prev = __shfl_up_sync(0xFFFFFFFFu, w[5], 1);
    uint32_t v[6];   // (w[k] << 8 ph) | (w[k-1] >> (32 - 8 ph)); ph == 0: the word itself
    v[0] = __funnelshift_l(prev, w[0], 8 * ph);
#pragma unroll
    for (int k = 1; k < 6; ++k) v[k] = __funnelshift_l(w[k - 1], w[k], 8 * ph);
    if (s.lane >= 1) {
        const uint32_t a = s.ob_s + 24u * (uint32_t)(s.lane - 1);
#pragma unroll
        for (int g = 0; g < 3; ++g)
            asm volatile("st.shared.v2.u32 [%0], {%1,%2};" ::"r"(a + 8 * g), "r"(v[2 * g]), "r"(v[2 * g + 1]) : "memory");
    }
    __syncwarp();
    // buffer byte ph + i = output byte i of the segment; buffer word q <-> the aligned global word at grow - ph + 4 q
    const int tot = ph + s.olen;
    int w_lo = 0, w_hi = (tot + 3) >> 2;
    if (s.first_strip | s.last_strip) {  // (warp-uniform, constant over the tile)
        if (s.first_strip && ph != 0) {  // the word before the row's first byte belongs to the previous row
            w_lo = 1;
            if (s.lane < 4 - ph && s.lane < s.olen) {
                uint32_t b;
                asm volatile("ld.shared.u8 %0, [%1];" : "=r"(b) : "r"(s.ob_s + ph + s.lane));
                s.grow[s.lane] = (uint8_t)b;
            }
        }
        if (s.last_strip) {              // ... and the bytes after the row's last one to the next row
            w_hi = tot >> 2;
            const int tail = tot & 3, q = 4 * w_hi - ph + (s.lane - 8);   // output byte handled by lanes 8..10
            if (s.lane >= 8 && s.lane - 8 < tail && q >= 0 && !(w_lo == 1 && w_hi == 0)) {
                uint32_t b;
                asm volatile("ld.shared.u8 %0, [%1];" : "=r"(b) : "r"(s.ob_s + ph + q));
                s.grow[q] = (uint8_t)b;
            }
        }
    }
    uint8_t* gb = s.grow - ph + 4 * s.lane;
    const uint32_t sb = s.ob_s + 4u * (uint32_t)s.lane;
#pragma unroll
    for (int k = 0; k < 6; ++k) {
        const int q = s.lane + 32 * k;
        if (q >= w_lo && q < w_hi) {
            uint32_t b;
            asm volatile("ld.shared.u32 %0, [%1];" : "=r"(b) : "r"(sb + 128 * k));
            stg4s(gb + 128 * k, b);
        }
    }
    s.ob_s ^= s.ob_flip;
    s.grow += s.dp;
    ++s.r;
}

__device__ __forceinline__ void x2i_lane_consts(uint32_t lc_s, float al[12], float nal[12]) {
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        asm volatile("ld.shared.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(al[4 * k]), "=f"(al[4 * k + 1]), "=f"(al[4 * k + 2]), "=f"(al[4 * k + 3]) : "r"(lc_s + 512u * k));
        asm volatile("ld.shared.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(nal[4 * k]), "=f"(nal[4 * k + 1]), "=f"(nal[4 * k + 2]), "=f"(nal[4 * k + 3]) : "r"(lc_s + 512u * (3 + k)));
    }
}

template <bool CARRY>
__device__ __forceinline__ void x2i_row(X2iState& s, X2gLane& c, int st, uint4& hp_next, const uint4* hp_fetch,
                                        float carry[12], float* xnew, const float* xprev, int Y1) {
    cp_async_wait<kX2hStages - 2>();
    __syncwarp();
    uint32_t wa[7], wb[7];
    {
        const uint32_t sl = s.in0 + (uint32_t)((st & (kX2hStages - 1)) * (2 * kX2pRowBytes));
        x2i_window(s, sl, wa);
        x2i_window(s, sl + kX2pRowBytes, wb);
    }
    x2i_issue(s);
    const uint4 hp = hp_next;
    hp_next = __ldg(hp_fetch);
    const int ra_end = (int)(hp.w & 0xFFFFu) + (int)((hp.w >> 16) & 0xFFu);
    const int na = min(ra_end, Y1) - s.r, b_end = min(ra_end + (int)(hp.w >> 24), Y1);
    const float4 rc0 = ldg_early16(s.rc_tab + min(s.r, s.H - 1)), rc1 = ldg_early16(s.rc_tab + min(s.r + 1, s.H - 1));
    float acc[12];
    {
        float al[12], nal[12];
        x2i_lane_consts(s.lc_s, al, nal);
        if (CARRY) {
            x2g_vmac(carry, __uint_as_float(hp.x), true, acc);
            {
                float ha[12];
                x2g_hrow_pre(wa, al, nal, ha);
                x2g_vmac(ha, __uint_as_float(hp.y), false, acc);
            }
            x2g_hrow_pre(wb, al, nal, carry);   // source row 2j + 2: also the first tap row of low-res row j + 1
            x2g_vmac(carry, __uint_as_float(hp.z), false, acc);
        } else {
            float ha[12];
            x2g_hrow_pre(wa, al, nal, ha);
            x2g_vmac(ha, __uint_as_float(hp.x), true, acc);
            x2g_hrow_pre(wb, al, nal, ha);
            x2g_vmac(ha, __uint_as_float(hp.y), false, acc);
        }
    }
    uint32_t own[3];
    x2g_round12(acc, own);
    {
        uint32_t coef[8];
#pragma unroll
        for (int k = 0; k < 2; ++k)
            asm volatile("ld.shared.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(coef[4 * k]), "=r"(coef[4 * k + 1]), "=r"(coef[4 * k + 2]), "=r"(coef[4 * k + 3])
                         : "r"(s.lc_s + 512u * (6 + k)));
        x2g_expand(c, own, coef, xnew);
    }
    if (na >= 1) {
        x2i_emit_row(s, xprev, xnew, rc0);
        if (na >= 2) {
            x2i_emit_row(s, xprev, xnew, rc1);
#pragma unroll 1
            for (int k = 2; k < na; ++k) x2i_emit_row(s, xprev, xnew, __ldg(s.rc_tab + s.r));
        }
    }
#pragma unroll 1
    while (s.r < b_end) x2i_emit_row(s, xnew, xnew, __ldg(s.rc_tab + s.r));
}

template <bool CARRY>
__device__ __forceinline__ void x2i_tile(const LowresX2wParams& p, const Tile& t, const DevImage& im, const DevShape& sh,
                                         X2iWarpSmem& ws, int lane) {
    constexpr int PRE = CARRY ? 1 : 0;
    const uint8_t* simg = p.src + im.src_off;
    uint8_t* dimg = p.dst + im.dst_off;
    const int n = 3 * im.w, nw = sh.nw, H = im.h, W = im.w;
    const int nchunks = (W + 7) >> 3;
    const int c0 = kX2wChunksPerStrip * t.c;
    const int cc = min(max(c0 - 1 + lane, 0), nchunks - 1);
    const int cs = max(c0 - 1, 0), ce = min(c0 + kX2wChunksPerStrip, nchunks - 1);
    X2gLane c;
    c.soff = 24 * (cc - cs);
    c.valid = nw - 4 * cc;
    c.first = (cc == 0);
    c.last = (cc == nchunks - 1);
    __syncwarp();  // the previous tile's reads of the ring and of the lane constants are done
    {
        float al[12];
        uint32_t coef[8];
        const float* xalpha = reinterpret_cast<const float*>(p.tab + sh.ax_alpha);
        const int32_t* lx_s0 = reinterpret_cast<const int32_t*>(p.tab + sh.lx_s0);
        const uint32_t* lx_a = p.tab + sh.lx_a;
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            const int dx = min(4 * cc + q, nw - 1);
#pragma unroll
            for (int tp = 0; tp < 3; ++tp) al[3 * q + tp] = __ldg(xalpha + 3 * dx + tp);
        }
        c.slip = 0;
#pragma unroll
        for (int x = 0; x < 8; ++x) {
            const int xa = min(8 * cc + x, W - 1);
            coef[x] = __ldg(lx_a + xa);
            if ((x & 1) && __ldg(lx_s0 + xa) == ((xa - 1) >> 1) - 1) c.slip |= 1u << (x >> 1);
        }
#pragma unroll
        for (int k = 0; k < 3; ++k) {
            ws.lc[k][lane] = make_float4(al[4 * k], al[4 * k + 1], al[4 * k + 2], al[4 * k + 3]);
            ws.lc[3 + k][lane] = make_float4(fmul(al[4 * k], -8388608.0f), fmul(al[4 * k + 1], -8388608.0f),
                                             fmul(al[4 * k + 2], -8388608.0f), fmul(al[4 * k + 3], -8388608.0f));
        }
#pragma unroll
        for (int k = 0; k < 2; ++k)
            ws.lc[6 + k][lane] = make_float4(__uint_as_float(coef[4 * k]), __uint_as_float(coef[4 * k + 1]),
                                             __uint_as_float(coef[4 * k + 2]), __uint_as_float(coef[4 * k + 3]));
    }
    const uint32_t* ly_s = p.tab + sh.ly_s;
    const uint4* hyp = reinterpret_cast<const uint4*>(p.tab + sh.hy_pack);
    const int Y0 = t.a, Y1 = t.b;
    const int j_first = (int)(__ldg(ly_s + Y0) & 0xFFFFu), j_last = (int)(__ldg(ly_s + Y1 - 1) >> 16);

    X2iState s;
    s.lc_s = (uint32_t)__cvta_generic_to_shared(&ws.lc[0][lane]);
    s.lane = lane;
    s.in_s = (uint32_t)__cvta_generic_to_shared(&ws.in[0][0][0]) + 16 * lane;
    s.sp = im.src_pitch; s.dp = im.dst_pitch;
    s.slen = min(24 * (ce + 1) + 3, n) - 24 * cs;          // staged bytes of a row: + the ninth pixel of chunk ce
    s.olen = min(24 * (c0 + kX2wChunksPerStrip), n) - 24 * c0;
    s.in0 = (uint32_t)__cvta_generic_to_shared(&ws.in[0][0][0]) + (uint32_t)c.soff;
    s.ob_s = (uint32_t)__cvta_generic_to_shared(ws.out[0]);
    s.ob_flip = s.ob_s ^ (uint32_t)__cvta_generic_to_shared(ws.out[1]);
    s.first_strip = (c0 == 0);
    s.last_strip = (c0 + kX2wChunksPerStrip >= nchunks);
    s.grow = dimg + 24 * c0 + (int64_t)Y0 * s.dp;
    s.rc_tab = reinterpret_cast<const float4*>(p.tab + sh.ly_rc3);
    s.r = Y0; s.H = H;
    // CARRY: stage 0 holds source row 2 j_first alone (second row slot), stage st >= 1 rows 2j + 1, 2j + 2 (j = j_first + st - 1);
    // else stage st holds rows 2j, 2j + 1 (j = j_first + st)
    s.n_stages = j_last - j_first + 1 + PRE;
    s.gnext = simg + 24 * cs + (int64_t)(2 * j_first) * s.sp;
    s.gread = s.gnext;
    __syncwarp();  // the previous tile's reads of the ring are done
    s.next_stage = 0;
    if (CARRY) {
        x2i_stage_row(s, s.in_s + kX2pRowBytes);
        cp_async_commit();
        s.next_stage = 1;
    }
#pragma unroll
    for (int q = PRE; q < kX2hStages - 1; ++q) x2i_issue(s);
    uint4 hp_next = __ldg(hyp + j_first);

    float xe[24], xo[24];
    float carry[12];
    if (CARRY) {   // stage 0: the horizontal pass of source row 2 j_first
        cp_async_wait<kX2hStages - 2>();
        __syncwarp();
        uint32_t wb[7];
        x2i_window(s, s.in0 + (uint32_t)kX2pRowBytes, wb);
        x2i_issue(s);
        float al[12], nal[12];
        x2i_lane_consts(s.lc_s, al, nal);
        x2g_hrow_pre(wb, al, nal, carry);
    }
#pragma unroll 1
    for (int jj = j_first & ~1; jj <= j_last; jj += 2) {
        if (jj >= j_first) x2i_row<CARRY>(s, c, jj - j_first + PRE, hp_next, hyp + min(jj + 1, j_last), carry, xe, xo, Y1);
        if (jj + 1 <= j_last) x2i_row<CARRY>(s, c, jj - j_first + 1 + PRE, hp_next, hyp + min(jj + 2, j_last), carry, xo, xe, Y1);
    }
    cp_async_wait<0>();
}

template <bool CARRY>
__global__ void __launch_bounds__(128, kX2iCtasPerSm) lowres_x2i_kernel(LowresX2wParams p) {
    extern __shared__ __align__(16) uint8_t smem[];
    const int lane = threadIdx.x & 31;
    X2iWarpSmem& ws = reinterpret_cast<X2iWarpSmem*>(smem)[threadIdx.x >> 5];
    for (;;) {
        int ti = 0;
        if (lane == 0) ti = (int)atomicAdd(p.counter, 1u);
        ti = __shfl_sync(0xFFFFFFFFu, ti, 0);
        if (ti >= p.n_tiles) break;
        const Tile t = p.tiles[ti];
        if (p.opcodes != nullptr && p.opcodes[t.img] != ROD_OP_LOWRES) continue;
        const DevImage im = p.images[t.img];
        const DevShape sh = p.shapes[im.shape_id];
        x2i_tile<CARRY>(p, t, im, sh, ws, lane);
    }
}

namespace {
// The launches of one LowRes call touch disjoint images, so they may run concurrently: with more than one non-empty
// tile list they are spread over the caller's stream and two plan-owned streams forked from / joined into it (events:
// capturable), so that the persistent CTAs of the next kernel move in while the last tiles of the previous one finish.
struct LrStreams {
    cudaStream_t s[3];
    int n, i;
    cudaStream_t pick() { const cudaStream_t r = s[i]; i = (i + 1) % n; return r; }
};

using BandKernel = void (*)(LowresX2wParams);
// staged kernels by copy unit: 16, 8, 4 bytes
const BandKernel kX2pKernels[3] = {lowres_x2p_kernel<16>, lowres_x2p_kernel<8>, lowres_x2p_kernel<4>};
const BandKernel kX2fKernels[3] = {lowres_x2f_kernel<16>, lowres_x2f_kernel<8>, lowres_x2f_kernel<4>};
const BandKernel kX2hKernels[3] = {lowres_x2h_kernel<16>, lowres_x2h_kernel<8>, lowres_x2h_kernel<4>};

// The order of the launches decides the stream each one is dealt to: generic, x2g, x2i, the staged kernels, x2w, strips.
int launch_lowres_lists(const rod_plan* plan, const uint8_t* src, uint8_t* dst, const uint8_t* opcodes, LrStreams& ls,
                        int img_lo, int img_hi) {
    // tile list `l` with a band kernel: four warps per CTA take tiles from a fresh work counter (launches of one plan may
    // overlap on different streams), grid sized for `per_sm` resident CTAs
    auto band = [&](int l, BandKernel kernel, size_t smem, int per_sm) -> int {
        const auto [tiles, n_tiles] = plan->lowres[l].range(img_lo, img_hi);
        if (n_tiles == 0) return ROD_OK;
        LowresX2wParams p;
        const cudaStream_t lst = ls.pick();
        p.images = plan->d_images;
        p.tiles = tiles;
        p.n_tiles = n_tiles;
        p.shapes = plan->d_shapes;
        p.tab = plan->d_tab;
        p.src = src; p.dst = dst; p.opcodes = opcodes;
        p.counter = plan->d_counters + (plan->launch_seq.fetch_add(1u) & (kCounterRing - 1u));
        ROD_CUDA(cudaMemsetAsync(p.counter, 0, sizeof(unsigned int), lst));
        ROD_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        kernel<<<grid_for(plan, (n_tiles + 3) / 4, per_sm), 128, smem, lst>>>(p);
        ROD_CUDA(cudaGetLastError());
        return ROD_OK;
    };
    // generic tiles (shapes that are not exact-2x in x)
    if (const auto [tiles, n_tiles] = plan->lowres[LR_GENERIC].range(img_lo, img_hi); n_tiles > 0) {
        LowresParams p;
        const cudaStream_t lst = ls.pick();
        p.images = plan->d_images;
        p.tiles = tiles;
        p.n_tiles = n_tiles;
        p.shapes = plan->d_shapes;
        p.tab = plan->d_tab;
        p.src = src; p.dst = dst; p.opcodes = opcodes;
        p.half_rows = plan->lowres_half_rows;
        p.p_pitch = (3 * (plan->lowres_half_cols + 3) + 15) & ~15;
        p.hb_pitch = 3 * plan->lowres_half_cols + 1;
        const size_t un = (std::max((size_t)plan->lowres_src_rows * p.hb_pitch * 4, (size_t)p.half_rows * kHxPitch * 2) + 15) & ~(size_t)15;
        p.union_bytes = (int)un;
        const size_t smem = (((size_t)p.half_rows * p.p_pitch + 15) & ~(size_t)15) + un + (size_t)p.half_rows * (2 + kMaxAreaTaps) * 4 + 16;
        if (smem > 227 * 1024) return ROD_ERR_UNSUPPORTED;
        ROD_CUDA(cudaFuncSetAttribute(lowres_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        int ctas_per_sm = (int)((220 * 1024) / (smem + 1024));
        ctas_per_sm = ctas_per_sm < 1 ? 1 : (ctas_per_sm > 3 ? 3 : ctas_per_sm);
        lowres_kernel<<<grid_for(plan, p.n_tiles, ctas_per_sm), 256, smem, lst>>>(p);
        ROD_CUDA(cudaGetLastError());
    }
    // odd widths at factor 0.5: the staged odd-width kernel (no alignment requirement) ...
    int rc = band(LR_X2G, lowres_x2g_kernel, 4 * sizeof(X2fWarpSmem), kX2gCtasPerSm);
    // ... and of those, the shapes with a regular y axis: the low-res-row loop kernel (odd h: carried tap row; even h)
    if (rc == ROD_OK) rc = band(LR_X2I_CARRY, lowres_x2i_kernel<true>, 4 * sizeof(X2iWarpSmem), kX2iCtasPerSm);
    if (rc == ROD_OK) rc = band(LR_X2I_EVEN, lowres_x2i_kernel<false>, 4 * sizeof(X2iWarpSmem), kX2iCtasPerSm);
    if (rc != ROD_OK) return rc;
    // exact-2x shapes: warp-marching kernels when the rows are 4-byte aligned, full-width strips otherwise
    int n_packed = 0;
    for (int l = LR_X2P16; l <= LR_X2H4; ++l) n_packed += plan->lowres[l].n;
    const bool use_bands = (plan->lowres[LR_X2W8].n + plan->lowres[LR_X2W4].n + n_packed) > 0 &&
                           (((uintptr_t)src) & 3) == 0 && (n_packed == 0 || (((uintptr_t)dst) & 3) == 0);
    if (use_bands) {
        // staged kernels (packed-integer: exact 2x in both axes; float taps: exact-2x width only; regular three-tap), one
        // launch per copy-unit class.  The list's copy unit holds for offsets and pitches; the base pointers may be less
        // aligned.
        const uintptr_t base = (uintptr_t)src | (uintptr_t)dst;
        const int base_unit = (base & 15) == 0 ? 0 : ((base & 7) == 0 ? 1 : 2);
        for (int u = 0; u < 3 && rc == ROD_OK; ++u)
            rc = band(LR_X2P16 + u, kX2pKernels[std::max(u, base_unit)], 4 * sizeof(X2pWarpSmem), kX2pCtasPerSm);
        for (int u = 0; u < 3 && rc == ROD_OK; ++u)
            rc = band(LR_X2F16 + u, kX2fKernels[std::max(u, base_unit)], 4 * sizeof(X2fWarpSmem), kX2fCtasPerSm);
        for (int u = 0; u < 3 && rc == ROD_OK; ++u)
            rc = band(LR_X2H16 + u, kX2hKernels[std::max(u, base_unit)], 4 * sizeof(X2hWarpSmem), kX2hCtasPerSm);
        // warp-marching kernel: images with 8-byte aligned rows (64-bit loads), then the others
        const BandKernel x2w8 = (((uintptr_t)src) & 7) == 0 ? lowres_x2w_kernel<true> : lowres_x2w_kernel<false>;
        if (rc == ROD_OK) rc = band(LR_X2W8, x2w8, 4 * sizeof(X2wWarpTables), kX2wCtasPerSm);
        if (rc == ROD_OK) rc = band(LR_X2W4, lowres_x2w_kernel<false>, 4 * sizeof(X2wWarpTables), kX2wCtasPerSm);
        if (rc != ROD_OK) return rc;
    }
    if (const auto [tiles, n_tiles] = plan->lowres[use_bands ? LR_X2_REST : LR_X2_STRIP].range(img_lo, img_hi); n_tiles > 0) {
        LowresX2Params p;
        const cudaStream_t lst = ls.pick();
        p.images = plan->d_images;
        p.tiles = tiles;
        p.n_tiles = n_tiles;
        p.shapes = plan->d_shapes;
        p.tab = plan->d_tab;
        p.src = src; p.dst = dst; p.opcodes = opcodes;
        const size_t smem = plan->lowres_x2_smem;
        int ctas_per_sm = (int)((220 * 1024) / (smem + 1024));
        ctas_per_sm = ctas_per_sm < 1 ? 1 : ctas_per_sm;
        ROD_CUDA(cudaFuncSetAttribute(lowres_x2_kernel<128>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        lowres_x2_kernel<128><<<grid_for(plan, p.n_tiles, ctas_per_sm > 4 ? 4 : ctas_per_sm), 128, smem, lst>>>(p);
        ROD_CUDA(cudaGetLastError());
    }
    return ROD_OK;
}
}  // namespace

int launch_lowres(const rod_plan* plan, const uint8_t* src, uint8_t* dst, const uint8_t* opcodes,
                  cudaStream_t stream, int img_lo, int img_hi) {
    int n_lists = 0;  // the full strip list replaces the others when it runs
    for (int l = 0; l < LR_NUM_LISTS; ++l) n_lists += l != LR_X2_STRIP && plan->lowres[l].range(img_lo, img_hi).second > 0;
    LrStreams ls;
    ls.s[0] = stream; ls.s[1] = ls.s[2] = nullptr;
    ls.n = 1; ls.i = 0;
    if (n_lists < 2) return launch_lowres_lists(plan, src, dst, opcodes, ls, img_lo, img_hi);
    // the fork / join of one call must not interleave with another host thread's on the same plan
    std::lock_guard<std::mutex> lock(plan->lr_mutex);
    if (plan->lr_ev_fork == nullptr) {  // created as a whole or not at all
        cudaStream_t s2[2] = {nullptr, nullptr};
        cudaEvent_t ef = nullptr, ej[2] = {nullptr, nullptr};
        cudaError_t e = cudaSuccess;
        for (auto& s : s2)
            if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&s, cudaStreamNonBlocking);
        if (e == cudaSuccess) e = cudaEventCreateWithFlags(&ef, cudaEventDisableTiming);
        for (auto& ev : ej)
            if (e == cudaSuccess) e = cudaEventCreateWithFlags(&ev, cudaEventDisableTiming);
        if (e != cudaSuccess) {
            for (auto& s : s2) if (s) cudaStreamDestroy(s);
            if (ef) cudaEventDestroy(ef);
            for (auto& ev : ej) if (ev) cudaEventDestroy(ev);
            return cuda_fail(e);
        }
        plan->lr_streams[0] = s2[0]; plan->lr_streams[1] = s2[1];
        plan->lr_ev_join[0] = ej[0]; plan->lr_ev_join[1] = ej[1];
        plan->lr_ev_fork = ef;
    }
    ROD_CUDA(cudaEventRecord(plan->lr_ev_fork, stream));
    for (auto& s : plan->lr_streams) ROD_CUDA(cudaStreamWaitEvent(s, plan->lr_ev_fork, 0));
    ls.s[1] = plan->lr_streams[0]; ls.s[2] = plan->lr_streams[1];
    ls.n = 3;
    int rc = launch_lowres_lists(plan, src, dst, opcodes, ls, img_lo, img_hi);
    for (int i = 0; i < 2; ++i) {  // the join is executed on every path
        cudaError_t e = cudaEventRecord(plan->lr_ev_join[i], plan->lr_streams[i]);
        if (e == cudaSuccess) e = cudaStreamWaitEvent(stream, plan->lr_ev_join[i], 0);
        if (e != cudaSuccess && rc == ROD_OK) rc = cuda_fail(e);
    }
    return rc;
}

}  // namespace rod
