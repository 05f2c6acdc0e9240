// rod_tables.h -- host-side (plain C++) construction of the resize tables and tile lists.
//
// Restates, in double/float arithmetic identical to OpenCV 4.13.0's resize.cpp, the
// coefficient tables of cv::resize(INTER_AREA) (computeResizeAreaTab) and of the 8-bit
// INTER_LINEAR path (fixed point, INTER_RESIZE_COEF_BITS = 11) that
// scripts/augmentations.py:44-45 invokes.  Used by plan.cu (uploaded to the GPU) and by
// the CPU emulation harness in tests/emu (no CUDA needed).
#pragma once
#include <math.h>
#include <stdint.h>
#include <string.h>

#include <algorithm>
#include <vector>

#include "rod_core.h"

namespace rod {

struct AreaAxis {
    std::vector<int32_t> first, count;
    std::vector<float> alpha;  // [dsize * taps]
    int taps = 1;
};

// computeResizeAreaTab: taps of destination d are consecutive source indices.
inline AreaAxis build_area_axis(int ssize, int dsize) {
    AreaAxis ax;
    ax.first.assign(dsize, 0);
    ax.count.assign(dsize, 0);
    std::vector<std::vector<float>> rows(dsize);
    double scale = (double)ssize / (double)dsize;
    for (int d = 0; d < dsize; ++d) {
        double f1 = d * scale;
        double f2 = f1 + scale;
        double cell = std::min(scale, ssize - f1);
        int s1 = (int)ceil(f1), s2 = (int)floor(f2);
        s2 = std::min(s2, ssize - 1);
        s1 = std::min(s1, s2);
        bool have = false;
        auto emit = [&](int s, float a) {
            if (!have) { ax.first[d] = s; have = true; }
            rows[d].push_back(a);
        };
        if (s1 - f1 > 1e-3) emit(s1 - 1, (float)((s1 - f1) / cell));
        for (int s = s1; s < s2; ++s) emit(s, (float)(1.0 / cell));
        if (f2 - s2 > 1e-3) emit(s2, (float)(std::min(std::min(f2 - s2, 1.0), cell) / cell));
        ax.count[d] = (int)rows[d].size();
        ax.taps = std::max(ax.taps, ax.count[d]);
    }
    ax.alpha.assign((size_t)dsize * ax.taps, 0.0f);
    for (int d = 0; d < dsize; ++d)
        for (int t = 0; t < ax.count[d]; ++t) ax.alpha[(size_t)d * ax.taps + t] = rows[d][t];
    return ax;
}

struct LinearAxis {
    std::vector<int32_t> s0, s1;     // clipped source indices
    std::vector<uint32_t> coef;      // a0 | a1 << 16   (11-bit fixed point)
};

// 8-bit INTER_LINEAR tables.  clamp_x = true: the x axis (index and fraction clamped at both
// ends); false: the y axis (fraction kept, only the two row indices are clipped).
inline LinearAxis build_linear_axis(int ssize, int dsize, bool clamp_x) {
    LinearAxis ax;
    ax.s0.resize(dsize);
    ax.s1.resize(dsize);
    ax.coef.resize(dsize);
    double scale = 1.0 / ((double)dsize / (double)ssize);
    for (int d = 0; d < dsize; ++d) {
        float f = (float)((d + 0.5) * scale - 0.5);
        int s = (int)floorf(f);
        f -= (float)s;
        if (clamp_x) {
            if (s < 0) { s = 0; f = 0.f; }
            if (s >= ssize - 1) { s = ssize - 1; f = 0.f; }
        }
        volatile float c0 = 1.f - f;
        volatile float m0 = c0 * 2048.f, m1 = f * 2048.f;
        int a0 = (int)lrintf(m0), a1 = (int)lrintf(m1);
        ax.s0[d] = std::min(std::max(s, 0), ssize - 1);
        ax.s1[d] = std::min(std::max(s + 1, 0), ssize - 1);
        ax.coef[d] = (uint32_t)(a0 & 0xFFFF) | ((uint32_t)(a1 & 0xFFFF) << 16);
    }
    return ax;
}

inline void lowres_small_size(int h, int w, double factor, int* nh, int* nw) {
    // augmentations.py:43: max(1, int(w * factor)) -- Python float multiply then truncation
    *nw = std::max(1, (int)((double)w * factor));
    *nh = std::max(1, (int)((double)h * factor));
}

// Append a 32-bit-word array to the blob and return its word offset.
template <typename T>
inline uint32_t blob_push(std::vector<uint32_t>& blob, const std::vector<T>& v) {
    static_assert(sizeof(T) == 4, "table entries are 32-bit");
    uint32_t off = (uint32_t)blob.size();
    blob.resize(blob.size() + v.size());
    if (!v.empty()) memcpy(blob.data() + off, v.data(), v.size() * 4);
    while (blob.size() % 4) blob.push_back(0);  // keep every table 16-byte aligned
    return off;
}

// Tables of the lowres round trip for one (h, w).  Returns false if unsupported (too many taps).
inline bool build_lowres_shape(int h, int w, double factor, int max_taps, std::vector<uint32_t>& blob,
                               DevShape* out) {
    DevShape sh;
    memset(&sh, 0, sizeof(sh));
    sh.h = h; sh.w = w;
    lowres_small_size(h, w, factor, &sh.nh, &sh.nw);
    if (sh.nh > h || sh.nw > w) return false;
    sh.lin_identity = (sh.nh == h && sh.nw == w) ? 1 : 0;
    sh.x2 = (w == 2 * sh.nw) ? 1 : 0;
    sh.xt = sh.yt = 1;
    sh.ix = sh.iy = 1;
    sh.inv_area = 1.0f;
    if (sh.lin_identity) {
        sh.area_mode = AREA_IDENTITY;
    } else if (w == 2 * sh.nw && h == 2 * sh.nh) {
        sh.area_mode = AREA_FAST2;
        sh.ix = sh.iy = 2;
    } else if (w % sh.nw == 0 && h % sh.nh == 0) {
        sh.area_mode = AREA_FASTN;
        sh.ix = w / sh.nw;
        sh.iy = h / sh.nh;
        sh.inv_area = (float)(1.0 / (sh.ix * sh.iy));
    } else {
        sh.area_mode = AREA_GENERAL;
        AreaAxis ax = build_area_axis(w, sh.nw);
        AreaAxis ay = build_area_axis(h, sh.nh);
        if (ax.taps > max_taps || ay.taps > max_taps) return false;
        sh.xt = ax.taps; sh.yt = ay.taps;
        sh.ax_first = blob_push(blob, ax.first);
        sh.ax_count = blob_push(blob, ax.count);
        sh.ax_alpha = blob_push(blob, ax.alpha);
        sh.ay_first = blob_push(blob, ay.first);
        sh.ay_count = blob_push(blob, ay.count);
        sh.ay_alpha = blob_push(blob, ay.alpha);
        if (ay.taps <= 3) {  // packed {first, beta0, beta1, beta2} per low-res row (unused taps are 0)
            std::vector<uint32_t> pk((size_t)sh.nh * 4, 0u);
            for (int d = 0; d < sh.nh; ++d) {
                pk[4 * d] = (uint32_t)ay.first[d];
                for (int q = 0; q < ay.count[d]; ++q) memcpy(&pk[4 * d + 1 + q], &ay.alpha[(size_t)d * ay.taps + q], 4);
            }
            sh.ay_pack = blob_push(blob, pk);
            sh.ay_packed = 1;
        }
    }
    if (!sh.lin_identity) {
        LinearAxis lx = build_linear_axis(sh.nw, w, true);
        LinearAxis ly = build_linear_axis(sh.nh, h, false);
        std::vector<uint32_t> ys(h);
        for (int y = 0; y < h; ++y) ys[y] = (uint32_t)ly.s0[y] | ((uint32_t)ly.s1[y] << 16);
        sh.lx_s0 = blob_push(blob, lx.s0);
        sh.lx_a = blob_push(blob, lx.coef);
        sh.ly_s = blob_push(blob, ys);
        sh.ly_b = blob_push(blob, ly.coef);
        // Row schedule of the kernels that loop over LOW-RES rows (lowres_x2h_kernel, lowres_x2i_kernel), one uint4 per
        // low-res row j: {beta0, beta1, beta2, r0 | nA << 16 | nB << 24}.  Once row j exists, the output rows whose lower
        // tap row is j leave: first the nA rows that blend (j-1, j), then the nB rows that blend (j, j) (top and bottom of
        // the image only); r0 is the first of them.  Requires the regular y taps first[j] = 2j, count[j] = taps.
        auto build_row_schedule = [&](int taps) -> bool {
            if (sh.hy_pack != 0) return true;
            if (sh.area_mode != AREA_GENERAL || !sh.ay_packed || h < taps) return false;
            const int32_t* yf = (const int32_t*)(blob.data() + sh.ay_first);
            const int32_t* yc = (const int32_t*)(blob.data() + sh.ay_count);
            for (int j = 0; j < sh.nh; ++j)
                if (yf[j] != 2 * j || yc[j] != taps || 2 * j + taps - 1 > h - 1) return false;
            std::vector<uint32_t> hp((size_t)sh.nh * 4, 0u);
            int r = 0;
            for (int j = 0; j < sh.nh; ++j) {
                const int r0 = r;
                int na = 0, nb = 0;
                while (r < h && ly.s1[r] == j && ly.s0[r] == j - 1) { ++na; ++r; }
                while (r < h && ly.s1[r] == j && ly.s0[r] == j) { ++nb; ++r; }
                if (na > 255 || nb > 255 || r0 > 65535) return false;
                const uint32_t* pk = blob.data() + sh.ay_pack + 4 * (size_t)j;
                hp[4 * j] = pk[1]; hp[4 * j + 1] = pk[2]; hp[4 * j + 2] = pk[3];
                hp[4 * j + 3] = (uint32_t)r0 | ((uint32_t)na << 16) | ((uint32_t)nb << 24);
            }
            if (r != h) return false;
            sh.hy_pack = blob_push(blob, hp);
            return true;
        };
        // odd widths at factor 0.5 (lowres_x2g_kernel): every low-res column has the three x taps 2dx, 2dx+1, 2dx+2; even
        // output pixels x blend low-res (x/2 - 1, x/2), odd ones ((x-1)/2, +1) or, from the slip column on, ((x-1)/2 - 1, +1)
        if (sh.area_mode == AREA_GENERAL && sh.ay_packed && sh.xt == 3 && w == 2 * sh.nw + 1 && sh.nw >= 1 && h >= 2) {
            const int32_t* xf = (const int32_t*)(blob.data() + sh.ax_first);
            const int32_t* xc = (const int32_t*)(blob.data() + sh.ax_count);
            bool ok = true;
            for (int dx = 0; dx < sh.nw && ok; ++dx) ok = (xf[dx] == 2 * dx && xc[dx] == 3);
            for (int x = 0; x < w && ok; ++x) {
                const int i = (x & 1) ? (x - 1) / 2 : x / 2 - 1;
                ok = (x & 1) ? (lx.s0[x] == i || (i >= 1 && lx.s0[x] == i - 1)) : (lx.s0[x] == std::max(i, 0));
            }
            if (ok) {
                std::vector<float> rc3((size_t)h * 4);
                for (int y = 0; y < h; ++y) {
                    const X2Row r = x2g_row_consts(ly.coef[y]);
                    rc3[4 * y] = r.c0s; rc3[4 * y + 1] = r.c1s; rc3[4 * y + 2] = r.k0; rc3[4 * y + 3] = r.k2;
                }
                sh.ly_rc3 = blob_push(blob, rc3);
                sh.x2g = 1;
                if (build_row_schedule(3)) sh.x2i = 1;
                else if (build_row_schedule(2)) sh.x2i = 2;
            }
        }
        if (sh.x2) {  // vertical-stage constants of the exact-2x kernels, one float4 per output row
            std::vector<float> rc((size_t)h * 4);
            for (int y = 0; y < h; ++y) {
                const X2Row r = x2_row_consts(ly.coef[y]);
                rc[4 * y] = r.c0s; rc[4 * y + 1] = r.c1s; rc[4 * y + 2] = r.k0; rc[4 * y + 3] = r.k2;
            }
            sh.ly_rc = blob_push(blob, rc);
            std::vector<uint32_t> rc2((size_t)h * 4);
            for (int y = 0; y < h; ++y) {
                const X2Row r = x2_row_consts(ly.coef[y]);
                const float k0p = r.k0 + 2.0f;
                memcpy(&rc2[4 * y], &r.c0s, 4); memcpy(&rc2[4 * y + 1], &r.c1s, 4); memcpy(&rc2[4 * y + 2], &k0p, 4);
                rc2[4 * y + 3] = x2_vertical_cfix(ly.coef[y]);
            }
            sh.ly_rc2 = blob_push(blob, rc2);
            sh.x2w = ((w & 3) == 0 && h >= 2 && (sh.area_mode == AREA_FAST2 || (sh.area_mode == AREA_GENERAL && sh.ay_packed))) ? 1 : 0;
            // packed-integer kernel: exact 2x in both axes; it derives the row pairs and the (1536, 512) / (512, 1536) y
            // coefficients from the row parity, so check that OpenCV's tables say the same
            bool packed = sh.x2w && sh.area_mode == AREA_FAST2;
            for (int y = 0; y < h && packed; ++y) {
                const int s0 = (y & 1) ? (y - 1) / 2 : std::max(y / 2 - 1, 0);
                const int s1 = (y & 1) ? std::min(s0 + 1, sh.nh - 1) : y / 2;
                const uint32_t coef = (y & 1) ? (1536u | (512u << 16)) : (512u | (1536u << 16));
                packed = (ly.s0[y] == s0 && ly.s1[y] == s1 && ly.coef[y] == coef);
            }
            sh.x2p = packed ? 1 : 0;
            // regular three-tap kernel (lowres_x2h_kernel): low-res row j reads source rows 2j, 2j+1, 2j+2 (every h = 2 nh + 1
            // up to ~2000), so row 2j+2 is shared with row j+1 and the source rows can be staged as fixed pairs
            if (sh.x2w && sh.area_mode == AREA_GENERAL && sh.ay_packed && build_row_schedule(3)) sh.x2h = 1;
        }
    }
    *out = sh;
    return true;
}

// Exact-2x shapes are processed in full-width strips (lowres_x2_kernel).  Pick the strip height that
// fills the 128-thread CTA best: items = (strip_rows / 8) * ceil(w / 8); fewer apron rows is better too.
// Sets sh->strip_rows / strip_half_rows (0 = use the generic tiled kernel) and returns the shared bytes.
inline size_t choose_strip_rows(DevShape* sh, const uint32_t* blob) {
    const size_t max_smem = 54 * 1024;  // 4 CTAs of 128 threads per SM (lowres_x2_kernel)
    const int nthreads = 128;
    sh->strip_rows = 0;
    sh->strip_half_rows = 0;
    if (!sh->x2 || sh->lin_identity) return 0;
    const size_t pitch = (size_t)((3 * sh->nw + 24 + 15) & ~15);
    const uint32_t* ly = blob + sh->ly_s;
    const int nchunks = (sh->w + 7) / 8;
    double best = -1.0;
    size_t best_smem = 0;
    for (int R = 16; R <= 64; R += 8) {
        int nj = 1;
        for (int y0 = 0; y0 < sh->h; y0 += R) {
            const int y1 = std::min(sh->h, y0 + R) - 1;
            nj = std::max(nj, (int)(ly[y1] >> 16) - (int)(ly[y0] & 0xFFFF) + 1);
        }
        const size_t smem = (size_t)nj * pitch;
        if (smem > max_smem) continue;
        const int rows = std::min(R, sh->h);
        const int items = ((rows + 7) / 8) * nchunks;
        const double fill = (double)items / (double)(((items + nthreads - 1) / nthreads) * nthreads);
        const double apron = (double)rows / (2.0 * nj);  // useful low-res rows / computed low-res rows (for 0.5x)
        const double score = fill * std::min(1.0, apron);
        if (score > best + 1e-9) { best = score; sh->strip_rows = R; sh->strip_half_rows = nj; best_smem = smem; }
    }
    return best_smem;
}

inline void build_strip_tiles(const std::vector<DevImage>& imgs, const std::vector<DevShape>& shapes, bool want_x2,
                              int th, int twb, std::vector<Tile>& tiles) {
    for (int i = 0; i < (int)imgs.size(); ++i) {
        const DevShape& sh = shapes[imgs[i].shape_id];
        const bool is_x2 = sh.strip_rows > 0;
        if (is_x2 != want_x2) continue;
        if (is_x2) {
            for (int y = 0; y < imgs[i].h; y += sh.strip_rows) tiles.push_back(Tile{i, y, 0, 0});
        } else {
            for (int y = 0; y < imgs[i].h; y += th)
                for (int b = 0; b < 3 * imgs[i].w; b += twb) tiles.push_back(Tile{i, y, b, 0});
        }
    }
}

// Ultralytics 8.3.x LetterBox geometry (auto=False, scaleup=True, center=True).
inline void letterbox_geometry(int h, int w, int out_h, int out_w, int* new_h, int* new_w, int* top, int* left) {
    double r = std::min((double)out_h / h, (double)out_w / w);
    // Python round(): half to even on the double
    *new_w = (int)nearbyint(w * r);
    *new_h = (int)nearbyint(h * r);
    double dw = (out_w - *new_w) / 2.0, dh = (out_h - *new_h) / 2.0;
    *top = (int)nearbyint(dh - 0.1);
    *left = (int)nearbyint(dw - 0.1);
}

// The 256-entry table of the Philox-mode table generator (rod_core.h): X[i] = round(128 sigma y_i) with
//   z_i = 256 (phi(q_i) - phi(q_i+1)), q_i = Phi^-1(i / 256)      mean of N(0, 1) over the i-th of 256 equiprobable cells
//   y_i = z_i (1 + A z_i^4 + B z_i^8) / sqrt(mean_j (z_j (1 + A z_j^4 + B z_j^8))^2)
// (A, B = ROD_GAUSS_H4_STRETCH_*: unit variance, 4th moment 3, 6th moment 15).  Antisymmetric by construction:
// X[255 - i] = -X[i] (the upper half is computed, the lower half mirrored), so the mean is exactly 0.
inline void build_gauss_table(float sigma, int32_t* X) {
    double y[256], q[257], ph[257];
    for (int i = 128; i <= 256; ++i) {
        q[i] = (i == 256) ? 0.0 : (i == 128 ? 0.0 : -ndtri_double((256 - i) / 256.0));
        ph[i] = (i == 256) ? 0.0 : exp(-0.5 * q[i] * q[i]) * 0.39894228040143267794;
    }
    double m2 = 0.0;
    for (int i = 128; i < 256; ++i) {
        const double z = 256.0 * (ph[i] - ph[i + 1]);
        const double z4 = (z * z) * (z * z);
        y[i] = z * (1.0 + ROD_GAUSS_H4_STRETCH_A * z4 + ROD_GAUSS_H4_STRETCH_B * (z4 * z4));
        m2 += y[i] * y[i];
    }
    const double norm = 128.0 * (double)sigma / sqrt(m2 / 128.0);
    for (int i = 128; i < 256; ++i) {
        X[i] = (int32_t)floor(norm * y[i] + 0.5);
        X[255 - i] = -X[i];
    }
}

inline void build_noise_tiles(const std::vector<DevImage>& imgs, int span, std::vector<Tile>& tiles) {
    for (int i = 0; i < (int)imgs.size(); ++i) {
        const DevImage& im = imgs[i];
        int64_t row = 3LL * im.w;
        if (im.contiguous) {
            int64_t n = row * im.h;
            for (int64_t e = 0; e < n; e += span)
                tiles.push_back(Tile{i, (int32_t)e, (int32_t)std::min<int64_t>(span, n - e), -1});
        } else {
            for (int y = 0; y < im.h; ++y)
                for (int64_t e = 0; e < row; e += span)
                    tiles.push_back(Tile{i, (int32_t)e, (int32_t)std::min<int64_t>(span, row - e), y});
        }
    }
}

inline void build_blur_tiles(const std::vector<DevImage>& imgs, int rows_per_tile, std::vector<Tile>& tiles) {
    for (int i = 0; i < (int)imgs.size(); ++i)
        for (int y = 0; y < imgs[i].h; y += rows_per_tile)
            tiles.push_back(Tile{i, y, std::min(rows_per_tile, imgs[i].h - y), 0});
}

// Tiles of th rows x twb BYTE columns (b = first byte column of the tile inside a row).
inline void build_grid_tiles(const std::vector<DevImage>& imgs, int th, int twb, std::vector<Tile>& tiles) {
    for (int i = 0; i < (int)imgs.size(); ++i)
        for (int y = 0; y < imgs[i].h; y += th)
            for (int b = 0; b < 3 * imgs[i].w; b += twb) tiles.push_back(Tile{i, y, b, 0});
}

// Worst-case low-res footprint (rows, pixel columns) and source-row footprint of one lowres tile of this shape.
inline void lowres_tile_footprint(const DevShape& sh, const uint32_t* blob, int th, int twb, int* rows, int* cols,
                                  int* src_rows = nullptr) {
    const int32_t* lx = (const int32_t*)(blob + sh.lx_s0);
    const uint32_t* ly = blob + sh.ly_s;
    const int32_t* yf = (const int32_t*)(blob + sh.ay_first);
    const int32_t* yc = (const int32_t*)(blob + sh.ay_count);
    int mr = 1, mc = 1, ms = 1;
    for (int y0 = 0; y0 < sh.h; y0 += th) {
        const int y1 = std::min(sh.h, y0 + th) - 1;
        const int j_lo = (int)(ly[y0] & 0xFFFF), j_hi = (int)(ly[y1] >> 16);
        mr = std::max(mr, j_hi - j_lo + 1);
        if (sh.area_mode == AREA_GENERAL) ms = std::max(ms, yf[j_hi] + yc[j_hi] - yf[j_lo]);
        else ms = std::max(ms, (j_hi - j_lo + 1) * sh.iy);
    }
    for (int b0 = 0; b0 < 3 * sh.w; b0 += twb) {
        const int x0 = b0 / 3, x1 = (std::min(3 * sh.w, b0 + twb) - 1) / 3;
        mc = std::max(mc, std::min(lx[x1] + 1, sh.nw - 1) - lx[x0] + 1);
    }
    *rows = mr;
    *cols = mc;
    if (src_rows) *src_rows = ms;
}

}  // namespace rod
