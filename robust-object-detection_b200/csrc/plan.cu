// plan.cu -- batch plans: descriptor upload, tile lists, resize tables (host side of librod_b200.so).
#include <map>
#include <new>

#include "rod_internal.h"
#include "rod_tables.h"

namespace rod {

thread_local int g_last_cuda_error = 0;

int grid_for(const rod_plan* plan, int n_tiles, int ctas_per_sm) {
    long long cap = (long long)plan->sm_count * ctas_per_sm;
    return (int)(n_tiles < cap ? n_tiles : cap);
}

// The device arrays of a plan come from the block cache (jpeg.cu) and go back to it: a batch driver builds and drops a plan
// per batch, and ~30 cudaMalloc / cudaFree calls per plan (each a device-wide synchronisation) cost more than its kernels.
static cudaError_t plan_alloc(const rod_plan* plan, void** p, size_t n) {
    const cudaError_t e = block_cache_alloc(plan->device, p, n);
    if (e == cudaSuccess) {
        std::lock_guard<std::mutex> lock(plan->cached_mutex);
        plan->cached_blocks.push_back({*p, n});
    }
    return e;
}
static void plan_free(const rod_plan* plan, void* p) {
    if (p == nullptr) return;
    {
        std::lock_guard<std::mutex> lock(plan->cached_mutex);
        for (size_t i = 0; i < plan->cached_blocks.size(); ++i)
            if (plan->cached_blocks[i].first == p) {
                block_cache_free(plan->device, p, plan->cached_blocks[i].second);
                plan->cached_blocks.erase(plan->cached_blocks.begin() + (long)i);
                return;
            }
    }
    cudaFree(p);   // allocated elsewhere (staging buffers of the host entry points)
}

template <typename T>
static int upload(const rod_plan* plan, const std::vector<T>& v, T** dptr) {
    *dptr = nullptr;
    if (v.empty()) return ROD_OK;
    ROD_CUDA(plan_alloc(plan, (void**)dptr, v.size() * sizeof(T)));
    ROD_CUDA(cudaMemcpy(*dptr, v.data(), v.size() * sizeof(T), cudaMemcpyHostToDevice));
    return ROD_OK;
}

// Replaces the device copy of `list` with `tiles` (in image order) and indexes it by image.
static int upload_tiles(const rod_plan* plan, const std::vector<Tile>& tiles, TileList* list) {
    plan_free(plan, list->d);
    list->d = nullptr;
    list->n = 0;
    list->start.assign(plan->n_images + 1, (int)tiles.size());
    for (int t = (int)tiles.size() - 1; t >= 0; --t) list->start[tiles[t].img] = t;
    for (int i = plan->n_images - 1; i >= 0; --i) list->start[i] = std::min(list->start[i], list->start[i + 1]);
    const int rc = upload(plan, tiles, &list->d);
    if (rc == ROD_OK) list->n = (int)tiles.size();
    return rc;
}

int ensure_lowres_tables(rod_plan* plan, double factor) {
    if (plan->d_shapes != nullptr && plan->lowres_factor == factor) return ROD_OK;
    if (!(factor > 0.0) || factor > 1.0) return ROD_ERR_UNSUPPORTED;
    std::vector<uint32_t> blob;
    std::vector<DevShape> shapes(plan->shapes.size());
    bool all_identity = true;
    int max_rows = 1, max_cols = 1, max_src_rows = 1;
    size_t x2_smem = 0;
    for (size_t s = 0; s < plan->shapes.size(); ++s) {
        const int h = plan->shapes[s].h, w = plan->shapes[s].w;
        if (!build_lowres_shape(h, w, factor, kMaxAreaTaps, blob, &shapes[s])) return ROD_ERR_UNSUPPORTED;
        DevShape& sh = shapes[s];
        if (sh.lin_identity) continue;
        all_identity = false;
        x2_smem = std::max(x2_smem, choose_strip_rows(&sh, blob.data()));
        if (sh.strip_rows > 0) continue;
        int rows, cols, srows;
        lowres_tile_footprint(sh, blob.data(), kLowresTH, kLowresTWB, &rows, &cols, &srows);
        max_rows = std::max(max_rows, rows);
        max_cols = std::max(max_cols, cols);
        max_src_rows = std::max(max_src_rows, srows);
    }
    if (blob.empty()) blob.push_back(0);
    // warp-marching kernel: one tile = (band of rows, strip of 30 chunks); band height from the amount of work
    // (aim at >= 4 tiles per resident warp; 16 warps per SM)
    auto march_image = [&](int i) {
        const DevImage& im = plan->h_images[i];
        return shapes[im.shape_id].x2w != 0 && (im.src_pitch & 3) == 0 && (im.src_off & 3) == 0;
    };
    auto al8_image = [&](int i) {
        const DevImage& im = plan->h_images[i];
        return (im.src_pitch & 7) == 0 && (im.src_off & 7) == 0 && (im.w & 7) == 0;
    };
    auto n_strips = [&](int w) { return ((w + 7) / 8 + 29) / 30; };
    int band_rows = 0;
    {
        long long strip_rows = 0;
        for (int i = 0; i < plan->n_images; ++i)
            if (march_image(i)) strip_rows += (long long)plan->h_images[i].h * n_strips(plan->h_images[i].w);
        band_rows = (int)(strip_rows / (80LL * plan->sm_count));  // ~5 tiles per resident warp (measured best on B200)
        band_rows = std::max(24, std::min(256, band_rows & ~7));  // <= kX2wMaxBandRows (per-warp shared tables)
    }
    // packed-integer kernel (exact 2x in both axes): additionally needs 4-byte aligned destination rows (32 / 64-bit stores)
    auto packed_image = [&](int i) {
        const DevImage& im = plan->h_images[i];
        return shapes[im.shape_id].x2p != 0 && (im.dst_pitch & 3) == 0 && (im.dst_off & 3) == 0;
    };
    auto packed_class = [&](int i) {  // 0: 16-byte copy units, 1: 8-byte, 2: 4-byte
        const DevImage& im = plan->h_images[i];
        const uint64_t a = (uint64_t)im.src_pitch | (uint64_t)im.dst_pitch | im.src_off | im.dst_off;
        if ((im.w & 15) == 0 && (a & 15) == 0) return 0;
        if ((im.w & 7) == 0 && (a & 7) == 0) return 1;
        return 2;
    };
    // float-tap staged kernel (exact-2x width, general y taps): 4-byte aligned destination rows, and a y scale small
    // enough for its ring of 8 source rows
    auto float_image = [&](int i) {
        const DevImage& im = plan->h_images[i];
        const DevShape& sh = shapes[im.shape_id];
        return sh.x2w != 0 && sh.area_mode == AREA_GENERAL && sh.ay_packed && (im.dst_pitch & 3) == 0 &&
               (im.dst_off & 3) == 0 && (sh.h <= 8 || 4LL * sh.h <= 9LL * sh.nh);
    };
    auto regular_image = [&](int i) { return float_image(i) && shapes[plan->h_images[i].shape_id].x2h != 0; };
    // odd-width staged kernel: regular 3-tap / one-slip shapes whose y scale fits the ring of 8 source rows
    auto odd_image = [&](int i) {
        const DevShape& sh = shapes[plan->h_images[i].shape_id];
        return sh.x2g != 0 && (sh.h <= 8 || 4LL * sh.h <= 9LL * sh.nh);
    };
    std::vector<Tile> lists[LR_NUM_LISTS], gen_all;
    build_strip_tiles(plan->h_images, shapes, false, kLowresTH, kLowresTWB, gen_all);
    for (const Tile& t : gen_all)
        if (!odd_image(t.img)) lists[LR_GENERIC].push_back(t);
    build_strip_tiles(plan->h_images, shapes, true, kLowresTH, kLowresTWB, lists[LR_X2_STRIP]);
    int band_rows_odd = 0;
    {
        long long strip_rows = 0;
        for (int i = 0; i < plan->n_images; ++i)
            if (odd_image(i)) strip_rows += (long long)plan->h_images[i].h * n_strips(plan->h_images[i].w);
        band_rows_odd = std::max(24, std::min(256, (int)(strip_rows / (60LL * plan->sm_count)) & ~7));  // ~60 tiles per SM
    }
    for (int i = 0; i < plan->n_images; ++i) {
        const DevShape& sh = shapes[plan->h_images[i].shape_id];
        if (odd_image(i)) {
            std::vector<Tile>& list = lists[sh.x2i != 0 ? LR_X2I_CARRY + sh.x2i - 1 : LR_X2G];
            for (int y = 0; y < plan->h_images[i].h; y += band_rows_odd)
                for (int st = 0; st < n_strips(plan->h_images[i].w); ++st)
                    list.push_back(Tile{i, y, std::min(plan->h_images[i].h, y + band_rows_odd), st});
            continue;
        }
        if (sh.strip_rows <= 0) continue;
        if (march_image(i)) {
            const int l = packed_image(i) ? LR_X2P16 + packed_class(i) : regular_image(i) ? LR_X2H16 + packed_class(i)
                          : float_image(i) ? LR_X2F16 + packed_class(i) : al8_image(i) ? LR_X2W8 : LR_X2W4;
            for (int y = 0; y < plan->h_images[i].h; y += band_rows)
                for (int st = 0; st < n_strips(plan->h_images[i].w); ++st)
                    lists[l].push_back(Tile{i, y, std::min(plan->h_images[i].h, y + band_rows), st});
        } else {
            for (int y = 0; y < plan->h_images[i].h; y += sh.strip_rows) lists[LR_X2_REST].push_back(Tile{i, y, 0, 0});
        }
    }
    plan->lowres_factor = -1.0;  // tables are incomplete until every upload below succeeded
    plan_free(plan, plan->d_shapes);
    plan_free(plan, plan->d_tab);
    plan->d_shapes = nullptr;
    plan->d_tab = nullptr;
    int rc = upload(plan, shapes, &plan->d_shapes);
    if (rc == ROD_OK) rc = upload(plan, blob, &plan->d_tab);
    for (int l = 0; l < LR_NUM_LISTS && rc == ROD_OK; ++l) rc = upload_tiles(plan, lists[l], &plan->lowres[l]);
    if (rc != ROD_OK) return rc;
    plan->lowres_x2_smem = x2_smem;
    plan->lowres_factor = factor;
    plan->lowres_all_identity = all_identity;
    plan->lowres_all_x2w = true;
    for (const DevShape& sh : shapes)
        if (!sh.lin_identity && !sh.x2w) plan->lowres_all_x2w = false;
    for (int i = 0; i < plan->n_images; ++i)  // 32-bit source loads in the fused kernel
        if ((plan->h_images[i].src_pitch & 3) != 0 || (plan->h_images[i].src_off & 3) != 0) plan->lowres_all_x2w = false;
    plan->lowres_half_rows = max_rows;
    plan->lowres_half_cols = max_cols;
    plan->lowres_src_rows = max_src_rows;
    return ROD_OK;
}

int ensure_letterbox_tables(rod_plan* plan, int out_h, int out_w) {
    if (plan->d_lb != nullptr && plan->lb_out_h == out_h && plan->lb_out_w == out_w) return ROD_OK;
    if (out_h < 1 || out_w < 1) return ROD_ERR_INVALID_ARG;
    std::vector<uint32_t> blob;
    std::vector<DevLetterbox> lbs(plan->shapes.size());
    for (size_t s = 0; s < plan->shapes.size(); ++s) {
        DevLetterbox g;
        memset(&g, 0, sizeof(g));
        g.h = plan->shapes[s].h; g.w = plan->shapes[s].w;
        letterbox_geometry(g.h, g.w, out_h, out_w, &g.new_h, &g.new_w, &g.top, &g.left);
        if (g.new_h < 1 || g.new_w < 1 || g.h > 65535 || g.w > 65535) return ROD_ERR_UNSUPPORTED;
        g.identity = (g.new_h == g.h && g.new_w == g.w);
        g.area2 = (!g.identity && g.h == 2 * g.new_h && g.w == 2 * g.new_w);
        if (!g.identity && !g.area2) {
            LinearAxis lx = build_linear_axis(g.w, g.new_w, true);
            LinearAxis ly = build_linear_axis(g.h, g.new_h, false);
            std::vector<uint32_t> ys(g.new_h);
            for (int y = 0; y < g.new_h; ++y) ys[y] = (uint32_t)ly.s0[y] | ((uint32_t)ly.s1[y] << 16);
            g.lx_s0 = blob_push(blob, lx.s0);
            g.lx_a = blob_push(blob, lx.coef);
            g.ly_s = blob_push(blob, ys);
            g.ly_b = blob_push(blob, ly.coef);
            std::vector<uint32_t> pack((size_t)2 * out_w);
            for (int X = 0; X < out_w; ++X) {
                const int cx = X - g.left;
                const bool in = cx >= 0 && cx < g.new_w;
                pack[2 * X] = in ? (uint32_t)(3 * lx.s0[cx]) : 0xFFFFFFFFu;
                pack[2 * X + 1] = in ? lx.coef[cx] : 0u;
            }
            g.lx_pack = blob_push(blob, pack);
            // The fused kernel's lane l resamples output columns 2l, 2l+1 (+64 per step) from six-byte windows that lie
            // 2 * 3 * (w / new_w) bytes apart.  If p lanes further the window is a multiple of 128 bytes away (within a word),
            // lanes l, l+p, l+2p, ... hit the same bank: the kernel then shifts every such group by one step.
            const double stride_words = 2.0 * 3.0 * ((double)g.w / (double)g.new_w) / 4.0;
            g.lane_group = 0;
            for (int pp = 2; pp <= 16; ++pp) {
                const double x = pp * stride_words / 32.0;
                if (fabs(x - nearbyint(x)) * 32.0 < 1.0) { g.lane_group = pp; break; }
            }
        }
        lbs[s] = g;
    }
    if (blob.empty()) blob.push_back(0);
    std::vector<Tile> tiles;
    for (int i = 0; i < plan->n_images; ++i)
        for (int y = 0; y < out_h; y += kLbTH)
            for (int x = 0; x < out_w; x += kLbTW) tiles.push_back(Tile{i, y, x, 0});
    if (plan->d_lb) { plan_free(plan, plan->d_lb); plan->d_lb = nullptr; }
    if (plan->d_lb_tab) { plan_free(plan, plan->d_lb_tab); plan->d_lb_tab = nullptr; }
    int rc = upload(plan, lbs, &plan->d_lb);
    if (rc != ROD_OK) return rc;
    rc = upload(plan, blob, &plan->d_lb_tab);
    if (rc != ROD_OK) return rc;
    rc = upload_tiles(plan, tiles, &plan->lb_tiles);
    if (rc != ROD_OK) return rc;
    plan->lb_all_linear = true;
    for (const DevLetterbox& g : lbs)
        if (g.identity || g.area2) plan->lb_all_linear = false;
    plan->lb_out_h = out_h;
    plan->lb_out_w = out_w;
    return ROD_OK;
}

int ensure_chw_tables(rod_plan* plan) {
    if (plan->d_chw_off != nullptr) return ROD_OK;
    std::vector<Tile> tiles;
    for (int i = 0; i < plan->n_images; ++i)
        for (int y = 0; y < plan->h_images[i].h; y += kChwBandRows)
            tiles.push_back(Tile{i, y, std::min(plan->h_images[i].h, y + kChwBandRows), 0});
    int rc = upload_tiles(plan, tiles, &plan->chw_tiles);
    uint64_t* off = nullptr;
    if (rc == ROD_OK) rc = upload(plan, plan->chw_off, &off);
    if (rc != ROD_OK) {
        plan_free(plan, off);
        return rc;
    }
    plan->d_chw_off = off;  // set last: it marks the tables complete
    return ROD_OK;
}

}  // namespace rod

using namespace rod;

extern "C" int rod_plan_create(const rod_image_desc* images, int n_images, rod_plan** out_plan) {
    if (out_plan == nullptr) return ROD_ERR_INVALID_ARG;
    *out_plan = nullptr;
    if (images == nullptr || n_images < 1) return ROD_ERR_INVALID_ARG;
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
        cudaGetLastError();
        return ROD_ERR_NO_DEVICE;
    }
    rod_plan* plan = new (std::nothrow) rod_plan();
    if (plan == nullptr) return ROD_ERR_OOM;
    cudaError_t e = cudaGetDevice(&plan->device);
    if (e == cudaSuccess) e = cudaDeviceGetAttribute(&plan->sm_count, cudaDevAttrMultiProcessorCount, plan->device);
    if (e != cudaSuccess) { delete plan; return cuda_fail(e); }
    plan->n_images = n_images;
    plan->descs.assign(images, images + n_images);
    plan->h_images.resize(n_images);
    std::map<std::pair<int, int>, int> shape_ids;
    uint64_t elem = 0;
    for (int i = 0; i < n_images; ++i) {
        const rod_image_desc& d = images[i];
        if (d.height < 1 || d.width < 1 || d.width > 65535 || d.height > 65535 || d.src_pitch < 3LL * d.width ||
            d.dst_pitch < 3LL * d.width || (uint64_t)d.height * d.width * 3 > 0x7FFFFFFFull) {
            delete plan;
            return ROD_ERR_INVALID_ARG;
        }
        DevImage& im = plan->h_images[i];
        im.src_off = d.src_offset; im.dst_off = d.dst_offset;
        im.src_pitch = d.src_pitch; im.dst_pitch = d.dst_pitch;
        im.h = d.height; im.w = d.width;
        im.elem_base = elem;
        im.contiguous = (d.src_pitch == 3LL * d.width && d.dst_pitch == 3LL * d.width) ? 1 : 0;
        elem += (uint64_t)d.height * d.width * 3;
        auto key = std::make_pair(d.height, d.width);
        auto it = shape_ids.find(key);
        if (it == shape_ids.end()) {
            it = shape_ids.emplace(key, (int)plan->shapes.size()).first;
            plan->shapes.push_back(HostShape{d.height, d.width});
        }
        im.shape_id = it->second;
        plan->max_w = std::max(plan->max_w, d.width);
        plan->all_contiguous = plan->all_contiguous && im.contiguous;
        plan->src_min_offset = (i == 0) ? d.src_offset : std::min<uint64_t>(plan->src_min_offset, d.src_offset);
        plan->src_extent = std::max<uint64_t>(plan->src_extent, d.src_offset + (uint64_t)(d.height - 1) * d.src_pitch + 3ull * d.width);
        plan->dst_extent = std::max<uint64_t>(plan->dst_extent, d.dst_offset + (uint64_t)(d.height - 1) * d.dst_pitch + 3ull * d.width);
    }
    plan->payload_bytes = elem;
    // CHW float32 output layout (include/rod_b200.h rod_plan_chw_offset): blocks of 3*H*W floats rounded up to 64 floats
    plan->chw_off.resize(n_images + 1);
    plan->chw_off[0] = 0;
    for (int i = 0; i < n_images; ++i)
        plan->chw_off[i + 1] = plan->chw_off[i] + (3ull * images[i].height * images[i].width + 63) / 64 * 64;
    std::vector<Tile> nt, bt;
    build_noise_tiles(plan->h_images, kNoiseSpan, nt);
    build_blur_tiles(plan->h_images, kBlurRowsPerTile, bt);
    for (int i = 1; i < n_images; ++i) {
        const rod_image_desc& a = images[i - 1];
        const rod_image_desc& b = images[i];
        if (b.src_offset < a.src_offset + (uint64_t)a.height * a.src_pitch - (a.src_pitch - 3ull * a.width) ||
            b.dst_offset < a.dst_offset + (uint64_t)a.height * a.dst_pitch - (a.dst_pitch - 3ull * a.width))
            plan->monotonic = false;
    }
    if (plan_alloc(plan, (void**)&plan->d_counters, kCounterRing * sizeof(unsigned int)) != cudaSuccess) { rod_plan_destroy(plan); return ROD_ERR_OOM; }
    if (plan_alloc(plan, (void**)&plan->d_blur_counters, 2 * kCounterRing * sizeof(unsigned int)) != cudaSuccess) { rod_plan_destroy(plan); return ROD_ERR_OOM; }
    // block-cache memory comes back recycled: zero the blur pairs once, done before the plan is handed out
    e = cudaMemset(plan->d_blur_counters, 0, 2 * kCounterRing * sizeof(unsigned int));
    if (e == cudaSuccess) e = cudaStreamSynchronize(0);
    if (e != cudaSuccess) { rod_plan_destroy(plan); return cuda_fail(e); }
    int rc = upload(plan, plan->h_images, &plan->d_images);
    if (rc == ROD_OK) rc = upload_tiles(plan, nt, &plan->noise_tiles);
    if (rc == ROD_OK) rc = upload_tiles(plan, bt, &plan->blur_tiles);
    if (rc != ROD_OK) { rod_plan_destroy(plan); return rc; }
    *out_plan = plan;
    return ROD_OK;
}

// Installs (kernel != NULL) or removes (NULL) a general k x k float32 blur kernel: while installed, ROD_OP_BLUR runs
// the 2-D filter (filter2d.cu) instead of the horizontal box.
extern "C" int rod_set_blur_kernel(rod_plan* plan, const float* kernel, int k) {
    if (plan == nullptr) return ROD_ERR_INVALID_ARG;
    if (kernel == nullptr) {
        plan->f2d_ntaps = 0;
        plan->f2d_k = 0;
        return ROD_OK;
    }
    if (k < 1 || (k & 1) == 0) return ROD_ERR_INVALID_ARG;
    if (k * k >= kF2dMaxElems) return ROD_ERR_UNSUPPORTED;  // OpenCV's DFT path: not reproducible bit-exactly
    std::vector<float4> taps;
    for (int dy = 0; dy < k; ++dy)
        for (int dx = 0; dx < k; ++dx) {
            const float w = kernel[dy * k + dx];
            if (w == 0.0f) continue;
            float4 t;
            const int dxb = 3 * dx;
            memcpy(&t.x, &dy, 4);
            memcpy(&t.y, &dxb, 4);
            t.z = w;
            t.w = 0.f;
            taps.push_back(t);
        }
    if (taps.empty()) return ROD_ERR_INVALID_ARG;
    if (plan->d_f2d_taps) { plan_free(plan, plan->d_f2d_taps); plan->d_f2d_taps = nullptr; }
    int rc = upload(plan, taps, &plan->d_f2d_taps);
    if (rc != ROD_OK) return rc;
    if (plan->f2d_tiles.d == nullptr) {
        std::vector<Tile> tiles;
        build_grid_tiles(plan->h_images, kF2dTH, kF2dTWB, tiles);
        rc = upload_tiles(plan, tiles, &plan->f2d_tiles);
        if (rc != ROD_OK) return rc;
    }
    plan->f2d_ntaps = (int)taps.size();
    plan->f2d_k = k;
    return ROD_OK;
}

extern "C" void rod_plan_destroy(rod_plan* plan) {
    if (plan == nullptr) return;
    if (plan->inner) rod_plan_destroy(plan->inner);
    // the arrays go back to a cache and may be handed to the next plan at once: kernels of this plan that are still running
    // must be done first (what the implicit synchronisation of cudaFree used to guarantee, once instead of thirty times)
    cudaDeviceSynchronize();
    if (plan->d_patch_clean) cudaFree(plan->d_patch_clean);
    if (plan->d_patch_corrupted) cudaFree(plan->d_patch_corrupted);
    void* ptrs[] = {plan->d_images, plan->noise_tiles.d, plan->blur_tiles.d, plan->d_shapes, plan->d_tab, plan->d_lb,
                    plan->d_lb_tab, plan->lb_tiles.d, plan->d_scratch, plan->d_stage_src, plan->d_f2d_taps,
                    plan->f2d_tiles.d, plan->d_counters, plan->d_blur_counters, plan->d_stage_dst, plan->d_stage_noise, plan->d_stage_ops,
                    plan->chw_tiles.d, plan->d_chw_off};
    for (void* p : ptrs) plan_free(plan, p);
    for (const TileList& l : plan->lowres) plan_free(plan, l.d);
    for (cudaStream_t s : plan->streams)
        if (s) cudaStreamDestroy(s);
    for (cudaStream_t s : plan->aux_streams)
        if (s) cudaStreamDestroy(s);
    for (cudaStream_t s : plan->lr_streams)
        if (s) cudaStreamDestroy(s);
    if (plan->lr_ev_fork) cudaEventDestroy(plan->lr_ev_fork);
    for (cudaEvent_t e : plan->lr_ev_join)
        if (e) cudaEventDestroy(e);
    if (plan->ev_fork) cudaEventDestroy(plan->ev_fork);
    for (cudaEvent_t e : plan->ev_join)
        if (e) cudaEventDestroy(e);
    delete plan;
}

extern "C" int rod_plan_num_images(const rod_plan* plan) { return plan ? plan->n_images : 0; }
extern "C" uint64_t rod_plan_payload_bytes(const rod_plan* plan) { return plan ? plan->payload_bytes : 0; }
extern "C" uint64_t rod_plan_chw_offset(const rod_plan* plan, int i) {
    return (plan != nullptr && i >= 0 && i <= plan->n_images) ? plan->chw_off[i] : 0;
}
