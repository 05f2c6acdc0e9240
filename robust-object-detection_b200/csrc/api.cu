// api.cu -- extern "C" entry points of librod_b200.so (declared in include/rod_b200.h).
#include <algorithm>
#include <vector>

#include "rod_internal.h"
#include "rod_tables.h"

using namespace rod;

namespace {

constexpr float kPhiloxMaxSigma = 2048.0f;  // floor(K s) must fit int16 (rod_core.h noise_floor16)

bool blur_supported(int k, double angle) { return angle == 0.0 && k >= 1 && k <= 31 && (k & 1) == 1; }

int run_op(rod_plan* plan, int op, const uint8_t* src, uint8_t* dst, const float* noise, float sigma, int k,
           double factor, uint64_t seed, uint64_t first_image, uint32_t offset, const uint8_t* opcodes,
           cudaStream_t stream, int img_lo, int img_hi) {
    switch (op) {
        case ROD_OP_NONE:
            return launch_noise(plan, NOISE_COPY, src, dst, nullptr, nullptr, 0.f, 0, 0, 0, opcodes, ROD_OP_NONE,
                                stream, img_lo, img_hi);
        case ROD_OP_NOISE:
            if (noise == nullptr && sigma > kPhiloxMaxSigma) return ROD_ERR_UNSUPPORTED;
            return launch_noise(plan, noise ? NOISE_COMPAT : NOISE_PHILOX, src, dst, noise, nullptr, sigma, seed,
                                first_image, offset, opcodes, ROD_OP_NOISE, stream, img_lo, img_hi);
        case ROD_OP_BLUR:
            if (plan->f2d_ntaps > 0) return launch_filter2d(plan, src, dst, opcodes, stream, img_lo, img_hi);
            if (!blur_supported(k, 0.0)) return ROD_ERR_UNSUPPORTED;
            if (k == 1)
                return launch_noise(plan, NOISE_COPY, src, dst, nullptr, nullptr, 0.f, 0, 0, 0, opcodes, ROD_OP_BLUR,
                                    stream, img_lo, img_hi);
            return launch_blur(plan, src, dst, k, opcodes, stream, img_lo, img_hi);
        case ROD_OP_LOWRES: {
            int rc = ensure_lowres_tables(plan, factor);
            if (rc != ROD_OK) return rc;
            if (plan->lowres_all_identity)
                return launch_noise(plan, NOISE_COPY, src, dst, nullptr, nullptr, 0.f, 0, 0, 0, opcodes,
                                    ROD_OP_LOWRES, stream, img_lo, img_hi);
            return launch_lowres(plan, src, dst, opcodes, stream, img_lo, img_hi);
        }
        default:
            return ROD_ERR_INVALID_ARG;
    }
}

// The kernels of ops [op_lo, ROD_OP_LOWRES] of a mixed batch.  Each touches only the images of its own op-code, so
// they are independent: for small batches (no single op fills the GPU) they run concurrently on two auxiliary
// streams forked from / joined into `stream` with events (graph-capturable).
int run_mixed_ops(rod_plan* plan, int op_lo, const uint8_t* src, uint8_t* dst, const uint8_t* opcodes, const float* noise,
                  float sigma, int k, double factor, uint64_t seed, uint64_t first_image, uint32_t offset,
                  cudaStream_t stream) {
    // validate every op's parameters BEFORE anything is launched or forked: an unsupported k / factor / sigma must not
    // leave the auxiliary streams un-joined (stream capture, ordering) or dst half written
    if (noise == nullptr && sigma > kPhiloxMaxSigma) return ROD_ERR_UNSUPPORTED;
    if (plan->f2d_ntaps == 0 && !blur_supported(k, 0.0)) return ROD_ERR_UNSUPPORTED;
    {
        const int rc = ensure_lowres_tables(plan, factor);
        if (rc != ROD_OK) return rc;
    }
    const bool fork = plan->n_images <= 128;
    if (fork && plan->ev_fork == nullptr) {  // created as a whole or not at all (a failed creation is retried next call)
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
        plan->aux_streams[0] = s2[0]; plan->aux_streams[1] = s2[1];
        plan->ev_join[0] = ej[0]; plan->ev_join[1] = ej[1];
        plan->ev_fork = ef;
    }
    if (fork) {
        ROD_CUDA(cudaEventRecord(plan->ev_fork, stream));
        for (auto& s : plan->aux_streams) ROD_CUDA(cudaStreamWaitEvent(s, plan->ev_fork, 0));
    }
    int first_rc = ROD_OK;
    for (int op = op_lo; op <= ROD_OP_LOWRES && first_rc == ROD_OK; ++op) {
        // lowres (the longest) stays on the caller's stream; blur and noise go to the auxiliary streams
        cudaStream_t st = stream;
        if (fork && op == ROD_OP_BLUR) st = plan->aux_streams[0];
        if (fork && op == ROD_OP_NOISE) st = plan->aux_streams[1];
        first_rc = run_op(plan, op, src, dst, noise, sigma, k, factor, seed, first_image, offset, opcodes, st, 0, plan->n_images);
    }
    if (fork) {  // the join is executed on every path, also after a failed launch
        for (int i = 0; i < 2; ++i) {
            cudaError_t e = cudaEventRecord(plan->ev_join[i], plan->aux_streams[i]);
            if (e == cudaSuccess) e = cudaStreamWaitEvent(stream, plan->ev_join[i], 0);
            if (e != cudaSuccess && first_rc == ROD_OK) first_rc = cuda_fail(e);
        }
    }
    return first_rc;
}

// The plan's scratch: corrupted images at the dst descriptors, read by the letterbox and CHW kernels.
int ensure_scratch(rod_plan* plan) {
    if (plan->d_scratch == nullptr || plan->scratch_bytes < plan->dst_extent) {
        if (plan->d_scratch) cudaFree(plan->d_scratch);
        plan->d_scratch = nullptr;
        ROD_CUDA(cudaMalloc((void**)&plan->d_scratch, plan->dst_extent + 64));
        plan->scratch_bytes = plan->dst_extent;
    }
    return ROD_OK;
}

}  // namespace

extern "C" const char* rod_version(void) { return "rod_b200 0.1.0 (sm_100a)"; }

extern "C" int rod_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) {
        cudaGetLastError();
        return 0;
    }
    return n;
}

extern "C" int rod_last_cuda_error(void) { return g_last_cuda_error; }

extern "C" const char* rod_status_string(int status) {
    switch (status) {
        case ROD_OK: return "ok";
        case ROD_ERR_INVALID_ARG: return "invalid argument";
        case ROD_ERR_UNSUPPORTED: return "parameter outside the exact-parity domain (no approximation, no CPU fallback)";
        case ROD_ERR_CUDA: return "CUDA error";
        case ROD_ERR_NO_DEVICE: return "no CUDA device (there is no CPU fallback)";
        case ROD_ERR_OOM: return "out of memory";
        default: return "unknown status";
    }
}

extern "C" int rod_plan_launches(const rod_plan* plan, int op) {
    if (plan == nullptr) return 0;
    switch (op) {
        case ROD_OP_NONE: case ROD_OP_NOISE: case ROD_OP_BLUR: return 1;
        case ROD_OP_LOWRES: {  // one launch per non-empty tile list (known once the resize tables exist)
            if (plan->d_shapes == nullptr) return 1;
            // except the full strip list: it runs only when the source base (or, with staged lists, the destination base)
            // is not 4-byte aligned, in place of the band lists and X2_REST; such a call launches fewer kernels
            int n = 0;
            for (int l = 0; l < LR_NUM_LISTS; ++l) n += l != LR_X2_STRIP && plan->lowres[l].n > 0;
            return n > 0 ? n : 1;
        }
        case 100: return 4;  // rod_corrupt_batch_u8: copy + noise + blur + lowres
        case 101: return 4;  // rod_corrupt_letterbox_f16: noise + blur + lowres + letterbox (clean images are read in place)
        case 102: return 4;  // rod_corrupt_chw_f32: noise + blur + lowres + conversion (clean images are read in place)
        default: return 0;
    }
}

extern "C" int rod_noise_u8(const rod_plan* plan, const uint8_t* src, uint8_t* dst, const float* noise, float sigma,
                            uint64_t seed, uint64_t first_image_index, uint32_t offset, const uint8_t* opcodes,
                            void* stream) {
    if (plan == nullptr || src == nullptr || dst == nullptr) return ROD_ERR_INVALID_ARG;
    if (!(sigma >= 0.0f)) return ROD_ERR_INVALID_ARG;
    if (noise == nullptr && sigma > kPhiloxMaxSigma) return ROD_ERR_UNSUPPORTED;
    return launch_noise(plan, noise ? NOISE_COMPAT : NOISE_PHILOX, src, dst, noise, nullptr, sigma, seed,
                        first_image_index, offset, opcodes, ROD_OP_NOISE, (cudaStream_t)stream, 0, plan->n_images);
}

extern "C" int rod_noise_prewarm(int device, float sigma) {
    if (!(sigma >= ROD_GAUSS_TABLE_MIN_SIGMA && sigma <= ROD_GAUSS_TABLE_MAX_SIGMA)) return ROD_OK;
    int prev = 0;
    ROD_CUDA(cudaGetDevice(&prev));
    ROD_CUDA(cudaSetDevice(device));
    const int32_t* t = nullptr;
    const int rc = rod::gauss_table_for(device, sigma, &t);
    cudaSetDevice(prev);
    return rc;
}

extern "C" int rod_gauss_table_i32(float sigma, int32_t* out256) {
    if (out256 == nullptr || !(sigma >= ROD_GAUSS_TABLE_MIN_SIGMA && sigma <= ROD_GAUSS_TABLE_MAX_SIGMA)) return ROD_ERR_INVALID_ARG;
    rod::build_gauss_table(sigma, out256);
    return ROD_OK;
}

extern "C" int rod_plan_set_gaussian_generator(rod_plan* plan, int generator) {
    if (plan == nullptr || (generator != ROD_GAUSS_AUTO && generator != ROD_GAUSS_BOXMULLER && generator != ROD_GAUSS_TABLE_PHILOX7)) return ROD_ERR_INVALID_ARG;
    plan->gauss_generator = generator;
    if (plan->inner != nullptr) plan->inner->gauss_generator = generator;
    return ROD_OK;
}

extern "C" int rod_noise_field_f32(const rod_plan* plan, float* out_field, float sigma, uint64_t seed,
                                   uint64_t first_image_index, uint32_t offset, void* stream) {
    if (plan == nullptr || out_field == nullptr) return ROD_ERR_INVALID_ARG;
    if (!(sigma >= 0.0f) || sigma > kPhiloxMaxSigma) return ROD_ERR_UNSUPPORTED;
    return launch_noise(plan, NOISE_FIELD, nullptr, nullptr, nullptr, out_field, sigma, seed, first_image_index,
                        offset, nullptr, ROD_OP_NOISE, (cudaStream_t)stream, 0, plan->n_images);
}

extern "C" int rod_blur_h_u8(const rod_plan* plan, const uint8_t* src, uint8_t* dst, int k, double angle_deg,
                             const uint8_t* opcodes, void* stream) {
    if (plan == nullptr || src == nullptr || dst == nullptr) return ROD_ERR_INVALID_ARG;
    // a general angle needs its rotated kernel installed with rod_set_blur_kernel (then k must match it)
    if (plan->f2d_ntaps > 0 ? (k != plan->f2d_k) : !blur_supported(k, angle_deg)) return ROD_ERR_UNSUPPORTED;
    return run_op(const_cast<rod_plan*>(plan), ROD_OP_BLUR, src, dst, nullptr, 0.f, k, 0.0, 0, 0, 0, opcodes,
                  (cudaStream_t)stream, 0, plan->n_images);
}

extern "C" int rod_lowres_u8(rod_plan* plan, const uint8_t* src, uint8_t* dst, double factor, const uint8_t* opcodes,
                             void* stream) {
    if (plan == nullptr || src == nullptr || dst == nullptr) return ROD_ERR_INVALID_ARG;
    return run_op(plan, ROD_OP_LOWRES, src, dst, nullptr, 0.f, 0, factor, 0, 0, 0, opcodes, (cudaStream_t)stream, 0,
                  plan->n_images);
}

extern "C" int rod_corrupt_batch_u8(rod_plan* plan, const uint8_t* src, uint8_t* dst, const uint8_t* opcodes,
                                    const float* noise, float sigma, int k, double factor, uint64_t seed,
                                    uint64_t first_image_index, uint32_t offset, void* stream) {
    if (plan == nullptr || src == nullptr || dst == nullptr || opcodes == nullptr) return ROD_ERR_INVALID_ARG;
    // parameters are validated before the first launch (run_mixed_ops repeats the check for its other callers)
    if (noise == nullptr && sigma > kPhiloxMaxSigma) return ROD_ERR_UNSUPPORTED;
    if (plan->f2d_ntaps == 0 && !blur_supported(k, 0.0)) return ROD_ERR_UNSUPPORTED;
    int rc = ensure_lowres_tables(plan, factor);
    if (rc != ROD_OK) return rc;
    rc = run_op(plan, ROD_OP_NONE, src, dst, noise, sigma, k, factor, seed, first_image_index, offset, opcodes,
                (cudaStream_t)stream, 0, plan->n_images);
    if (rc != ROD_OK) return rc;
    return run_mixed_ops(plan, ROD_OP_NOISE, src, dst, opcodes, noise, sigma, k, factor, seed, first_image_index, offset,
                         (cudaStream_t)stream);
}

extern "C" int rod_corrupt_letterbox_f16(rod_plan* plan, const uint8_t* src, const uint8_t* opcodes, void* out_f16,
                                         int out_h, int out_w, int pad_value, const float* noise, float sigma, int k,
                                         double factor, uint64_t seed, uint64_t first_image_index, uint32_t offset,
                                         void* stream) {
    if (plan == nullptr || src == nullptr || out_f16 == nullptr || opcodes == nullptr) return ROD_ERR_INVALID_ARG;
    if (pad_value < 0 || pad_value > 255) return ROD_ERR_INVALID_ARG;
    // The training path always uses the Box-Muller generator: the fused kernel spends its shared memory on row
    // buffers (no room for the 64 KB table), and the unfused fallback must produce the same bytes as the fused kernel.
    struct GeneratorScope {
        rod_plan* p; int saved;
        explicit GeneratorScope(rod_plan* pl) : p(pl), saved(pl->gauss_generator) { p->gauss_generator = ROD_GAUSS_BOXMULLER; }
        ~GeneratorScope() { p->gauss_generator = saved; }
    } generator_scope(plan);
    int rc = ensure_letterbox_tables(plan, out_h, out_w);
    if (rc != ROD_OK) return rc;
    rc = ensure_scratch(plan);
    if (rc != ROD_OK) return rc;
    // Fused path: noise / blur / clean rows are produced inside the letterbox kernel (no full-resolution round trip);
    // only LowRes images go through the scratch.  Needs an even output width (two columns per lane, half2 stores), plain
    // linear letterboxes, the angle-0 blur and Philox sigma in range.
    const bool fused = (out_w & 1) == 0 && plan->lb_all_linear && plan->f2d_ntaps == 0 && blur_supported(k, 0.0) &&
                       k >= 3 && (noise != nullptr || sigma <= kPhiloxMaxSigma);
    if (fused) {
        rc = ensure_lowres_tables(plan, factor);
        if (rc != ROD_OK) return rc;
        // LowRes rows are produced inside the kernel as well when every shape is exact-2x (w % 4 == 0, 4-byte aligned
        // rows); otherwise the resize kernels write the LowRes images to the scratch first
        const bool in_kernel = plan->lowres_all_x2w && (((uintptr_t)src) & 3) == 0;
        if (!in_kernel) {
            rc = run_op(plan, ROD_OP_LOWRES, src, plan->d_scratch, noise, sigma, k, factor, seed, first_image_index, offset,
                        opcodes, (cudaStream_t)stream, 0, plan->n_images);
            if (rc != ROD_OK) return rc;
        }
        rc = launch_fused_letterbox(plan, src, plan->d_scratch, opcodes, noise, out_f16, pad_value, sigma, k, seed,
                                    first_image_index, offset, in_kernel, (cudaStream_t)stream);
        if (rc != ROD_ERR_UNSUPPORTED) return rc;  // rows too wide for the per-warp buffers: unfused path below
    }
    // images that stay clean are read from `src` by the letterbox kernel itself: no copy into the scratch
    rc = run_mixed_ops(plan, ROD_OP_NOISE, src, plan->d_scratch, opcodes, noise, sigma, k, factor, seed, first_image_index,
                       offset, (cudaStream_t)stream);
    if (rc != ROD_OK) return rc;
    return launch_letterbox(plan, plan->d_scratch, src, opcodes, out_f16, pad_value, (cudaStream_t)stream);
}

// train_frcnn_augmented.py:61-67: RandomCorruption(0.5) + ToImage + ToDtype(float32, scale=True) for a batch.
extern "C" int rod_corrupt_chw_f32(rod_plan* plan, const uint8_t* src, const uint8_t* opcodes, float* out, const float* noise,
                                   float sigma, int k, double factor, uint64_t seed, uint64_t first_image_index,
                                   uint32_t offset, void* stream) {
    if (plan == nullptr || src == nullptr || out == nullptr || opcodes == nullptr) return ROD_ERR_INVALID_ARG;
    if (((uintptr_t)out & 255) != 0) return ROD_ERR_INVALID_ARG;  // the layout's 256-byte alignment starts at `out`
    // the checks of rod_corrupt_batch_u8, before anything is launched
    if (noise == nullptr && sigma > kPhiloxMaxSigma) return ROD_ERR_UNSUPPORTED;
    if (plan->f2d_ntaps == 0 && !blur_supported(k, 0.0)) return ROD_ERR_UNSUPPORTED;
    int rc = ensure_lowres_tables(plan, factor);
    if (rc == ROD_OK) rc = ensure_chw_tables(plan);
    if (rc == ROD_OK) rc = ensure_scratch(plan);
    if (rc != ROD_OK) return rc;
    // corrupted images go to the scratch; clean ones are read from `src` by the conversion itself
    rc = run_mixed_ops(plan, ROD_OP_NOISE, src, plan->d_scratch, opcodes, noise, sigma, k, factor, seed, first_image_index,
                       offset, (cudaStream_t)stream);
    if (rc != ROD_OK) return rc;
    return launch_chw_f32(plan, src, plan->d_scratch, opcodes, out, (cudaStream_t)stream);
}

extern "C" int rod_resize_linear_u8(const uint8_t* src, int h, int w, int64_t src_pitch, uint8_t* dst, int nh, int nw,
                                    int64_t dst_pitch, void* stream) {
    if (src == nullptr || dst == nullptr || h < 1 || w < 1 || nh < 1 || nw < 1 || src_pitch < 3LL * w || dst_pitch < 3LL * nw ||
        h > 65535 || w > 65535 || nh > 65535 || nw > 65535)
        return ROD_ERR_INVALID_ARG;
    if (nh < h || nw < w) return ROD_ERR_UNSUPPORTED;  // reductions: OpenCV may switch to INTER_AREA (exact 2x); not this entry point
    return launch_resize_linear(src, h, w, src_pitch, dst, nh, nw, dst_pitch, (cudaStream_t)stream);
}

// SURVEY 8f rank 4: RestorationDataset.__getitem__ (train_restoration.py:104-129) for a batch of patches.
extern "C" int rod_restoration_pairs_f32(rod_plan* plan, const uint8_t* src, const uint8_t* flips, const uint8_t* opcodes,
                                         float* corrupted_out, float* clean_out, const float* noise, float sigma, int k,
                                         double factor, uint64_t seed, uint64_t first_image_index, uint32_t offset,
                                         void* stream) {
    if (plan == nullptr || src == nullptr || opcodes == nullptr || corrupted_out == nullptr || clean_out == nullptr)
        return ROD_ERR_INVALID_ARG;
    const int n = plan->n_images;
    for (int i = 1; i < n; ++i)  // one patch size per batch: the outputs are dense [N,3,P,P] tensors
        if (plan->descs[i].height != plan->descs[0].height || plan->descs[i].width != plan->descs[0].width)
            return ROD_ERR_INVALID_ARG;
    if (plan->inner == nullptr) {  // built as a whole or not at all: nothing is committed to the plan until every piece exists
        std::vector<rod_image_desc> d(n);
        const uint64_t bytes = 3ull * plan->descs[0].height * plan->descs[0].width;
        const uint64_t stride = (bytes + 255) / 256 * 256;
        for (int i = 0; i < n; ++i) {
            d[i].src_offset = d[i].dst_offset = i * stride;
            d[i].height = plan->descs[0].height;
            d[i].width = plan->descs[0].width;
            d[i].src_pitch = d[i].dst_pitch = 3ll * d[i].width;
        }
        rod_plan* inner = nullptr;
        int rc = rod_plan_create(d.data(), n, &inner);
        if (rc != ROD_OK) return rc;
        uint8_t *pc = nullptr, *pp = nullptr;
        cudaError_t e = cudaMalloc((void**)&pc, n * stride + 64);
        if (e == cudaSuccess) e = cudaMalloc((void**)&pp, n * stride + 64);
        if (e != cudaSuccess) {
            if (pc) cudaFree(pc);
            rod_plan_destroy(inner);
            return cuda_fail(e);
        }
        inner->gauss_generator = plan->gauss_generator;
        plan->d_patch_clean = pc;
        plan->d_patch_corrupted = pp;
        plan->inner = inner;
    }
    cudaStream_t st = (cudaStream_t)stream;
    int rc = launch_gather_patches(plan, plan->inner, src, plan->d_patch_clean, flips, st);
    if (rc != ROD_OK) return rc;
    rc = rod_corrupt_batch_u8(plan->inner, plan->d_patch_clean, plan->d_patch_corrupted, opcodes, noise, sigma, k, factor,
                              seed, first_image_index, offset, stream);
    if (rc != ROD_OK) return rc;
    return launch_format_pairs(plan->inner, plan->d_patch_clean, plan->d_patch_corrupted, clean_out, corrupted_out, st);
}

// Host-buffer path: chunks of images are pipelined over three streams so the H2D copy of chunk
// c+1, the kernel of chunk c and the D2H copy of chunk c-1 overlap.
extern "C" int rod_apply_host(rod_plan* plan, int op, const uint8_t* src_host, uint8_t* dst_host,
                              const float* noise_host, float sigma, int k, double factor, uint64_t seed,
                              uint64_t first_image_index, uint32_t offset) {
    if (plan == nullptr || src_host == nullptr || dst_host == nullptr) return ROD_ERR_INVALID_ARG;
    if (op < ROD_OP_NONE || op > ROD_OP_LOWRES) return ROD_ERR_INVALID_ARG;
    if (op == ROD_OP_BLUR && plan->f2d_ntaps == 0 && !blur_supported(k, 0.0)) return ROD_ERR_UNSUPPORTED;
    if (op == ROD_OP_LOWRES) {
        int rc = ensure_lowres_tables(plan, factor);
        if (rc != ROD_OK) return rc;
    }
    if (plan->d_stage_dst == nullptr) {  // staging buffers + streams: committed to the plan only when all of them exist
        uint8_t *ss = nullptr, *sd = nullptr;
        cudaStream_t st3[3] = {nullptr, nullptr, nullptr};
        cudaError_t e = cudaMalloc((void**)&ss, plan->src_extent + 64);
        if (e == cudaSuccess) e = cudaMalloc((void**)&sd, plan->dst_extent + 64);
        for (auto& s : st3)
            if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&s, cudaStreamNonBlocking);
        if (e != cudaSuccess) {
            if (ss) cudaFree(ss);
            if (sd) cudaFree(sd);
            for (auto& s : st3) if (s) cudaStreamDestroy(s);
            return cuda_fail(e);
        }
        plan->d_stage_src = ss;
        for (int i = 0; i < 3; ++i) plan->streams[i] = st3[i];
        plan->d_stage_dst = sd;
    }
    const bool compat = (op == ROD_OP_NOISE && noise_host != nullptr);
    if (compat && plan->d_stage_noise == nullptr)
        ROD_CUDA(cudaMalloc((void**)&plan->d_stage_noise, plan->payload_bytes * sizeof(float) + 64));

    // chunking: ~16 MiB of payload per chunk when the layout allows per-chunk byte ranges
    // (measured e2e on a B200 box: 16 MiB 13.9 k img/s, 32: 13.6, 64: 13.7, 128: 13.3)
    const uint64_t chunk_bytes = 16ull << 20;
    const int n = plan->n_images;
    std::vector<int> cuts{0};
    if (plan->monotonic && n > 1) {
        uint64_t acc = 0;
        for (int i = 0; i < n; ++i) {
            acc += 3ull * plan->descs[i].height * plan->descs[i].width;
            if (acc >= chunk_bytes && i + 1 < n) { cuts.push_back(i + 1); acc = 0; }
        }
    }
    cuts.push_back(n);
    bool dst_packed = plan->monotonic;
    for (int i = 0; i < n && dst_packed; ++i) {
        const rod_image_desc& d = plan->descs[i];
        if (d.dst_pitch != 3ll * d.width) dst_packed = false;
        if (i + 1 < n && plan->descs[i + 1].dst_offset != d.dst_offset + 3ull * d.width * d.height) dst_packed = false;
    }
    // every CUDA call below records its error and falls through to the stream synchronisation at the end: copies into
    // the caller's buffers may be in flight, so no early return
    int rc = ROD_OK;
    auto cu = [&](cudaError_t e) {
        if (e != cudaSuccess && rc == ROD_OK) rc = cuda_fail(e);
        return e == cudaSuccess;
    };
    for (size_t c = 0; c + 1 < cuts.size() && rc == ROD_OK; ++c) {
        const int lo = cuts[c], hi = cuts[c + 1];
        cudaStream_t st = plan->streams[c % 3];
        const rod_image_desc& a = plan->descs[lo];
        const rod_image_desc& b = plan->descs[hi - 1];
        // byte range of the chunk's images.  A monotonic plan has increasing disjoint extents, so [first image start,
        // last image end) covers exactly the chunk; any other plan (reversed, shuffled or aliased offsets: one chunk)
        // uploads the whole span the descriptors touch.
        const uint64_t s_lo = plan->monotonic ? a.src_offset : plan->src_min_offset;
        const uint64_t s_hi = plan->monotonic ? b.src_offset + (uint64_t)(b.height - 1) * b.src_pitch + 3ull * b.width : plan->src_extent;
        const uint64_t d_lo = a.dst_offset, d_hi = b.dst_offset + (uint64_t)(b.height - 1) * b.dst_pitch + 3ull * b.width;
        if (!cu(cudaMemcpyAsync(plan->d_stage_src + s_lo, src_host + s_lo, s_hi - s_lo, cudaMemcpyHostToDevice, st))) break;
        if (compat) {
            const uint64_t e_lo = plan->h_images[lo].elem_base;
            const uint64_t e_hi = plan->h_images[hi - 1].elem_base + 3ull * b.height * b.width;
            if (!cu(cudaMemcpyAsync(plan->d_stage_noise + e_lo, noise_host + e_lo, (e_hi - e_lo) * sizeof(float),
                                    cudaMemcpyHostToDevice, st))) break;
        }
        rc = run_op(plan, op, plan->d_stage_src, plan->d_stage_dst, compat ? plan->d_stage_noise : nullptr, sigma, k,
                    factor, seed, first_image_index, offset, nullptr, st, lo, hi);
        if (rc != ROD_OK) break;
        if (dst_packed) {
            if (!cu(cudaMemcpyAsync(dst_host + d_lo, plan->d_stage_dst + d_lo, d_hi - d_lo, cudaMemcpyDeviceToHost, st))) break;
        } else {  // never write the caller's pitch padding / gaps: one 2-D copy per image
            for (int i = lo; i < hi; ++i) {
                const rod_image_desc& d = plan->descs[i];
                if (!cu(cudaMemcpy2DAsync(dst_host + d.dst_offset, (size_t)d.dst_pitch, plan->d_stage_dst + d.dst_offset,
                                          (size_t)d.dst_pitch, 3ull * d.width, (size_t)d.height, cudaMemcpyDeviceToHost, st)))
                    break;
            }
        }
    }
    for (auto& s : plan->streams) {
        cudaError_t e = cudaStreamSynchronize(s);
        if (e != cudaSuccess && rc == ROD_OK) rc = cuda_fail(e);
    }
    return rc;
}
