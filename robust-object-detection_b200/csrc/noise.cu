// noise.cu -- a1: fused uint8 -> fp32 -> saturate -> uint8 Gaussian-noise kernel (sm_100a).
//
// Reference: scripts/augmentations.py:30-33 (apply_noise).  Two sources for the field:
//   NOISE_COMPAT  a supplied float32 tensor (what np.random.normal(...).astype(f32) drew) -> bit-exact
//   NOISE_PHILOX  Philox4x32-10 keyed by (seed, global image index, element/8, offset), no HBM traffic for
//                 the field; two Gaussian generators on the same Philox blocks (rod_core.h):
//                   table      (3 <= sigma <= 20, noise_table_kernel): four 8-bit draws per Philox word from a 256-entry
//                              table in shared memory, mixed by a 4 x 4 Hadamard transform in integer arithmetic:
//                              one Philox block per 16 elements, no MUFU, no bank conflicts
//                   Box-Muller (any sigma <= 2048, noise_kernel<NOISE_PHILOX>): 4 MUFU per pair, XU-pipe bound
// plus NOISE_COPY (ROD_OP_NONE images of a mixed batch) and NOISE_FIELD (dump the Philox field).
//
// HBM-bound elementwise op: one work item is a span of <= 16384 consecutive bytes; each
// thread moves 16 bytes per step with 128-bit loads/stores that bypass L1.  Spans whose
// addresses are not 16-byte aligned (pitched rows of strided views) take a byte path.

#include <mutex>
#include <vector>

#include "rod_internal.h"
#include "rod_tables.h"

namespace rod {

struct NoiseParams {
    const DevImage* images;
    const Tile* tiles;
    int n_tiles;
    const uint8_t* src;
    uint8_t* dst;
    const float* noise;
    float* field_out;
    float sigma;
    uint32_t key0, key1;
    PhiloxKeys keys;        // the ten round keys of (key0, key1)
    uint64_t first_image;
    uint32_t offset;
    const uint8_t* opcodes;
    int my_op;
    unsigned int* counter;  // zeroed before the launch
    int piece_shift;        // table kernel: a work item is 1 / (1 << piece_shift) of a span
    const int32_t* table;   // table generator: the 256 entries X[i] (device global; expanded into shared memory)
};

__device__ __forceinline__ uint4 ldg_stream16(const void* p) {
    uint4 r;
    asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];"
                 : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w)
                 : "l"(p));
    return r;
}
__device__ __forceinline__ float4 ldg_stream16f(const void* p) {
    float4 r;
    asm volatile("ld.global.nc.L1::no_allocate.v4.f32 {%0,%1,%2,%3}, [%4];"
                 : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w)
                 : "l"(p));
    return r;
}
__device__ __forceinline__ uint32_t ldg_stream4(const void* p) {
    uint32_t r;
    asm volatile("ld.global.nc.L1::no_allocate.u32 %0, [%1];" : "=r"(r) : "l"(p));
    return r;
}
__device__ __forceinline__ void stg4(void* p, uint32_t v) {
    asm volatile("st.global.L1::no_allocate.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ void stg16(void* p, uint4 v) {
    asm volatile("st.global.L1::no_allocate.v4.u32 [%0], {%1,%2,%3,%4};" ::"l"(p), "r"(v.x), "r"(v.y), "r"(v.z),
                 "r"(v.w)
                 : "memory");
}

// byte b of word -> exact float, without I2F: 0x4B0000bb is 2^23 + bb
__device__ __forceinline__ float byte_to_float(uint32_t word, int b) {
    return __uint_as_float(__byte_perm(word, 0x4B000000u, 0x7440 | b)) - 8388608.0f;
}

__device__ __forceinline__ uint32_t noise_word(uint32_t word, float n0, float n1, float n2, float n3) {
    uint32_t o0 = noise_px(byte_to_float(word, 0), n0);
    uint32_t o1 = noise_px(byte_to_float(word, 1), n1);
    uint32_t o2 = noise_px(byte_to_float(word, 2), n2);
    uint32_t o3 = noise_px(byte_to_float(word, 3), n3);
    return o0 | (o1 << 8) | (o2 << 16) | (o3 << 24);
}

// One Philox group: the eight factors s[0..7] of elements 8g .. 8g+7 (rod_core.h gauss8).
__device__ __forceinline__ void group_gauss8(const NoiseParams& p, uint32_t ig_lo, uint32_t ig_hi, uint32_t g,
                                             float s[8]) {
    uint32_t r[4];
    philox4x32_10_rk(g, ig_lo, ig_hi, p.offset, p.keys, r);
    if (philox_needs_tail(r)) {  // 2^-14 of the groups: refine the radius of the words whose high half is 0
        uint32_t t[4];
        philox4x32_10(g, ig_lo, ig_hi ^ ROD_PHILOX_TAIL_FLIP, p.offset, p.key0, p.key1, t);
        gauss8(r, t, s);
    } else {
        gauss8(r, nullptr, s);
    }
}

template <int MODE>
__global__ void __launch_bounds__(256, 4) noise_kernel(NoiseParams p) {
    const float K = p.sigma * ROD_NOISE_K_PER_SIGMA;
    // a warp takes a quarter span (<= 4096 bytes) at a time from a shared counter: no tail, no block-level coupling
    const uint32_t lane = threadIdx.x & 31u;
    for (;;) {
        uint32_t id = 0;
        if (lane == 0) id = atomicAdd(p.counter, 1u);
        id = __shfl_sync(0xFFFFFFFFu, id, 0);
        if ((int)(id >> 2) >= p.n_tiles) break;
        Tile t = p.tiles[id >> 2];
        if (p.opcodes != nullptr && p.opcodes[t.img] != p.my_op) continue;
        const int piece0 = (int)(id & 3u) * (kNoiseSpan / 4);
        if (piece0 >= t.b) continue;
        t.a += piece0;
        t.b = min(kNoiseSpan / 4, t.b - piece0);
        const DevImage im = p.images[t.img];
        const uint64_t img_global = p.first_image + (uint64_t)t.img;
        const uint32_t ig_lo = (uint32_t)img_global, ig_hi = (uint32_t)(img_global >> 32);
        const uint8_t* s = nullptr;
        uint8_t* d = nullptr;
        uint32_t e0;  // element index (inside the image) of the span's first byte
        if (t.c < 0) {
            e0 = (uint32_t)t.a;
            if (MODE != NOISE_FIELD) { s = p.src + im.src_off + e0; d = p.dst + im.dst_off + e0; }
        } else {
            e0 = (uint32_t)t.c * 3u * (uint32_t)im.w + (uint32_t)t.a;
            if (MODE != NOISE_FIELD) {
                s = p.src + im.src_off + (int64_t)t.c * im.src_pitch + t.a;
                d = p.dst + im.dst_off + (int64_t)t.c * im.dst_pitch + t.a;
            }
        }
        const uint32_t n = (uint32_t)t.b;
        const float* nzp = (MODE == NOISE_COMPAT) ? p.noise + im.elem_base + e0 : nullptr;
        float* fout = (MODE == NOISE_FIELD) ? p.field_out + im.elem_base + e0 : nullptr;

        uint32_t done = 0;  // elements of the span finished by the vector paths
        if (MODE == NOISE_COMPAT) {
            // 4 pixels (one word) + one float4 of the field per thread step; every warp instruction is fully
            // coalesced (128 B of pixels, 512 B of field); four independent steps in flight per thread
            const bool vec4 = (e0 & 3u) == 0 && ((((uintptr_t)s) | ((uintptr_t)d)) & 3) == 0 && (((uintptr_t)nzp) & 15) == 0;
            const uint32_t nw = vec4 ? (n >> 2) : 0;
            for (uint32_t base = lane; base < nw; base += 4 * 32u) {
                uint32_t px[4];
                float4 f[4];
#pragma unroll
                for (int u = 0; u < 4; ++u) {
                    const uint32_t idx = base + u * 32u;
                    if (idx < nw) {
                        px[u] = ldg_stream4(s + 4 * idx);
                        f[u] = ldg_stream16f(nzp + 4 * idx);
                    }
                }
#pragma unroll
                for (int u = 0; u < 4; ++u) {
                    const uint32_t idx = base + u * 32u;
                    if (idx < nw) stg4(d + 4 * idx, noise_word(px[u], f[u].x, f[u].y, f[u].z, f[u].w));
                }
            }
            done = nw << 2;
        } else {
            // 16 bytes per thread step = two Philox groups: needs the span to start on a group boundary
            bool vec = (e0 & 7u) == 0;
            if (MODE != NOISE_FIELD) vec = vec && ((((uintptr_t)s) | ((uintptr_t)d)) & 15) == 0;
            if (MODE == NOISE_FIELD) vec = vec && (((uintptr_t)fout) & 15) == 0;
            const uint32_t nvec = vec ? (n >> 4) : 0;
            for (uint32_t i = lane; i < nvec; i += 32u) {
                const uint32_t e = 16u * i;
                uint4 v = make_uint4(0, 0, 0, 0);
                if (MODE != NOISE_FIELD) v = ldg_stream16(s + e);
                if (MODE == NOISE_COPY) {
                    stg16(d + e, v);
                    continue;
                }
                const uint32_t in[4] = {v.x, v.y, v.z, v.w};
                uint32_t out[4];
#pragma unroll
                for (int h = 0; h < 2; ++h) {
                    float sf[8];
                    group_gauss8(p, ig_lo, ig_hi, ((e0 + e) >> 3) + h, sf);
                    if (MODE == NOISE_FIELD) {
                        float4* fo = reinterpret_cast<float4*>(fout + e + 8 * h);
                        fo[0] = make_float4(K * sf[0], K * sf[1], K * sf[2], K * sf[3]);
                        fo[1] = make_float4(K * sf[4], K * sf[5], K * sf[6], K * sf[7]);
                    } else {
                        out[2 * h] = philox_word(in[2 * h], sf, K);
                        out[2 * h + 1] = philox_word(in[2 * h + 1], sf + 4, K);
                    }
                }
                if (MODE != NOISE_FIELD) stg16(d + e, make_uint4(out[0], out[1], out[2], out[3]));
            }
            done = nvec << 4;
        }

        // remainder (and the whole span when unaligned): one Philox group (<= 8 elements) per thread step
        const uint32_t r0 = done;                // first element not yet done, relative to the span
        if (r0 < n) {
            const uint32_t ea = e0 + r0, eb = e0 + n;      // absolute element range [ea, eb)
            const uint32_t g_first = ea >> 3, g_last = (eb - 1) >> 3;
            for (uint32_t g = g_first + lane; g <= g_last; g += 32u) {
                float sf[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
                if (MODE == NOISE_PHILOX || MODE == NOISE_FIELD) group_gauss8(p, ig_lo, ig_hi, g, sf);
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                    const uint32_t e = 8u * g + j;
                    if (e < ea || e >= eb) continue;
                    const uint32_t rel = e - e0;
                    if (MODE == NOISE_FIELD) { fout[rel] = K * sf[j]; continue; }
                    const uint32_t v = s[rel];
                    if (MODE == NOISE_COPY) { d[rel] = (uint8_t)v; continue; }
                    if (MODE == NOISE_COMPAT) d[rel] = (uint8_t)noise_px(__uint_as_float(0x4B000000u | v) - 8388608.0f, nzp[rel]);
                    else d[rel] = (uint8_t)noise_philox_px(v, sf[j], K);
                }
            }
        }
    }
}

// ---------------------------------------------------------------------------------------------------
// Table generator of Philox mode (definition: rod_core.h).
// ---------------------------------------------------------------------------------------------------
// Shared-memory layout of the table kernel: 256 rows of 256 bytes at a 64 KB-ALIGNED shared address `tbase`; row i holds,
// for each of the 32 lanes, the (x, x) form of entry i at byte 4 * lane and the (x, -x) form at byte 128 + 4 * lane.  The
// address of a draw is therefore ONE byte permute -- byte 1 = the index byte of the Philox word, bytes 0, 2, 3 = the
// lane's base -- and every lane reads its own bank: no conflicts, one wavefront per load (the 15-bit shared table this
// replaces cost 3.6 wavefronts per random 16-bit load and had the LSU pipe at 82 %).
constexpr uint32_t kTabSmemBytes = 65536u + 65536u;  // table + slack to reach the next 64 KB boundary

__device__ __forceinline__ uint32_t lds_u32(uint32_t addr) {
    uint32_t v;
    asm("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(addr));
    return v;
}
__device__ __forceinline__ uint32_t prmt(uint32_t a, uint32_t b, uint32_t sel) {
    uint32_t d;
    asm("prmt.b32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(sel));
    return d;
}

// One Philox word -> the four elements it makes: f01 / f23 = int16 pairs (k + 128) of elements (0, 1) / (2, 3).
// base_s / base_d: tbase + 4 * lane (+ 128): the lane's column of the (x, x) / (x, -x) forms.
__device__ __forceinline__ void table_word4(uint32_t r, uint32_t base_s, uint32_t base_d, uint32_t& f01, uint32_t& f23) {
    const uint32_t A = lds_u32(prmt(r, base_s, 0x7604u)), B = lds_u32(prmt(r, base_d, 0x7614u));
    const uint32_t C = lds_u32(prmt(r, base_s, 0x7624u)), D = lds_u32(prmt(r, base_d, 0x7634u));
    uint32_t e01, e23;
    h4_combine(A, B, C, D, &e01, &e23);
    f01 = prmt(e01, 0u, 0x4341u);  // bytes 1 and 3 -> the two halves
    f23 = prmt(e23, 0u, 0x4341u);
}

// four pixels (one word) + two packed pairs -> four output bytes: clamp((v - 128) + kb, 0, 255) = clamp(v + k, 0, 255)
__device__ __forceinline__ uint32_t table_word(uint32_t word, uint32_t f01, uint32_t f23) {
    const uint32_t w = word ^ 0x80808080u;  // int8(v ^ 0x80) = v - 128
    const uint32_t v01 = prmt(w, 0u, 0x9180u), v23 = prmt(w, 0u, 0xB3A2u);  // sign-extended to int16 pairs
    const uint32_t q01 = __viaddmin_s16x2_relu(f01, v01, 0x00FF00FFu);
    const uint32_t q23 = __viaddmin_s16x2_relu(f23, v23, 0x00FF00FFu);
    return __byte_perm(q01, q23, 0x6420);
}

// One group (16 elements), element by element, restricted to the absolute element range [ea, eb): the remainder of
// spans whose start is not on a group boundary / not 16-byte aligned (pitched rows).  e0 = element index of s[0] / d[0].
template <int MODE, int ROUNDS>
__device__ __noinline__ void table_group_slow(const NoiseParams& p, uint32_t base_s, uint32_t base_d, uint32_t ig_lo,
                                              uint32_t ig_hi, uint32_t g, uint32_t e0, uint32_t ea, uint32_t eb,
                                              const uint8_t* s, uint8_t* d, float* fout) {
    uint32_t r[4];
    philox4x32_rk<ROUNDS>(g, ig_lo, ig_hi, p.offset, p.keys, r);
#pragma unroll
    for (int q = 0; q < 4; ++q) {
        uint32_t f01, f23;
        table_word4(r[q], base_s, base_d, f01, f23);
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const uint32_t e = 16u * g + 4u * q + j;
            if (e < ea || e >= eb) continue;
            const int k = (int)(((j & 2) ? f23 : f01) >> (16 * (j & 1)) & 0xFFFFu) - 128;
            const uint32_t rel = e - e0;
            if (MODE == NOISE_FIELD) fout[rel] = (float)k;
            else d[rel] = (uint8_t)noise_table_px(s[rel], k);
        }
    }
}

// Same work hand-out as noise_kernel (warps take quarter spans from a shared counter); the CTA first expands the
// 256-entry table (1 KB in global memory) into its lane-replicated two-form shared copy.  MODE: NOISE_PHILOX or NOISE_FIELD.
template <int MODE, int THREADS, int UNROLL, int ROUNDS>
__global__ void __launch_bounds__(THREADS, 1) noise_table_kernel(NoiseParams p) {
    extern __shared__ __align__(16) uint8_t s_raw[];
    const uint32_t tbase = ((uint32_t)__cvta_generic_to_shared(s_raw) + 0xFFFFu) & ~0xFFFFu;
    for (int i = threadIdx.x; i < 256 * 64; i += THREADS) {
        const int row = i >> 6, col = i & 63;  // col < 32: (x, x) form of lane col; else (x, -x) form of lane col - 32
        const int32_t x = __ldg(p.table + row);
        const uint32_t v = col < 32 ? h4_form_same(x) : h4_form_diff(x);
        asm volatile("st.shared.u32 [%0], %1;" ::"r"(tbase + 4u * (uint32_t)i), "r"(v) : "memory");
    }
    __syncthreads();
    const uint32_t lane = threadIdx.x & 31u;
    const uint32_t base_s = tbase + 4u * lane, base_d = base_s + 128u;
    // a warp takes a piece (a span, or a half / quarter of one: p.piece_shift) at a time from a shared counter
    // (prefetching the next counter value during the current piece measured +-1 %: not done)
    const uint32_t pmask = (1u << p.piece_shift) - 1u;
    const int piece_len = kNoiseSpan >> p.piece_shift;
    for (;;) {
        uint32_t id = 0;
        if (lane == 0) id = atomicAdd(p.counter, 1u);
        id = __shfl_sync(0xFFFFFFFFu, id, 0);
        if ((int)(id >> p.piece_shift) >= p.n_tiles) break;
        Tile t = p.tiles[id >> p.piece_shift];
        if (p.opcodes != nullptr && p.opcodes[t.img] != p.my_op) continue;
        const int piece0 = (int)(id & pmask) * piece_len;
        if (piece0 >= t.b) continue;
        t.a += piece0;
        t.b = min(piece_len, t.b - piece0);
        const DevImage im = p.images[t.img];
        const uint64_t img_global = p.first_image + (uint64_t)t.img;
        const uint32_t ig_lo = (uint32_t)img_global, ig_hi = (uint32_t)(img_global >> 32);
        const uint8_t* s = nullptr;
        uint8_t* d = nullptr;
        uint32_t e0;  // element index (inside the image) of the span's first byte
        if (t.c < 0) {
            e0 = (uint32_t)t.a;
            if (MODE != NOISE_FIELD) { s = p.src + im.src_off + e0; d = p.dst + im.dst_off + e0; }
        } else {
            e0 = (uint32_t)t.c * 3u * (uint32_t)im.w + (uint32_t)t.a;
            if (MODE != NOISE_FIELD) {
                s = p.src + im.src_off + (int64_t)t.c * im.src_pitch + t.a;
                d = p.dst + im.dst_off + (int64_t)t.c * im.dst_pitch + t.a;
            }
        }
        const uint32_t n = (uint32_t)t.b;
        float* fout = (MODE == NOISE_FIELD) ? p.field_out + im.elem_base + e0 : nullptr;

        // 16 bytes per thread step = one Philox group: needs the span to start on a group boundary
        bool vec = (e0 & 15u) == 0;
        if (MODE != NOISE_FIELD) vec = vec && ((((uintptr_t)s) | ((uintptr_t)d)) & 15) == 0;
        if (MODE == NOISE_FIELD) vec = vec && (((uintptr_t)fout) & 15) == 0;
        const uint32_t nvec = vec ? (n >> 4) : 0;
        const uint32_t g0 = e0 >> 4;
#pragma unroll UNROLL
        for (uint32_t i = lane; i < nvec; i += 32u) {
            const uint32_t e = 16u * i;
            uint4 v = make_uint4(0, 0, 0, 0);
            if (MODE != NOISE_FIELD) v = ldg_stream16(s + e);
            uint32_t r[4], f[8];
            philox4x32_rk<ROUNDS>(g0 + i, ig_lo, ig_hi, p.offset, p.keys, r);
#pragma unroll
            for (int q = 0; q < 4; ++q) table_word4(r[q], base_s, base_d, f[2 * q], f[2 * q + 1]);
            if (MODE == NOISE_FIELD) {
                float4* fo = reinterpret_cast<float4*>(fout + e);
#pragma unroll
                for (int q = 0; q < 4; ++q)
                    fo[q] = make_float4((float)((int)(f[2 * q] & 0xFFFFu) - 128), (float)((int)(f[2 * q] >> 16) - 128),
                                        (float)((int)(f[2 * q + 1] & 0xFFFFu) - 128), (float)((int)(f[2 * q + 1] >> 16) - 128));
            } else {
                stg16(d + e, make_uint4(table_word(v.x, f[0], f[1]), table_word(v.y, f[2], f[3]),
                                        table_word(v.z, f[4], f[5]), table_word(v.w, f[6], f[7])));
            }
        }
        // remainder (and the whole span when unaligned): one Philox group (<= 16 elements) per thread step
        const uint32_t r0 = nvec << 4;
        if (r0 < n) {
            const uint32_t ea = e0 + r0, eb = e0 + n;  // absolute element range [ea, eb)
            const uint32_t g_first = ea >> 4, g_last = (eb - 1) >> 4;
            for (uint32_t g = g_first + lane; g <= g_last; g += 32u)
                table_group_slow<MODE, ROUNDS>(p, base_s, base_d, ig_lo, ig_hi, g, e0, ea, eb, s, d, fout);
        }
    }
}

// Device copies of the 256-entry table, one per (device, sigma), built on first use.  rod_noise_prewarm() builds it ahead
// of time (the upload is synchronous: the FIRST Philox launch with a new sigma must not happen inside a stream capture).
struct GaussTable {
    int device;
    uint32_t sigma_bits;
    int32_t* d_tab;
};
static std::mutex g_tab_mutex;
static std::vector<GaussTable> g_tabs;

int gauss_table_for(int device, float sigma, const int32_t** out) {
    std::lock_guard<std::mutex> lock(g_tab_mutex);
    const uint32_t bits = fbits(sigma);
    for (const GaussTable& t : g_tabs)
        if (t.device == device && t.sigma_bits == bits) { *out = t.d_tab; return ROD_OK; }
    int32_t h[256];
    build_gauss_table(sigma, h);
    int32_t* d = nullptr;
    ROD_CUDA(cudaMalloc(&d, sizeof(h)));
    cudaError_t e = cudaMemcpy(d, h, sizeof(h), cudaMemcpyHostToDevice);
    if (e != cudaSuccess) { cudaFree(d); return cuda_fail(e); }
    g_tabs.push_back(GaussTable{device, bits, d});
    *out = d;
    return ROD_OK;
}

int launch_noise(const rod_plan* plan, int mode, const uint8_t* src, uint8_t* dst, const float* noise,
                 float* field_out, float sigma, uint64_t seed, uint64_t first_image, uint32_t offset,
                 const uint8_t* opcodes, int my_op, cudaStream_t stream, int img_lo, int img_hi, int generator) {
    const auto [tiles, n_tiles] = plan->noise_tiles.range(img_lo, img_hi);
    if (n_tiles == 0) return ROD_OK;
    if (generator < 0) generator = plan->gauss_generator;
    NoiseParams p;
    p.images = plan->d_images;
    p.tiles = tiles;
    p.n_tiles = n_tiles;
    p.src = src; p.dst = dst; p.noise = noise; p.field_out = field_out;
    p.sigma = sigma;
    p.key0 = (uint32_t)seed; p.key1 = (uint32_t)(seed >> 32);
    p.keys = philox_round_keys(p.key0, p.key1);
    p.first_image = first_image;
    p.offset = offset;
    p.opcodes = opcodes; p.my_op = my_op;
    p.table = nullptr;
    p.counter = plan->d_counters + (plan->launch_seq.fetch_add(1u) & (kCounterRing - 1u));
    ROD_CUDA(cudaMemsetAsync(p.counter, 0, sizeof(unsigned int), stream));
    const int per_sm = 4;  // CTAs per SM the grid is sized for: 4 are resident, a longer queue evens out the tail
    if ((mode == NOISE_PHILOX || mode == NOISE_FIELD) && (generator == ROD_GAUSS_AUTO || generator == ROD_GAUSS_TABLE_PHILOX7) &&
        sigma >= ROD_GAUSS_TABLE_MIN_SIGMA && sigma <= ROD_GAUSS_TABLE_MAX_SIGMA) {
        int rc = gauss_table_for(plan->device, sigma, &p.table);
        if (rc != ROD_OK) return rc;
        // one 1024-thread CTA per SM, each with its own copy of the table; warps take pieces of spans
        // Work item = a whole span when there are plenty (>= 8 per resident warp), else a half / quarter span so that
        // small batches still spread over all warps.  Measured on a B200, sigma 15, 1360x765: 256 images 5.10 TB/s with
        // whole spans vs 4.87 with quarter spans (fewer atomic -> tile -> image dependency chains); 16 images 2.74 TB/s
        // with quarter spans vs 2.38 with whole spans.
        const long warps = 32L * plan->sm_count;
        p.piece_shift = p.n_tiles >= 8 * warps ? 0 : (2L * p.n_tiles >= 8 * warps ? 1 : 2);
        const int ctas = grid_for(plan, ((p.n_tiles << p.piece_shift) + 31) / 32, 1);
#define ROD_TAB_LAUNCH(M, TH, UN, R)                                                                                       \
    do {                                                                                                                   \
        ROD_CUDA(cudaFuncSetAttribute(noise_table_kernel<M, TH, UN, R>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kTabSmemBytes)); \
        noise_table_kernel<M, TH, UN, R><<<ctas, TH, kTabSmemBytes, stream>>>(p);                                          \
    } while (0)
        const bool r7 = generator == ROD_GAUSS_TABLE_PHILOX7;
        if (mode == NOISE_FIELD) {
            if (r7) ROD_TAB_LAUNCH(NOISE_FIELD, 1024, 2, 7); else ROD_TAB_LAUNCH(NOISE_FIELD, 1024, 2, 10);
        } else if (r7) {
            ROD_TAB_LAUNCH(NOISE_PHILOX, 1024, 2, 7);
        } else {
            ROD_TAB_LAUNCH(NOISE_PHILOX, 1024, 2, 10);
        }
#undef ROD_TAB_LAUNCH
        ROD_CUDA(cudaGetLastError());
        return ROD_OK;
    }
    const int grid = grid_for(plan, (p.n_tiles + 1) / 2, per_sm);  // a CTA's 8 warps cover two spans at a time
    switch (mode) {
        case NOISE_COMPAT: noise_kernel<NOISE_COMPAT><<<grid, 256, 0, stream>>>(p); break;
        case NOISE_PHILOX: noise_kernel<NOISE_PHILOX><<<grid, 256, 0, stream>>>(p); break;
        case NOISE_COPY: noise_kernel<NOISE_COPY><<<grid, 256, 0, stream>>>(p); break;
        case NOISE_FIELD: noise_kernel<NOISE_FIELD><<<grid, 256, 0, stream>>>(p); break;
        default: return ROD_ERR_INVALID_ARG;
    }
    ROD_CUDA(cudaGetLastError());
    return ROD_OK;
}

}  // namespace rod
