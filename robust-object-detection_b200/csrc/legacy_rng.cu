// legacy_rng.cu -- the compat-mode noise field drawn on the GPU: NumPy's legacy MT19937 + polar Gaussian stream, bit for
// bit, with NumPy's generator state handed back exactly (rod_numpy_legacy_normal_f32_device).
//
// A call runs in rounds (one in practice); a round in two kernels over chunks of kStride blocks of the word stream:
//   legacy_count_kernel  chunk c >= 1 generates x_0 .. x_{19937 + 623} from the round's start block into shared memory,
//                        jumps to block c kStride - 1 (rod_mt.h jump_word with the host-built polynomial of row c) and
//                        generates block c kStride from it; chunk 0 starts from the key itself.  Each chunk stores its
//                        start block, then generates its blocks and counts the accepted candidates that start in them.
//   legacy_write_kernel  each chunk adds the counts of the chunks before it, regenerates its blocks from the stored start
//                        and writes accepted pair r to stream positions 2r, 2r + 1 (mapped to the caller's segments).
//                        The chunk holding the last needed pair stores the raw block that holds the last consumed word,
//                        `pos`, and that candidate's (x1, r2).  Outputs whose float32 could depend on the last ulps of
//                        the device log() (rod_mt.h guard_ok) are listed for the host, which recomputes them with libm
//                        log(), the function NumPy calls, and patches them with scatter_kernel.
// The candidate budget of a round is the expected 4/pi per pair plus 8 sqrt(pairs) + 64 (more than 13 standard
// deviations); a round that runs short, or a call larger than kMaxChunks chunks, continues from the state it reached.
#include <cuda_runtime.h>
#include <math.h>

#include <algorithm>
#include <mutex>
#include <vector>

#include "rod_internal.h"
#include "rod_mt.h"

namespace {
using namespace rodmt;

constexpr int kStride = 128;     // blocks per chunk, by measurement (B200 at 1000 W): 1.48 ms per 1360x765x3 field
                                 // (~12.7k blocks, 100 chunks) and 13.7 ms for 16 fields, against 2.11 / 23.8 ms with
                                 // 64 blocks -- the jumps (~10k shared-memory XORs per word) dominate a round
constexpr int kMaxChunks = 256;  // chunks per round = rows of the jump table; two CTAs per SM fit 296 at once
constexpr int kThreads = 640;    // one thread per word of a block
constexpr int kFixRead = 256;    // fix-up records read back with the end state (more: a second copy)
constexpr int kScatter = 256;    // host values per scatter launch (kernel parameters)
constexpr size_t kCountSmem = sizeof(uint32_t) * kWinBlocks * kN + sizeof(uint64_t) * kPolyWords;

struct EndState {
    uint32_t key[kN];
    int32_t pos, found;  // found: the round produced every pair it needed (else it used all its candidates)
    double x1, r2;       // the last candidate (found)
    uint64_t accepted;   // accepted candidates of the round (found: at least the pairs needed)
    uint32_t fix_count, pad;
};
struct FixRec {
    uint64_t v;  // output value index of the call
    double x1, x2, r2;
    uint32_t second, pad;  // 1: the pair's second value (f x1), 0: its first (f x2)
};
struct CountArgs {
    const uint32_t* key;
    const uint64_t* table;
    uint32_t* starts;
    uint32_t* counts;
    int p, b_end;
};
struct WriteArgs {
    const uint32_t* starts;
    const uint32_t* counts;
    int p, b_end, n_chunks, n_seg;
    uint64_t need, n_vals, v0;
    double sigma;
    const uint64_t* seg;  // n_seg + 1 value starts, then n_seg element offsets
    float* out;
    FixRec* fix;
    uint32_t fix_cap;
    EndState* end;
};
struct ScatterArgs {
    float* out;
    int n;
    uint64_t idx[kScatter];
    float val[kScatter];
};

// nw := the block after old (all threads of the CTA; ends synchronised)
__device__ __forceinline__ void gen_block(const uint32_t* old, uint32_t* nw, int t) {
    const int ph = t < kN ? gen_phase(t) : 3;
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        if (ph == k) nw[t] = next_word(old, nw, t);
        __syncthreads();
    }
}

// candidate t (< 156) of block b: its first word is at offset o of the block; cur = block b, nxt = block b + 1
__device__ __forceinline__ bool block_candidate(const uint32_t* cur, const uint32_t* nxt, int b, int p, int t, int* o_out,
                                                Cand* cd) {
    if (t >= kCandPerBlock) return false;
    const int o = (p & 3) + 4 * t;
    *o_out = o;
    if (b == 0 && o < p) return false;  // words the key had already given out
    uint32_t w[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) w[k] = o + k < kN ? cur[o + k] : nxt[o + k - kN];
    *cd = candidate(w[0], w[1], w[2], w[3]);
    return accepted(cd->r2);
}

__global__ void __launch_bounds__(kThreads, 2) legacy_count_kernel(CountArgs a) {
    extern __shared__ __align__(16) uint32_t sm[];
    const int c = blockIdx.x, t = threadIdx.x;
    uint32_t *cur = sm, *nxt = sm + kN;
    if (c == 0) {
        if (t < kN) cur[t] = a.key[t];
        __syncthreads();
    } else {
        uint32_t* w = sm;
        uint64_t* g = reinterpret_cast<uint64_t*>(sm + kWinBlocks * kN);
        if (t < kN) w[t] = a.key[t];
        for (int i = t; i < kPolyWords; i += kThreads) g[i] = a.table[(size_t)c * kPolyWords + i];
        __syncthreads();
        for (int b = 1; b < kWinBlocks; ++b) gen_block(w + (b - 1) * kN, w + b * kN, t);
        const uint32_t v = t < kN ? jump_word(g, w, t) : 0u;  // block c kStride - 1 (word 0 exact in its top bit only)
        __syncthreads();
        if (t < kN) w[t] = v;
        __syncthreads();
        gen_block(w, w + kN, t);  // block c kStride: exact
        cur = w + kN;
        nxt = w;
    }
    if (t < kN) a.starts[(size_t)c * kN + t] = cur[t];
    const int b_lo = c * kStride, b_hi = min(b_lo + kStride, a.b_end);
    uint32_t count = 0;
    for (int b = b_lo; b < b_hi; ++b) {
        gen_block(cur, nxt, t);
        int o;
        Cand cd;
        const bool ok = block_candidate(cur, nxt, b, a.p, t, &o, &cd);
        count += (uint32_t)__syncthreads_count(ok);
        uint32_t* s = cur;
        cur = nxt;
        nxt = s;
    }
    if (t == 0) a.counts[c] = count;
}

__device__ __forceinline__ void put_value(const WriteArgs& a, uint64_t q, double y, const Cand& cd, uint32_t second) {
    const uint64_t v = a.v0 + q;
    int lo = 0, hi = a.n_seg;  // the segment s with seg[s] <= v < seg[s + 1]
    while (hi - lo > 1) {
        const int mid = (lo + hi) >> 1;
        if (a.seg[mid] <= v) lo = mid; else hi = mid;
    }
    a.out[a.seg[a.n_seg + 1 + lo] + (v - a.seg[lo])] = __double2float_rn(y);
    if (!guard_ok(y)) {
        const uint32_t i = atomicAdd(&a.end->fix_count, 1u);
        if (i < a.fix_cap) a.fix[i] = FixRec{v, cd.x1, cd.x2, cd.r2, second, 0u};
    }
}

__global__ void __launch_bounds__(kThreads) legacy_write_kernel(WriteArgs a) {
    __shared__ uint32_t blk[2 * kN];
    __shared__ unsigned long long s_before, s_all;
    __shared__ uint32_t warp_cnt[kCandPerBlock / 32 + 1];
    __shared__ long long s_end_word;  // absolute index of the last consumed word, once known
    __shared__ double s_end_x1, s_end_r2;
    const int c = blockIdx.x, t = threadIdx.x, lane = t & 31, warp = t >> 5;
    if (t == 0) s_before = s_all = 0, s_end_word = -1;
    __syncthreads();
    unsigned long long before = 0, all = 0;
    for (int i = t; i < a.n_chunks; i += kThreads) {
        all += a.counts[i];
        if (i < c) before += a.counts[i];
    }
    if (before) atomicAdd(&s_before, before);
    if (all) atomicAdd(&s_all, all);
    __syncthreads();
    if (s_before >= a.need) return;
    const bool short_round = c == a.n_chunks - 1 && s_all < a.need;
    uint32_t *cur = blk, *nxt = blk + kN;
    if (t < kN) cur[t] = a.starts[(size_t)c * kN + t];
    __syncthreads();
    uint64_t rank = s_before;
    const int b_lo = c * kStride, b_hi = min(b_lo + kStride, a.b_end);
    for (int b = b_lo; b < b_hi; ++b) {
        gen_block(cur, nxt, t);
        int o = 0;
        Cand cd;
        const bool ok = block_candidate(cur, nxt, b, a.p, t, &o, &cd);
        const unsigned bal = __ballot_sync(0xffffffffu, ok);
        if (lane == 0 && warp <= kCandPerBlock / 32) warp_cnt[warp] = __popc(bal);
        __syncthreads();
        uint32_t off = __popc(bal & ((1u << lane) - 1u)), in_block = 0;
#pragma unroll
        for (int k = 0; k <= kCandPerBlock / 32; ++k) {
            in_block += warp_cnt[k];
            if (k < warp) off += warp_cnt[k];
        }
        const uint64_t r = rank + off;
        if (ok && r < a.need) {
            const double f = polar_f(log(cd.r2), cd.r2);
            put_value(a, 2 * r, polar_out(a.sigma, f, cd.x2), cd, 0u);
            if (2 * r + 1 < a.n_vals) put_value(a, 2 * r + 1, polar_out(a.sigma, f, cd.x1), cd, 1u);
            if (r == a.need - 1) {
                s_end_word = (long long)b * kN + o + 3;
                s_end_x1 = cd.x1;
                s_end_r2 = cd.r2;
            }
        }
        if (short_round && b == b_hi - 1 && t == kCandPerBlock - 1) s_end_word = (long long)b * kN + o + 3;
        __syncthreads();
        if (s_end_word >= 0) {
            const long long blk_no = s_end_word / kN;
            const uint32_t* src = blk_no == b ? cur : nxt;
            if (t < kN) a.end->key[t] = src[t];
            if (t == 0) {
                a.end->pos = (int32_t)(s_end_word - blk_no * kN + 1);
                a.end->found = short_round ? 0 : 1;
                a.end->x1 = s_end_x1;
                a.end->r2 = s_end_r2;
                a.end->accepted = s_all;
            }
            return;
        }
        rank += in_block;
        uint32_t* s = cur;
        cur = nxt;
        nxt = s;
    }
}

__global__ void scatter_kernel(ScatterArgs a) {
    if ((int)threadIdx.x < a.n) a.out[a.idx[threadIdx.x]] = a.val[threadIdx.x];
}

// ---- host side --------------------------------------------------------------------------------------------------

// The jump polynomials are the same for every state: built once per process, uploaded once per device.
std::mutex g_table_mutex;
std::vector<uint64_t> g_table;  // kPolyWords words per chunk (row 0 unused)
PolyMod* g_polymod = nullptr;

// rows [from, rows) of the table -> d_table on `stream` (the copy is staged before the lock is released)
int upload_table(uint64_t* d_table, int from, int rows, cudaStream_t stream) {
    std::lock_guard<std::mutex> lk(g_table_mutex);
    try {
        if (g_polymod == nullptr) {
            std::vector<uint64_t> phi;
            if (characteristic_polynomial(phi) != kMexp) return ROD_ERR_UNSUPPORTED;  // cannot happen for MT19937
            g_polymod = new PolyMod(phi);
        }
        extend_jump_table(g_table, *g_polymod, kStride, rows);
    } catch (const std::bad_alloc&) {
        return ROD_ERR_OOM;
    }
    ROD_CUDA(cudaMemcpyAsync(d_table + (size_t)from * kPolyWords, g_table.data() + (size_t)from * kPolyWords,
                             sizeof(uint64_t) * kPolyWords * (rows - from), cudaMemcpyHostToDevice, stream));
    return ROD_OK;
}

struct DeviceScratch {
    std::mutex mutex;
    bool ready = false;
    int table_rows = 0;  // rows uploaded
    uint64_t* d_table = nullptr;
    uint32_t *d_key = nullptr, *d_starts = nullptr, *d_counts = nullptr;
    EndState* d_end = nullptr;
    FixRec* d_fix = nullptr;
    uint32_t fix_cap = 0;
    uint64_t* d_seg = nullptr;
    size_t seg_cap = 0;  // words
    // page-locked staging
    uint32_t* h_key = nullptr;
    EndState* h_end = nullptr;
    FixRec* h_fix = nullptr;
    uint32_t h_fix_cap = 0;
    uint64_t* h_seg = nullptr;
    size_t h_seg_cap = 0;
};
constexpr int kMaxDevices = 64;
DeviceScratch g_scratch[kMaxDevices];

int ensure_scratch(DeviceScratch& s) {
    if (s.ready) return ROD_OK;
    ROD_CUDA(cudaFuncSetAttribute(legacy_count_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kCountSmem));
    ROD_CUDA(cudaMalloc(&s.d_table, sizeof(uint64_t) * kPolyWords * kMaxChunks));
    ROD_CUDA(cudaMalloc(&s.d_key, sizeof(uint32_t) * kN));
    ROD_CUDA(cudaMalloc(&s.d_starts, sizeof(uint32_t) * kN * kMaxChunks));
    ROD_CUDA(cudaMalloc(&s.d_counts, sizeof(uint32_t) * kMaxChunks));
    ROD_CUDA(cudaMalloc(&s.d_end, sizeof(EndState)));
    ROD_CUDA(cudaMallocHost(&s.h_key, sizeof(uint32_t) * kN));
    ROD_CUDA(cudaMallocHost(&s.h_end, sizeof(EndState)));
    s.ready = true;
    return ROD_OK;
}

template <class T>
int grow_device(T** p, size_t* cap, size_t need, cudaStream_t stream) {
    if (*cap >= need) return ROD_OK;
    if (*p) {
        ROD_CUDA(cudaStreamSynchronize(stream));  // earlier work of this call may still read it
        ROD_CUDA(cudaFree(*p));
        *p = nullptr;
        *cap = 0;
    }
    ROD_CUDA(cudaMalloc(p, sizeof(T) * need));
    *cap = need;
    return ROD_OK;
}
template <class T>
int grow_host(T** p, size_t* cap, size_t need) {
    if (*cap >= need) return ROD_OK;
    if (*p) ROD_CUDA(cudaFreeHost(*p));
    *p = nullptr;
    *cap = 0;
    ROD_CUDA(cudaMallocHost(p, sizeof(T) * need));
    *cap = need;
    return ROD_OK;
}

}  // namespace

extern "C" ROD_API int rod_numpy_legacy_normal_f32_device(uint32_t* key, int32_t* pos, int32_t* has_gauss, double* cached,
                                                          double sigma, const uint64_t* seg_offsets, const uint64_t* seg_counts,
                                                          int n_seg, float* out, int* host_fixups, void* stream_) {
    if (key == nullptr || pos == nullptr || has_gauss == nullptr || cached == nullptr) return ROD_ERR_INVALID_ARG;
    if (*pos < 0 || *pos > kN || n_seg < 0 || !(sigma >= 0.0) || isinf(sigma)) return ROD_ERR_INVALID_ARG;
    if (n_seg > 0 && (seg_offsets == nullptr || seg_counts == nullptr)) return ROD_ERR_INVALID_ARG;
    uint64_t n = 0;
    for (int s = 0; s < n_seg; ++s) {  // sorted, disjoint, no overflow
        const uint64_t end = seg_offsets[s] + seg_counts[s];
        if (end < seg_offsets[s] || n + seg_counts[s] < n) return ROD_ERR_INVALID_ARG;
        if (s + 1 < n_seg && end > seg_offsets[s + 1]) return ROD_ERR_INVALID_ARG;
        n += seg_counts[s];
    }
    if (host_fixups) *host_fixups = 0;
    if (n == 0) return ROD_OK;
    if (out == nullptr) return ROD_ERR_INVALID_ARG;
    int dev = 0;
    ROD_CUDA(cudaGetDevice(&dev));
    if (dev < 0 || dev >= kMaxDevices) return ROD_ERR_UNSUPPORTED;
    cudaStream_t stream = (cudaStream_t)stream_;
    DeviceScratch& S = g_scratch[dev];
    std::lock_guard<std::mutex> lk(S.mutex);
    if (int st = ensure_scratch(S)) return st;

    // segment table: value starts (n_seg + 1), then element offsets (n_seg)
    std::vector<uint64_t> seg((size_t)2 * n_seg + 1);
    seg[0] = 0;
    for (int s = 0; s < n_seg; ++s) {
        seg[s + 1] = seg[s] + seg_counts[s];
        seg[n_seg + 1 + s] = seg_offsets[s];
    }
    if (int st = grow_host(&S.h_seg, &S.h_seg_cap, seg.size())) return st;
    if (int st = grow_device(&S.d_seg, &S.seg_cap, seg.size(), stream)) return st;
    memcpy(S.h_seg, seg.data(), sizeof(uint64_t) * seg.size());
    ROD_CUDA(cudaMemcpyAsync(S.d_seg, S.h_seg, sizeof(uint64_t) * seg.size(), cudaMemcpyHostToDevice, stream));
    auto element_of = [&](uint64_t v) {
        const int s = (int)(std::upper_bound(seg.begin(), seg.begin() + n_seg + 1, v) - seg.begin()) - 1;
        return seg[n_seg + 1 + s] + (v - seg[s]);
    };

    std::vector<std::pair<uint64_t, float>> patches;  // (element offset, value) settled on the host
    uint64_t done = 0;
    int fixups = 0;
    if (*has_gauss) {  // legacy_gauss hands out the cached value first
        patches.push_back({element_of(0), (float)(0.0 + sigma * *cached)});
        done = 1;
    }
    uint32_t cur_key[kN];
    memcpy(cur_key, key, sizeof(cur_key));
    int cur_pos = *pos, end_has = 0;
    double end_cached = 0.0;
    while (done < n) {
        const uint64_t n_vals = n - done, need = (n_vals + 1) / 2;
        const uint64_t cand = (uint64_t)ceil((double)need * 1.2732395447351628) + 8 * (uint64_t)ceil(sqrt((double)need)) + 64;
        uint64_t b_end = ((uint64_t)cur_pos + 4 * cand + kN - 1) / kN;
        int n_chunks = (int)std::min<uint64_t>((b_end + kStride - 1) / kStride, kMaxChunks);
        b_end = std::min<uint64_t>(b_end, (uint64_t)n_chunks * kStride);
        if (n_chunks > S.table_rows) {
            if (int st = upload_table(S.d_table, S.table_rows, n_chunks, stream)) return st;
            S.table_rows = n_chunks;
        }
        memcpy(S.h_key, cur_key, sizeof(cur_key));
        ROD_CUDA(cudaMemcpyAsync(S.d_key, S.h_key, sizeof(cur_key), cudaMemcpyHostToDevice, stream));
        legacy_count_kernel<<<n_chunks, kThreads, kCountSmem, stream>>>(
            CountArgs{S.d_key, S.d_table, S.d_starts, S.d_counts, cur_pos, (int)b_end});
        ROD_CUDA(cudaGetLastError());
        // expected flags: ~2^-21.5 per value; the buffer holds ~1000x that
        size_t cap = S.fix_cap;
        if (int st = grow_device(&S.d_fix, &cap, (size_t)4096 + n_vals / 4096, stream)) return st;
        S.fix_cap = (uint32_t)cap;
        for (;;) {
            ROD_CUDA(cudaMemsetAsync(S.d_end, 0, sizeof(EndState), stream));
            WriteArgs wa{S.d_starts, S.d_counts, cur_pos, (int)b_end, n_chunks, n_seg, need, n_vals, done, sigma,
                         S.d_seg, out, S.d_fix, S.fix_cap, S.d_end};
            legacy_write_kernel<<<n_chunks, kThreads, 0, stream>>>(wa);
            ROD_CUDA(cudaGetLastError());
            size_t hcap = S.h_fix_cap;
            if (int st = grow_host(&S.h_fix, &hcap, (size_t)kFixRead)) return st;
            S.h_fix_cap = (uint32_t)hcap;
            ROD_CUDA(cudaMemcpyAsync(S.h_end, S.d_end, sizeof(EndState), cudaMemcpyDeviceToHost, stream));
            ROD_CUDA(cudaMemcpyAsync(S.h_fix, S.d_fix, sizeof(FixRec) * kFixRead, cudaMemcpyDeviceToHost, stream));
            ROD_CUDA(cudaStreamSynchronize(stream));  // the one host wait of a round: NumPy's state is known now
            if (S.h_end->fix_count <= S.fix_cap) break;
            cap = S.fix_cap;  // more flagged values than the buffer holds: write the round again with a larger one
            if (int st = grow_device(&S.d_fix, &cap, (size_t)S.h_end->fix_count * 2, stream)) return st;
            S.fix_cap = (uint32_t)cap;
        }
        const EndState& e = *S.h_end;
        const uint32_t nfix = e.fix_count;
        if (nfix > kFixRead) {
            size_t hcap = S.h_fix_cap;
            if (int st = grow_host(&S.h_fix, &hcap, (size_t)nfix)) return st;
            S.h_fix_cap = (uint32_t)hcap;
            ROD_CUDA(cudaMemcpyAsync(S.h_fix, S.d_fix, sizeof(FixRec) * nfix, cudaMemcpyDeviceToHost, stream));
            ROD_CUDA(cudaStreamSynchronize(stream));
        }
        for (uint32_t i = 0; i < nfix; ++i) {  // NumPy's arithmetic with the libm log() NumPy calls
            const FixRec& f = S.h_fix[i];
            const double fac = sqrt(-2.0 * log(f.r2) / f.r2);
            patches.push_back({element_of(f.v), (float)(0.0 + sigma * (fac * (f.second ? f.x1 : f.x2)))});
        }
        fixups += (int)nfix;
        memcpy(cur_key, e.key, sizeof(cur_key));
        cur_pos = e.pos;
        const uint64_t pairs = std::min<uint64_t>(e.accepted, need);
        if (e.found && (n_vals & 1)) {  // odd count: the second value of the last pair stays cached, as a double
            const double fac = sqrt(-2.0 * log(e.r2) / e.r2);
            end_has = 1;
            end_cached = fac * e.x1;
        }
        done += std::min<uint64_t>(2 * pairs, n_vals);
    }
    for (size_t i = 0; i < patches.size(); i += kScatter) {
        ScatterArgs sa;
        sa.out = out;
        sa.n = (int)std::min<size_t>(kScatter, patches.size() - i);
        for (int k = 0; k < sa.n; ++k) {
            sa.idx[k] = patches[i + k].first;
            sa.val[k] = patches[i + k].second;
        }
        scatter_kernel<<<1, kScatter, 0, stream>>>(sa);
        ROD_CUDA(cudaGetLastError());
    }
    memcpy(key, cur_key, sizeof(cur_key));
    *pos = cur_pos;
    *has_gauss = end_has;
    *cached = end_cached;
    if (host_fixups) *host_fixups = fixups;
    return ROD_OK;
}
