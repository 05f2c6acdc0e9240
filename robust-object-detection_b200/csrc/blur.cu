// blur.cu -- a2+a3: horizontal k-tap motion blur (angle 0) on interleaved 3-channel rows (sm_100a).
//
// Reference: scripts/augmentations.py:21-38 -> cv2.filter2D(img, -1, kernel) with the angle-0
// kernel = k taps of float32(1/k) on one row, BORDER_REFLECT_101, i.e. per channel
//     out[x] = round(sum_{j=-r..r} in[reflect101(x + j)] / k)  ==  (2 S + k) / (2 k)   (odd k).
//
// Rows are independent.  A CTA runs one producer warp and up to 8 consumer warps around a ring of row slots in shared
// memory.  The producer (one lane) claims 8-row tiles from a work counter, one claim ahead of use, and for each row waits
// until its slot is free, writes the slot's descriptor and starts one bulk async copy (cp.async.bulk, completing on the
// slot's "full" mbarrier) of the row's 16-byte-aligned interior, placed at the SAME 16-byte phase as the destination row.
// Consumer warp i takes rows i, i + W, i + 2W, ... of the CTA's sequence: it loads the (at most two) partial 16-byte
// edges itself, writes the reflected halo next to the row, and every lane then produces 16 output bytes per step from
// three 128-bit shared-memory loads and stores them with one 128-bit global store; then it frees the slot.  Rows whose
// source and destination phases differ are copied into the slot by the consumer byte by byte.
// So the bytes of the next rows are in flight while the consumers compute, and the claims are off their path.
//
// The work counter and a "done" counter are a pair of the plan's blur counters.  Each CTA counts itself done after its
// final, failing claim; the CTA that completes the count returns both to 0, so the next launch that takes the pair finds
// it zeroed without a memset.

#include <algorithm>

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
    int row_buf_bytes;      // shared bytes per row slot
    int slots;              // row slots per CTA (>= consumer warps)
    unsigned int* counters;  // {work counter, done counter}: 0 at the launch, returned to 0 by the last CTA
};

constexpr int kBlurLeft = 64;      // bytes in front of the 16-byte block that holds pixel 0 (>= 3*15 halo + 16)
constexpr int kBlurMaxSlots = 16;  // row slots per CTA
constexpr int kBlurCtasPerSm = 3;  // 16 slots of a 1360-wide row (4 224 B) each: 48 rows in flight per SM

// Per-slot header, in front of the row buffers.  The producer writes it before it arrives on `full`.
struct BlurSlot {
    uint64_t full, empty;  // mbarriers: full completes on the producer's arrival + the bulk copy, empty on the consumer's
    const uint8_t* srow;   // nullptr: no more rows for this consumer
    uint8_t* drow;
    int32_t w, pad[3];
};
static_assert(sizeof(BlurSlot) % 16 == 0, "row buffers follow the headers at 16-byte alignment");

__device__ __forceinline__ void stg16_blur(void* p, uint4 v) {
    asm volatile("st.global.L1::no_allocate.v4.u32 [%0], {%1,%2,%3,%4};" ::"l"(p), "r"(v.x), "r"(v.y), "r"(v.z),
                 "r"(v.w)
                 : "memory");
}
__device__ __forceinline__ uint32_t smem_addr(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
    asm volatile(
        "{\n.reg .pred p;\nBLUR_WAIT_%=:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@!p bra BLUR_WAIT_%=;\n}" ::"r"(bar), "r"(parity)
        : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
// claim the next tile.  ptxas still gives this atom its warp-aggregated form (a SHFL that waits for the result), but the
// wait falls on the producer lane, one tile ahead of the consumers
__device__ __forceinline__ unsigned int claim_tile(unsigned int* counter) {
    unsigned int v;
    asm volatile("atom.global.add.u32 %0, [%1], 1;" : "=r"(v) : "l"(counter));
    return v;
}

template <int K>  // K == 9: specialised fast path; K == 0: generic odd k
__global__ void __launch_bounds__(32 * (kBlurRowsPerTile + 1), kBlurCtasPerSm) blur_rows_kernel(BlurParams p) {
    extern __shared__ __align__(16) uint8_t smem[];
    BlurSlot* slots = reinterpret_cast<BlurSlot*>(smem);
    uint8_t* bufs = smem + (size_t)p.slots * sizeof(BlurSlot);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int consumers = (int)(blockDim.x >> 5) - 1;  // the last warp is the producer
    if (threadIdx.x == 0) {
        for (int s = 0; s < p.slots; ++s) {
            asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(smem_addr(&slots[s].full)));
            asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(smem_addr(&slots[s].empty)));
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();

    if (warp == consumers) {
        // ---- producer: one lane claims tiles and feeds their rows into the ring in order
        if (lane != 0) return;
        int s = 0;
        uint32_t ph = 0;  // parity of the ring pass the producer is filling
        auto next_slot = [&]() -> BlurSlot& {
            BlurSlot& sl = slots[s];
            mbar_wait(smem_addr(&sl.empty), ph ^ 1u);  // the consumer of the previous pass has freed it
            return sl;
        };
        auto advance = [&]() {
            if (++s == p.slots) { s = 0; ph ^= 1u; }
        };
        unsigned int next = claim_tile(p.counters);
        for (;;) {
            const unsigned int ti = next;
            if (ti >= (unsigned int)p.n_tiles) break;
            next = claim_tile(p.counters);  // in flight while this tile's rows are issued
            const Tile t = p.tiles[ti];
            if (p.opcodes != nullptr && p.opcodes[t.img] != ROD_OP_BLUR) continue;
            const DevImage im = p.images[t.img];
            const int n = 3 * im.w;
            for (int y = t.a; y < t.a + t.b; ++y) {
                const uint8_t* srow = p.src + im.src_off + (int64_t)y * im.src_pitch;
                uint8_t* drow = p.dst + im.dst_off + (int64_t)y * im.dst_pitch;
                const int shift = (int)((uintptr_t)drow & 15);
                const int jf0 = (shift != 0) ? 1 : 0, jf1 = (n + shift) >> 4;
                BlurSlot& sl = next_slot();
                sl.srow = srow;
                sl.drow = drow;
                sl.w = im.w;
                const uint32_t full = smem_addr(&sl.full);
                if (((((uintptr_t)srow ^ (uintptr_t)drow) & 15) == 0) && jf1 > jf0) {
                    const uint32_t bytes = 16u * (uint32_t)(jf1 - jf0);
                    const uint32_t dst_s = smem_addr(bufs + (size_t)s * p.row_buf_bytes + kBlurLeft + 16 * jf0);
                    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(full), "r"(bytes) : "memory");
                    asm volatile(
                        "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst_s),
                        "l"(srow - shift + 16 * jf0), "r"(bytes), "r"(full)
                        : "memory");
                } else {
                    mbar_arrive(full);
                }
                advance();
            }
        }
        // every claim of this CTA is back: count it done; the last CTA to do so returns the pair to 0
        __threadfence();
        if (atomicAdd(p.counters + 1, 1u) == gridDim.x - 1) {
            __threadfence();
            atomicExch(p.counters, 0u);
            atomicExch(p.counters + 1, 0u);
        }
        for (int c = 0; c < consumers; ++c) {  // one "no more rows" per consumer: the next `consumers` slots of the sequence
            BlurSlot& sl = next_slot();
            sl.srow = nullptr;
            mbar_arrive(smem_addr(&sl.full));
            advance();
        }
        return;
    }

    // ---- consumers: warp i takes slots i, i + consumers, ... of the ring
    const int k = (K == 0) ? p.k : K;
    const int halo = 3 * (k >> 1);
    int s = warp;
    uint32_t ph = 0;
    for (;; s += consumers) {
        if (s >= p.slots) { s -= p.slots; ph ^= 1u; }
        BlurSlot& sl = slots[s];
        // A parity wait only tells an mbarrier's current phase from the one before it.  The slot's previous pass may have
        // gone to another consumer (the slot count need not be a multiple of the consumer count), and bulk copies into
        // different slots complete out of order, so its "full" barrier can still be a phase behind: waiting on it directly
        // could return on that stale phase.  The previous pass is over once its consumer has freed the slot ("empty"
        // within one phase of it, since the producer waited for the pass before); only then does "full" mean this pass.
        // The producer waits for the same event before it starts this pass's copy, so this costs no time.
        mbar_wait(smem_addr(&sl.empty), ph ^ 1u);
        mbar_wait(smem_addr(&sl.full), ph);
        const uint8_t* srow = sl.srow;
        if (srow == nullptr) break;
        uint8_t* drow = sl.drow;
        const int w = sl.w;
        uint8_t* buf = bufs + (size_t)s * p.row_buf_bytes;
        const int n = 3 * w;
        const int shift = (int)((uintptr_t)drow & 15);
        uint8_t* row = buf + kBlurLeft + shift;  // byte of pixel 0
        // chunk j covers row positions [16j - shift, 16j - shift + 16); chunks [jf0, jf1) lie fully inside [0, n)
        const int jf0 = (shift != 0) ? 1 : 0;
        const int jf1 = (n + shift) >> 4;
        const bool right_edge = ((n + shift) & 15) != 0;

        // ---- complete the row: smem byte (kBlurLeft + shift + i) = in[i]
        if ((((uintptr_t)srow ^ (uintptr_t)drow) & 15) == 0) {
            // the interior came with the bulk copy; the (at most two) partial chunks: one byte per lane
            const int i = (lane < 16) ? (lane - shift) : (16 * jf1 - shift + lane - 16);
            if (((lane < 16) ? (shift != 0) : right_edge) && i >= 0 && i < n) row[i] = srow[i];
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
                if (w > (k >> 1)) rp = (px < 0) ? -px : 2 * (w - 1) - px;  // single reflection
                else rp = reflect101(px, w);                               // tiny rows: periodic
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
                const uint32_t win[12] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w, c.x, c.y, c.z, c.w};
                uint32_t out[4];
                blur9_chunk16(win, out);
                stg16_blur(dal + 16 * j, make_uint4(out[0], out[1], out[2], out[3]));
            }
            // partial chunks: lane 0 takes the left one, lane 1 the right one
            if (lane < 2 && ((lane == 0) ? (shift != 0) : right_edge)) {
                const int j = (lane == 0) ? 0 : jf1;
                const uint4* wp = reinterpret_cast<const uint4*>(buf + kBlurLeft + 16 * j - 16);
                const uint4 a = wp[0], b = wp[1], c = wp[2];
                const uint32_t win[12] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w, c.x, c.y, c.z, c.w};
                uint32_t out[4];
                blur9_chunk16(win, out);
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
        // the slot's bytes written here (edges, halo) must be ordered before the next bulk copy into it
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        __syncwarp();
        if (lane == 0) mbar_arrive(smem_addr(&sl.empty));
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
    // row slot: kBlurLeft | (shift + 3w rounded up to 16) | 16 (right window) + halo, 16-byte multiple
    const int row_bytes = 3 * plan->max_w;
    p.row_buf_bytes = kBlurLeft + ((15 + row_bytes + 15) & ~15) + 64;
    const size_t slot_bytes = sizeof(BlurSlot) + (size_t)p.row_buf_bytes;
    constexpr size_t kSmem = 227 * 1024, kPerCta = 1024;  // per-SM budget; the runtime reserves 1 KB per CTA
    // up to kBlurMaxSlots slots in a third of the SM; wider rows: at least one slot per consumer warp, down to one slot
    size_t slots = std::min<size_t>(kBlurMaxSlots, (kSmem / kBlurCtasPerSm - kPerCta) / slot_bytes);
    if (slots < (size_t)kBlurRowsPerTile) slots = std::min<size_t>(kBlurRowsPerTile, kSmem / slot_bytes);
    if (slots < 1) return ROD_ERR_UNSUPPORTED;  // a single row does not fit: wider than ~77 000 pixels
    p.slots = (int)slots;
    const int consumers = std::min(kBlurRowsPerTile, p.slots);
    const size_t smem = slots * slot_bytes;
    const int ctas_per_sm = std::max(1, std::min(kBlurCtasPerSm, (int)(kSmem / (smem + kPerCta))));
    p.counters = plan->d_blur_counters + 2 * (plan->launch_seq.fetch_add(1u) & (kCounterRing - 1u));
    const int grid = grid_for(plan, n_tiles, ctas_per_sm);
    const int threads = 32 * (consumers + 1);
    if (k == 9) {
        ROD_CUDA(cudaFuncSetAttribute(blur_rows_kernel<9>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        blur_rows_kernel<9><<<grid, threads, smem, stream>>>(p);
    } else {
        ROD_CUDA(cudaFuncSetAttribute(blur_rows_kernel<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        blur_rows_kernel<0><<<grid, threads, smem, stream>>>(p);
    }
    ROD_CUDA(cudaGetLastError());
    return ROD_OK;
}

}  // namespace rod
