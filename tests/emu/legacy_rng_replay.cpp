// Sequential CPU replay of the device draw of compat noise (csrc/legacy_rng.cu), built with g++ from the same rod_mt.h:
// rounds, chunks reached by jumps, per-chunk counts, the prefix over chunks, the write pass and the end state, with the
// chunk stride and the chunks per round as parameters so that small counts cross many chunk and round boundaries.
#include <math.h>
#include <stdint.h>
#include <string.h>

#include <algorithm>
#include <vector>

#include "../../robust-object-detection_b200/csrc/rod_mt.h"

using namespace rodmt;

namespace {
const PolyMod& polymod() {
    static PolyMod* pm = nullptr;
    if (!pm) {
        std::vector<uint64_t> phi;
        characteristic_polynomial(phi);
        pm = new PolyMod(phi);
    }
    return *pm;
}
// block `c stride` from block 0 = key, as legacy_count_kernel reaches it
void chunk_start(const uint32_t* key, const uint64_t* g, uint32_t* out) {
    std::vector<uint32_t> w((size_t)kWinBlocks * kN);
    memcpy(w.data(), key, sizeof(uint32_t) * kN);
    for (int b = 1; b < kWinBlocks; ++b)
        for (int i = 0; i < kN; ++i) w[(size_t)b * kN + i] = next_word(&w[(size_t)(b - 1) * kN], &w[(size_t)b * kN], i);
    uint32_t win[kN];
    for (int j = 0; j < kN; ++j) win[j] = jump_word(g, w.data(), j);
    for (int i = 0; i < kN; ++i) out[i] = next_word(win, out, i);
}
void gen(const uint32_t* old, uint32_t* nw) {
    for (int i = 0; i < kN; ++i) nw[i] = next_word(old, nw, i);
}
}  // namespace

extern "C" {

int replay_phi_degree() {
    std::vector<uint64_t> phi;
    return characteristic_polynomial(phi);
}

// Window at distance d words from block 0 = key (word 0 exact in its top bit only), and the block `blocks` reached as a
// chunk start (jump to blocks - 1, then one generated block).
void replay_jump(const uint32_t* key, uint64_t d, uint32_t* window, int blocks, uint32_t* block) {
    std::vector<uint64_t> g(kPolyWords, 0);
    g[0] = 1;
    polymod().mulx_pow(g.data(), d);
    std::vector<uint32_t> w((size_t)kWinBlocks * kN);
    words_from(key, w.data(), w.size());
    for (int j = 0; j < kN; ++j) window[j] = jump_word(g.data(), w.data(), j);
    if (blocks > 0) {
        g.assign(kPolyWords, 0);
        g[0] = 1;
        polymod().mulx_pow(g.data(), (uint64_t)(blocks - 1) * kN);
        chunk_start(key, g.data(), block);
    }
}

// The table rows of legacy_rng.cu for a stride: row c = x^((c stride - 1) 624) mod phi
void replay_table_row(int stride, int c, uint64_t* row) {
    std::vector<uint64_t> t;
    extend_jump_table(t, polymod(), stride, c + 1);
    memcpy(row, &t[(size_t)c * kPolyWords], sizeof(uint64_t) * kPolyWords);
}

// rod_numpy_legacy_normal_f32_device restated sequentially; returns the number of flagged values
int replay_normal(uint32_t* key, int32_t* pos, int32_t* has_gauss, double* cached, double sigma, uint64_t n, float* out,
                  int stride, int max_chunks) {
    std::vector<uint64_t> table;
    uint64_t done = 0;
    int flagged = 0;
    if (n > 0 && *has_gauss) {
        out[done++] = (float)(0.0 + sigma * *cached);
        *has_gauss = 0;
        *cached = 0.0;
    }
    while (done < n) {
        const uint64_t n_vals = n - done, need = (n_vals + 1) / 2;
        const uint64_t cand = (uint64_t)ceil((double)need * 1.2732395447351628) + 8 * (uint64_t)ceil(sqrt((double)need)) + 64;
        uint64_t b_end = ((uint64_t)*pos + 4 * cand + kN - 1) / kN;
        const int n_chunks = (int)std::min<uint64_t>((b_end + stride - 1) / stride, (uint64_t)max_chunks);
        b_end = std::min<uint64_t>(b_end, (uint64_t)n_chunks * stride);
        extend_jump_table(table, polymod(), stride, n_chunks);
        const int p = *pos;
        std::vector<uint32_t> starts((size_t)n_chunks * kN);
        std::vector<uint64_t> counts(n_chunks, 0);
        uint32_t buf[2][kN];
        auto cand_at = [&](const uint32_t* cur, const uint32_t* nxt, uint64_t b, int t, int* o, Cand* cd) {
            *o = (p & 3) + 4 * t;
            if (b == 0 && *o < p) return false;
            uint32_t w[4];
            for (int k = 0; k < 4; ++k) w[k] = *o + k < kN ? cur[*o + k] : nxt[*o + k - kN];
            *cd = candidate(w[0], w[1], w[2], w[3]);
            return accepted(cd->r2);
        };
        for (int c = 0; c < n_chunks; ++c) {  // legacy_count_kernel
            if (c == 0) memcpy(buf[0], key, sizeof(buf[0]));
            else chunk_start(key, &table[(size_t)c * kPolyWords], buf[0]);
            memcpy(&starts[(size_t)c * kN], buf[0], sizeof(buf[0]));
            int k = 0;
            for (uint64_t b = (uint64_t)c * stride; b < std::min<uint64_t>((uint64_t)(c + 1) * stride, b_end); ++b, k ^= 1) {
                gen(buf[k], buf[k ^ 1]);
                for (int t = 0; t < kCandPerBlock; ++t) {
                    int o;
                    Cand cd;
                    counts[c] += cand_at(buf[k], buf[k ^ 1], b, t, &o, &cd);
                }
            }
        }
        uint64_t all = 0;
        for (uint64_t v : counts) all += v;
        uint64_t rank = 0, end_word = 0;
        bool found = false;
        Cand last{};
        for (int c = 0; c < n_chunks && !found; ++c) {  // legacy_write_kernel
            memcpy(buf[0], &starts[(size_t)c * kN], sizeof(buf[0]));
            int k = 0;
            const uint64_t b_hi = std::min<uint64_t>((uint64_t)(c + 1) * stride, b_end);
            for (uint64_t b = (uint64_t)c * stride; b < b_hi && !found; ++b, k ^= 1) {
                gen(buf[k], buf[k ^ 1]);
                for (int t = 0; t < kCandPerBlock; ++t) {
                    int o;
                    Cand cd;
                    if (cand_at(buf[k], buf[k ^ 1], b, t, &o, &cd) && rank < need) {
                        const double f = polar_f(log(cd.r2), cd.r2);
                        const double y0 = polar_out(sigma, f, cd.x2), y1 = polar_out(sigma, f, cd.x1);
                        out[done + 2 * rank] = (float)y0;
                        flagged += !guard_ok(y0);
                        if (2 * rank + 1 < n_vals) {
                            out[done + 2 * rank + 1] = (float)y1;
                            flagged += !guard_ok(y1);
                        }
                        if (++rank == need) {
                            found = true;
                            last = cd;
                            end_word = b * kN + o + 3;
                            break;
                        }
                    }
                    if (all < need && c == n_chunks - 1 && b == b_hi - 1 && t == kCandPerBlock - 1) end_word = b * kN + o + 3;
                }
                if (found || (all < need && c == n_chunks - 1 && b == b_hi - 1)) {
                    const uint64_t blk = end_word / kN;
                    memcpy(key, blk == b ? buf[k] : buf[k ^ 1], sizeof(buf[0]));
                    *pos = (int32_t)(end_word - blk * kN + 1);
                }
            }
        }
        if (found && (n_vals & 1)) {
            *has_gauss = 1;
            *cached = sqrt(-2.0 * log(last.r2) / last.r2) * last.x1;
        }
        done += std::min<uint64_t>(2 * std::min(all, need), n_vals);
    }
    return flagged;
}

// The guard against a log() off by up to 2 ulps: over the first n_cand candidates from `key`, every output whose float32
// changes when log(r2) is replaced by a neighbour up to 2 ulps away must be flagged.  Returns the unflagged changes;
// *changed and *flagged count all changes and all flags.
int replay_guard_ok(double y) { return guard_ok(y); }

int replay_guard(const uint32_t* key, uint64_t n_cand, double sigma, uint64_t* changed, uint64_t* flagged) {
    std::vector<uint32_t> x(4 * n_cand + 4);
    words_from(key, x.data(), x.size());
    int missed = 0;
    *changed = *flagged = 0;
    for (uint64_t i = 0; i < n_cand; ++i) {
        const Cand cd = candidate(x[4 * i], x[4 * i + 1], x[4 * i + 2], x[4 * i + 3]);
        if (!accepted(cd.r2)) continue;
        const double lg = log(cd.r2);
        const double f = polar_f(lg, cd.r2);
        for (double xv : {cd.x2, cd.x1}) {
            const double y = polar_out(sigma, f, xv);
            const bool ok = guard_ok(y);
            *flagged += !ok;
            double alt[4] = {nextafter(lg, -INFINITY), nextafter(lg, INFINITY), 0, 0};
            alt[2] = nextafter(alt[0], -INFINITY);
            alt[3] = nextafter(alt[1], INFINITY);
            bool ch = false;
            for (double l : alt) ch |= (float)polar_out(sigma, polar_f(l, cd.r2), xv) != (float)y;
            *changed += ch;
            missed += ch && ok;
        }
    }
    return missed;
}
}

// libm log() element-wise: the function NumPy's legacy_gauss calls
extern "C" void replay_log(const double* x, double* y, uint64_t n) {
    for (uint64_t i = 0; i < n; ++i) y[i] = log(x[i]);
}
