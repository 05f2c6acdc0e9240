// rod_mt.h -- NumPy's legacy normal stream (MT19937 + polar Gaussian), per element, for the device draw of compat noise
// (legacy_rng.cu) and for its sequential CPU replay (tests/emu/legacy_rng_replay.cpp, built with g++ from this header).
//
// Word stream.  The raw MT19937 words x_0, x_1, ... come in blocks of 624: block b is x[624 b, 624 b + 624), block 0 is
// NumPy's `key`.  A candidate of the polar method takes four consecutive words; NumPy's `pos` is the next word of the key.
//
// Jump ahead.  MT19937 is linear over GF(2) with the characteristic polynomial phi of degree 19937.  For a distance D and
// g = x^D mod phi, word j of the window at D is  x_{D+j} = XOR over the set bits i of g of x_{i+j}  (Cayley-Hamilton on
// the 19937-bit state).  Only the top bit of x_0 belongs to the state, so the jumped window is exact for j >= 1 and in
// the top bit of j = 0: a jump lands on the block BEFORE the one wanted, and the wanted block is generated from it.
// phi comes from Berlekamp-Massey over 2 * 19937 output bits, x^D mod phi from carry-less arithmetic (host only, below).
//
// Bit-exactness of the Gaussian: every double operation is an explicit IEEE operation (on the device __dmul_rn & co.,
// so nvcc cannot contract x1 * x1 + x2 * x2 into an FMA; on the host the replay is built with -ffp-contract=off).  Only
// log() may differ from the libm NumPy calls: guard_ok() tells whether the float32 output is the same for every log
// result within a few ulps.
#pragma once
#include <fenv.h>
#include <math.h>
#include <stdint.h>
#include <string.h>

#include <vector>

#ifdef __CUDACC__
#define ROD_MT_HD __host__ __device__ __forceinline__
#else
#define ROD_MT_HD inline
#endif

namespace rodmt {

constexpr int kN = 624, kM = 397;
constexpr int kMexp = 19937;                   // degree of phi
constexpr int kPolyWords = (kMexp + 63) / 64;  // 312 uint64 words of a polynomial of degree < 19937
constexpr int kWinBlocks = 33;                 // the words x_0 .. x_{19937 + 623} a jump correlates, in whole blocks
constexpr int kCandPerBlock = kN / 4;          // 156 candidates start in every block
constexpr uint32_t kMatrixA = 0x9908b0dfu, kUpper = 0x80000000u, kLower = 0x7fffffffu;

ROD_MT_HD uint32_t twist(uint32_t a, uint32_t b) {
    const uint32_t y = (a & kUpper) | (b & kLower);
    return (y >> 1) ^ ((0u - (y & 1u)) & kMatrixA);
}
ROD_MT_HD uint32_t temper(uint32_t y) {
    y ^= y >> 11;
    y ^= (y << 7) & 0x9d2c5680u;
    y ^= (y << 15) & 0xefc60000u;
    y ^= y >> 18;
    return y;
}
// Word i of the block after `old`.  It reads nw[i - 227] (i >= 227) and nw[0] (i = 623), so a block is generated in
// three phases, i in [0, 227), [227, 454), [454, 624): gen_phase(i).
ROD_MT_HD uint32_t next_word(const uint32_t* old, const uint32_t* nw, int i) {
    if (i < kN - kM) return old[i + kM] ^ twist(old[i], old[i + 1]);
    if (i < kN - 1) return nw[i - (kN - kM)] ^ twist(old[i], old[i + 1]);
    return nw[kM - 1] ^ twist(old[kN - 1], nw[0]);
}
ROD_MT_HD int gen_phase(int i) { return i < kN - kM ? 0 : (i < 2 * (kN - kM) ? 1 : 2); }

// Word j of the window g(A) x0, w = x_0 .. x_{19936 + 623} generated from x0.
ROD_MT_HD uint32_t jump_word(const uint64_t* g, const uint32_t* w, int j) {
    uint32_t acc = 0;
    for (int k = 0; k < kPolyWords; ++k) {
        uint64_t bits = g[k];
        const uint32_t* wk = w + 64 * k + j;
        while (bits) {
#ifdef __CUDA_ARCH__
            const int b = __ffsll((long long)bits) - 1;
#else
            const int b = __builtin_ctzll(bits);
#endif
            acc ^= wk[b];
            bits &= bits - 1;
        }
    }
    return acc;
}

// One candidate from four raw words: mt19937_next_double twice, then 2d - 1 and r2 = x1 x1 + x2 x2 (legacy_gauss).
struct Cand {
    double x1, x2, r2;
};
ROD_MT_HD double dmul(double a, double b) {
#ifdef __CUDA_ARCH__
    return __dmul_rn(a, b);
#else
    return a * b;
#endif
}
ROD_MT_HD double dadd(double a, double b) {
#ifdef __CUDA_ARCH__
    return __dadd_rn(a, b);
#else
    return a + b;
#endif
}
ROD_MT_HD double ddiv(double a, double b) {
#ifdef __CUDA_ARCH__
    return __ddiv_rn(a, b);
#else
    return a / b;
#endif
}
ROD_MT_HD double dsqrt(double a) {
#ifdef __CUDA_ARCH__
    return __dsqrt_rn(a);
#else
    return sqrt(a);
#endif
}
ROD_MT_HD double next_double(uint32_t w0, uint32_t w1) {
    const int32_t a = (int32_t)(temper(w0) >> 5), b = (int32_t)(temper(w1) >> 6);
    return ddiv(dadd(dmul((double)a, 67108864.0), (double)b), 9007199254740992.0);
}
ROD_MT_HD Cand candidate(uint32_t w0, uint32_t w1, uint32_t w2, uint32_t w3) {
    Cand c;
    c.x1 = dadd(dmul(2.0, next_double(w0, w1)), -1.0);
    c.x2 = dadd(dmul(2.0, next_double(w2, w3)), -1.0);
    c.r2 = dadd(dmul(c.x1, c.x1), dmul(c.x2, c.x2));
    return c;
}
ROD_MT_HD bool accepted(double r2) { return !(r2 >= 1.0 || r2 == 0.0); }
// f = sqrt(-2 log(r2) / r2) from a given log(r2); the pair's outputs are 0.0 + sigma (f x2) first, 0.0 + sigma (f x1)
// second (the addition turns sigma = 0's -0.0 into +0.0, as NumPy's does)
ROD_MT_HD double polar_f(double lg, double r2) { return dsqrt(ddiv(dmul(-2.0, lg), r2)); }
ROD_MT_HD double polar_out(double sigma, double f, double x) { return dadd(0.0, dmul(sigma, dmul(f, x))); }

// True when float(y') == float(y) for every y' within |y| 2^-46 of y: the bounds y -+ |y| 2^-46, rounded down and up,
// convert to the same float32.  A log() result within 2 ulps of the correctly rounded one moves y by less than 2^-49 |y|
// through the division, the sqrt and the two products, so an unflagged y has the float32 NumPy produces whatever log
// returned.  Float rounding is monotone, so the comparison also covers subnormal results and overflow to infinity.
ROD_MT_HD bool guard_ok(double y) {
    const double e = fabs(y) * 0x1p-46;  // exact (a power-of-two scaling)
#ifdef __CUDA_ARCH__
    return __double2float_rn(__dadd_rd(y, -e)) == __double2float_rn(__dadd_ru(y, e));
#else
    const int mode = fegetround();
    fesetround(FE_DOWNWARD);
    volatile double lo = y - e;
    fesetround(FE_UPWARD);
    volatile double hi = y + e;
    fesetround(mode);
    return (float)lo == (float)hi;
#endif
}

// ---- host only: the jump polynomials ------------------------------------------------------------------------------

// The raw words x_0 .. x_{n-1} from the block `key` (x_0 = key[0]).
inline void words_from(const uint32_t* key, uint32_t* x, size_t n) {
    const size_t blocks = (n + kN - 1) / kN;
    std::vector<uint32_t> buf((blocks + 1) * kN);
    memcpy(buf.data(), key, sizeof(uint32_t) * kN);
    for (size_t b = 1; b < blocks; ++b)
        for (int i = 0; i < kN; ++i) buf[b * kN + i] = next_word(&buf[(b - 1) * kN], &buf[b * kN], i);
    memcpy(x, buf.data(), sizeof(uint32_t) * n);
}

// phi from Berlekamp-Massey over the top bits of 2 * 19937 words of a seeded generator.  Returns its degree; phi gets
// kPolyWords + 1 words, bit k = coefficient of x^k.
inline int characteristic_polynomial(std::vector<uint64_t>& phi) {
    const int n = 2 * kMexp;
    uint32_t key[kN];
    key[0] = 5489u;  // init_genrand(5489): any state not in the zero orbit will do
    for (int i = 1; i < kN; ++i) key[i] = 1812433253u * (key[i - 1] ^ (key[i - 1] >> 30)) + (uint32_t)i;
    std::vector<uint32_t> x(n);
    words_from(key, x.data(), n);
    const int words = n / 64 + 2;
    std::vector<uint64_t> rev(words + 1, 0), C(words, 0), B(words, 0), T;
    for (int k = 0; k < n; ++k)  // rev bit (n - 1 - k) = s_k, so s_{t-i} for i = 0, 1, ... are consecutive bits from n - 1 - t
        if (x[k] >> 31) rev[(n - 1 - k) >> 6] |= 1ull << ((n - 1 - k) & 63);
    auto bits64 = [&](int pos) {
        const int q = pos >> 6, r = pos & 63;
        return r ? (rev[q] >> r) | (rev[q + 1] << (64 - r)) : rev[q];
    };
    C[0] = B[0] = 1;
    int L = 0, m = 1;
    for (int t = 0; t < n; ++t) {
        uint64_t acc = 0;  // d = sum_{i=0..L} C_i s_{t-i}
        for (int k = 0; k <= L / 64; ++k) acc ^= C[k] & bits64(n - 1 - t + 64 * k);
        if (!(__builtin_popcountll(acc) & 1)) {
            ++m;
            continue;
        }
        const bool grow = 2 * L <= t;
        if (grow) T = C;
        const int q = m >> 6, r = m & 63;  // C += x^m B
        for (int k = words - 1; k >= q; --k) {
            uint64_t v = B[k - q] << r;
            if (r && k - q - 1 >= 0) v |= B[k - q - 1] >> (64 - r);
            C[k] ^= v;
        }
        if (grow) {
            L = t + 1 - L;
            B = T;
            m = 1;
        } else {
            ++m;
        }
    }
    phi.assign(kPolyWords + 1, 0);
    for (int i = 0; i <= L; ++i)  // phi(x) = x^L C(1/x)
        if ((C[i >> 6] >> (i & 63)) & 1) phi[(L - i) >> 6] |= 1ull << ((L - i) & 63);
    return L;
}

// Multiplication by x^k (k <= 64) modulo phi, with the top k bits folded back through byte tables:
// tab[8 * 256 * q + v] (kPolyWords words each) = v(x) x^(19937 + 8 q) mod phi.
struct PolyMod {
    std::vector<uint64_t> tab;
    explicit PolyMod(const std::vector<uint64_t>& phi) : tab((size_t)8 * 256 * kPolyWords, 0) {
        std::vector<uint64_t> p(phi.begin(), phi.begin() + kPolyWords);  // x^19937 mod phi = phi - x^19937
        p[kPolyWords - 1] &= (1ull << (kMexp - 64 * (kPolyWords - 1))) - 1;
        const uint64_t* low = p.data();
        std::vector<uint64_t> xb(64 * (size_t)kPolyWords);  // x^(19937 + b) mod phi, b < 64
        memcpy(&xb[0], low, sizeof(uint64_t) * kPolyWords);
        for (int b = 1; b < 64; ++b) {
            uint64_t* dst = &xb[(size_t)b * kPolyWords];
            const uint64_t* src = &xb[(size_t)(b - 1) * kPolyWords];
            const bool top = (src[kPolyWords - 1] >> (kMexp - 1 - 64 * (kPolyWords - 1))) & 1;
            for (int k = kPolyWords - 1; k > 0; --k) dst[k] = (src[k] << 1) | (src[k - 1] >> 63);
            dst[0] = src[0] << 1;
            dst[kPolyWords - 1] &= (1ull << (kMexp - 64 * (kPolyWords - 1))) - 1;
            if (top)
                for (int k = 0; k < kPolyWords; ++k) dst[k] ^= low[k];
        }
        for (int q = 0; q < 8; ++q)
            for (int v = 1; v < 256; ++v) {
                uint64_t* dst = &tab[((size_t)256 * q + v) * kPolyWords];
                for (int b = 0; b < 8; ++b)
                    if ((v >> b) & 1)
                        for (int k = 0; k < kPolyWords; ++k) dst[k] ^= xb[(size_t)(8 * q + b) * kPolyWords + k];
            }
    }
    // a := a x^k mod phi, 1 <= k <= 64
    void mulx(uint64_t* a, int k) const {
        constexpr int kTop = kMexp - 64 * (kPolyWords - 1);  // 33 bits used in the last word
        // the k bits that pass x^19937: bits [19937 - k, 19937) of a
        const int lo = kMexp - k;
        const int q = lo >> 6, r = lo & 63;
        uint64_t over = a[q] >> r;
        if (r && q + 1 < kPolyWords) over |= a[q + 1] << (64 - r);
        if (k < 64) over &= (1ull << k) - 1;
        const int wq = k >> 6, wr = k & 63;  // shift left by k
        for (int i = kPolyWords - 1; i >= 0; --i) {
            uint64_t v = i - wq >= 0 ? a[i - wq] << wr : 0;
            if (wr && i - wq - 1 >= 0) v |= a[i - wq - 1] >> (64 - wr);
            a[i] = v;
        }
        a[kPolyWords - 1] &= (1ull << kTop) - 1;
        for (int byte = 0; byte < 8 && over; ++byte, over >>= 8) {
            const uint64_t* t = &tab[((size_t)256 * byte + (over & 255)) * kPolyWords];
            for (int i = 0; i < kPolyWords; ++i) a[i] ^= t[i];
        }
    }
    // a := a x^d mod phi
    void mulx_pow(uint64_t* a, uint64_t d) const {
        for (; d >= 64; d -= 64) mulx(a, 64);
        if (d) mulx(a, (int)d);
    }
};

// The jump of chunk c of the device draw (legacy_rng.cu): chunk c >= 1 starts at block c * stride, reached by a jump to
// block c * stride - 1 (distance (c * stride - 1) * 624 words) and one generated block.  table gets kPolyWords words per
// chunk c = 0 .. n - 1 (row 0 unused) and is extended from its present size.
inline void extend_jump_table(std::vector<uint64_t>& table, const PolyMod& pm, int stride, int n) {
    int have = (int)(table.size() / kPolyWords);
    if (have >= n) return;
    table.resize((size_t)n * kPolyWords, 0);
    if (n <= 1) return;
    std::vector<uint64_t> g(kPolyWords, 0);
    if (have <= 1) {
        have = 1;
        g[0] = 1;  // x^0
        pm.mulx_pow(g.data(), (uint64_t)(stride - 1) * kN);
    } else {
        memcpy(g.data(), &table[(size_t)(have - 1) * kPolyWords], sizeof(uint64_t) * kPolyWords);
        pm.mulx_pow(g.data(), (uint64_t)stride * kN);
    }
    for (int c = have;; ++c) {
        memcpy(&table[(size_t)c * kPolyWords], g.data(), sizeof(uint64_t) * kPolyWords);
        if (c + 1 == n) break;
        pm.mulx_pow(g.data(), (uint64_t)stride * kN);
    }
}

}  // namespace rodmt
