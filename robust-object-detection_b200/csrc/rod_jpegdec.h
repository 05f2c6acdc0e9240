// rod_jpegdec.h -- arithmetic of a baseline JPEG decoder whose pixels equal cv2.imread's, written once for device and host.
//
// SURVEY 8f rank 1, the other half: scripts/build_corrupted_testsets.py reads every source frame with cv2.imread (:109 / :149).
// OpenCV 4.13.0 decodes with libjpeg-turbo 3.1.2 and its defaults: JDCT_ISLOW, fancy (triangle) chroma upsampling, output
// colour space BGR.  The integer algorithms restated here (published in the IJG / libjpeg-turbo sources, whose SIMD paths are
// bit-identical to their C paths for in-range data):
//   jdhuff.c   decode_mcu            canonical Huffman decoding, receive / extend, DC prediction per component
//   jidctint.c jpeg_idct_islow       13-bit fixed-point 8x8 inverse DCT (dequantisation folded in), range limit to 0..255
//   jdsample.c h2v2_fancy_upsample   chroma: 3/4 - 1/4 triangle filter in both axes, roundings 8 / 7 alternating by column
//   jdmainct.c context rows          above the first / below the last REAL chroma row the nearest real row is used
//   jdcolor.c  ycc_rgb_convert       16-bit fixed-point YCbCr -> RGB (written out as BGR)
//              h2v1_fancy_upsample   4:2:2 files: the same filter along the row only, roundings 1 / 2
// Supported layouts: baseline sequential (SOF0), 8 bit, one scan (with or without restart markers), either Y Cb Cr with the luma
// sampled 2x2 (4:2:0, what OpenCV itself writes), 2x1 (4:2:2) or 1x1 (4:4:4) against 1x1 chroma, or greyscale; and, when
// the caller asks for them, progressive (SOF2) files of the same layouts (jdphuff.c, below).  Anything else is reported as
// unsupported by the parser and the caller keeps the host codec for that file.
// The same functions are compiled into tests/emu (CPU check against cv2.imdecode) and into jpegdec.cu.
#pragma once
#include <stdint.h>

#include "rod_jpeg.h"   // RJ_HD, natural_order, Geometry

namespace rod {
namespace jpegdec {

constexpr int kLook = 10;   // bits of the first-level Huffman lookup (jdhuff.h uses 8; a wider table only saves slow-path steps)

// jdhuff.c jpeg_make_d_derived_tbl: one Huffman table in decoding form.
struct HuffTab {
    uint16_t look[1 << kLook];   // index = next kLook bits: (code length << 8) | symbol for codes of <= kLook bits, else 0
    int32_t maxcode[18];         // largest code of length l (-1: none); [17] = sentinel that ends the slow loop
    int32_t valoffset[17];       // huffval index of a code of length l = code + valoffset[l]
    uint8_t huffval[256];
};

// Everything of a file's DQT / DHT / SOF / SOS that the decoder needs; files written by the same encoder share one set.
struct TableSet {
    HuffTab dc[2], ac[2];
    uint16_t quant[3][64];       // per component, natural order
    uint8_t comp_dc[3], comp_ac[3];
    uint8_t pad[10];             // sizeof % 16 == 0: the quantisation tables of every set are read as 16-byte words
};
static_assert(sizeof(TableSet) % 16 == 0, "TableSet must keep 16-byte alignment in arrays");

// One image of a batch.  Offsets are bytes from the decoder's device buffers; the stream is the entropy-coded segment
// with the 0xFF00 stuffing removed, starting at a 4-byte aligned offset and followed by >= 16 zero bytes.
struct ImageRec {
    int32_t h, w;
    int32_t table_set;
    uint32_t stream_bytes;
    uint64_t stream_off;
    uint64_t coef_off;           // int16 units: Y blocks [vs mcu_h][hs mcu_w][64], then Cb [mcu_h][mcu_w][64], then Cr
    uint64_t plane_off;          // bytes: Y plane [8 vs mcu_h][8 hs mcu_w], then Cb [8 mcu_h][8 mcu_w], then Cr
    uint64_t dst_off;            // bytes into the caller's pixel buffer (HWC BGR)
    int64_t dst_pitch;
    uint8_t hs, vs;              // luma sampling factors (chroma: 1 x 1); greyscale: 1, 1
    uint8_t ncomp;               // 3 or 1
    uint8_t pad[5];
};

// MCU geometry of an image: an MCU is hs x vs luma blocks followed by one Cb and one Cr block (greyscale: one block).
struct Layout {
    int hs, vs, nl, nb;          // nl = hs * vs luma blocks, nb blocks per MCU
    int mcu_w, mcu_h;
    long mcus;
};
RJ_HD Layout layout_of(const ImageRec& im) {
    Layout L;
    L.hs = im.hs; L.vs = im.vs;
    L.nl = L.hs * L.vs;
    L.nb = L.nl + (im.ncomp == 3 ? 2 : 0);
    L.mcu_w = (im.w + 8 * L.hs - 1) / (8 * L.hs);
    L.mcu_h = (im.h + 8 * L.vs - 1) / (8 * L.vs);
    L.mcus = (long)L.mcu_w * L.mcu_h;
    return L;
}

// One restart interval of an image's scan (a scan without restart markers is one segment).  Its entropy-coded bytes sit
// at byte stream_off + byte0 of the stream buffer, stream_off 4-byte aligned (the reader loads words), so bit positions
// count from stream_off and the segment starts at bit 8 * byte0.  The DC predictions start from 0 in every segment.
struct SegRec {
    uint64_t stream_off;
    uint32_t image;
    uint32_t byte0;              // 0..3
    uint32_t stream_bytes;       // byte0 + length of the segment: the bytes a reader may use, counted from stream_off
    uint32_t first_block;        // global block index (MCU order) of the segment's first block
    uint32_t n_blocks;
    uint32_t pad;
};

// MSB-first reader over the unstuffed stream, 32 bits at a time.
struct BitReader {
    const uint32_t* words;
    uint32_t next;               // index of the next word to load
    uint32_t limit;              // words that may be read (the stream and its zero padding); beyond, zeros are supplied
    uint64_t acc;                // valid bits at the top
    int n;                       // number of valid bits
    RJ_HD void init(const uint8_t* stream, uint32_t stream_bytes) {
        words = reinterpret_cast<const uint32_t*>(stream);
        next = 0; acc = 0; n = 0;
        limit = (stream_bytes + 3u) / 4u + 2u;
    }
    RJ_HD void refill() {        // afterwards n >= 32: enough for the longest code (16) plus the longest value (16)
        if (n < 32) {
            uint32_t w = 0u;
            if (next < limit) {
#if defined(__CUDA_ARCH__)
                w = __byte_perm(__ldg(words + next), 0u, 0x0123);
#else
                const uint8_t* b = reinterpret_cast<const uint8_t*>(words + next);
                w = ((uint32_t)b[0] << 24) | ((uint32_t)b[1] << 16) | ((uint32_t)b[2] << 8) | b[3];
#endif
            }
            ++next;
            acc |= (uint64_t)w << (32 - n);
            n += 32;
        }
    }
    RJ_HD void init_at(const uint8_t* stream, uint32_t stream_bytes, uint32_t bit) {   // start at an arbitrary bit position
        init(stream, stream_bytes);
        next = bit >> 5;
        refill();
        skip((int)(bit & 31u));
    }
    RJ_HD uint32_t pos() const { return 32u * next - (uint32_t)n; }   // bit position of the next unread bit
    RJ_HD uint32_t peek(int k) const { return (uint32_t)(acc >> (64 - k)); }   // 1 <= k <= 32
    RJ_HD void skip(int k) { acc <<= k; n -= k; }
    RJ_HD uint64_t bits_used() const { return 32ull * next - (uint64_t)n; }
};

// one Huffman symbol; returns -1 on a code that is not in the table
RJ_HD int decode_symbol(BitReader& br, const HuffTab& t) {
    const uint32_t e = t.look[br.peek(kLook)];   // (the device keeps the tables in shared memory)
    if (e != 0u) {
        br.skip((int)(e >> 8));
        return (int)(e & 255u);
    }
    int l = kLook + 1;
    int32_t code = (int32_t)br.peek(l);
    while (code > t.maxcode[l]) {
        ++l;
        code = (int32_t)br.peek(l);
    }
    if (l > 16) {   // not a code of this table: corrupt data (or a speculative start inside a symbol, see decode_span)
        br.skip(16);
        return -1;
    }
    br.skip(l);
    return t.huffval[(code + t.valoffset[l]) & 255];
}

// jdhuff.c HUFF_EXTEND: the s-bit field v as a signed value
RJ_HD int extend(uint32_t v, int s) { return v < (1u << (s - 1)) ? (int)v - (1 << s) + 1 : (int)v; }

// One block: coefficients (as stored in the file: quantised) into natural order.  blk must be zero-initialised;
// nat[64]: zigzag position -> natural index (rod::jpeg::natural_order as a table).
// Returns false on a corrupt stream.
RJ_HD bool decode_block(BitReader& br, const HuffTab& dc, const HuffTab& ac, const uint8_t* nat, int* last_dc, int16_t* blk) {
    br.refill();
    int s = decode_symbol(br, dc);
    if (s < 0 || s > 16) return false;
    if (s) {
        br.refill();
        const uint32_t v = br.peek(s);
        br.skip(s);
        *last_dc += extend(v, s);
    }
    blk[0] = (int16_t)*last_dc;
    for (int k = 1; k < 64; ++k) {
        br.refill();
        const int sym = decode_symbol(br, ac);
        if (sym < 0) return false;
        const int r = sym >> 4;
        s = sym & 15;
        if (s) {
            k += r;
            if (k > 63) return false;
            const uint32_t v = br.peek(s);
            br.skip(s);
            blk[nat[k]] = (int16_t)extend(v, s);
        } else {
            if (r != 15) break;
            k += 15;
        }
    }
    return true;
}

// The whole scan of one image, sequentially, segment by segment (reference for the parallel passes below; CPU replay
// only).  coef: this image's zeroed coefficient area.  Returns 0, or 1 (corrupt code), 2 (ran past the end of a segment).
RJ_HD int16_t* block_of(int16_t* coef, const Layout& L, uint32_t g);
RJ_HD int decode_scan(const ImageRec& im, const SegRec* segs, int n_segs, const TableSet& ts, const uint8_t* nat,
                      const uint8_t* streams, int16_t* coef) {
    const Layout L = layout_of(im);
    for (int q = 0; q < n_segs; ++q) {
        const SegRec& sg = segs[q];
        BitReader br;
        br.init_at(streams + sg.stream_off, sg.stream_bytes, 8u * sg.byte0);
        int last_dc[3] = {0, 0, 0};
        for (uint32_t g = sg.first_block; g < sg.first_block + sg.n_blocks; ++g) {
            const int b = (int)(g % (uint32_t)L.nb), comp = b < L.nl ? 0 : b - L.nl + 1;
            if (!decode_block(br, ts.dc[ts.comp_dc[comp]], ts.ac[ts.comp_ac[comp]], nat, &last_dc[comp], block_of(coef, L, g))) return 1;
        }
        if (br.bits_used() > 8ull * sg.stream_bytes) return 2;
    }
    return 0;
}

// ---- parallel decoding of one scan (device: jpegdec.cu; CPU replay: tests/emu) ---------------------------------------
// A baseline scan without restart markers is one serial bit stream, but Huffman codes resynchronise: a decoder started at
// a wrong bit position / block position falls into step with the true symbol sequence after a few symbols, with high
// probability (the self-synchronisation used by Weissenberger & Schmidt's GPU Huffman / JPEG decoders).  The stream is cut
// into SUBSEQUENCES of kSubBits bits; subsequence s owns the symbols that START in [s kSubBits, (s + 1) kSubBits).
//   state of a decoder between two symbols: (bit position p, zigzag index k of the next coefficient -- 0: a DC symbol is
//   next --, block b of the MCU 0 .. nb - 1), packed with the number of blocks completed into one 64-bit word;
//   E[s] = end state of subsequence s = F_s(start state), where the start state of s is E[s - 1] (s = 0: the scan's start).
// With restart markers every interval (SegRec) is such a stream of its own with an exactly known start.
// Round 0 guesses every start state as (s kSubBits, 0, 0); later rounds re-decode the subsequences whose predecessor's end
// state changed, until a whole round changes nothing: then E[s] = F_s(E[s - 1]) for every s with E[0] exact, i.e. every end
// state is the sequential decoder's (induction over s).  A scan over the block counts gives every subsequence its first
// block; a last pass decodes from the exact states and writes the coefficients (DC differences; the prediction is a
// prefix sum per component afterwards).
constexpr uint32_t kSubBits = 1024;
RJ_HD uint64_t span_state(uint32_t p, uint32_t nblk, int k, int b) {
    return (uint64_t)p | ((uint64_t)(nblk & 0xFFFFu) << 32) | ((uint64_t)(uint32_t)k << 48) | ((uint64_t)(uint32_t)b << 56);
}
RJ_HD uint32_t state_p(uint64_t e) { return (uint32_t)e; }
RJ_HD uint32_t state_nblk(uint64_t e) { return (uint32_t)(e >> 32) & 0xFFFFu; }
RJ_HD int state_k(uint64_t e) { return (int)((e >> 48) & 0xFFu); }
RJ_HD int state_b(uint64_t e) { return (int)(e >> 56); }
// the part of a state a successor starts from (the block count belongs to the subsequence that produced it)
RJ_HD uint64_t state_start(uint64_t e) { return e & 0xFFFF0000FFFFFFFFull; }

// coefficient block of global block index g (MCU g / nb, block g % nb) inside an image's coefficient area
RJ_HD int16_t* block_of(int16_t* coef, const Layout& L, uint32_t g) {
    const uint32_t mcu = g / (uint32_t)L.nb, b = g - (uint32_t)L.nb * mcu;
    if ((int)b < L.nl) {
        const uint32_t my = mcu / (uint32_t)L.mcu_w, mx = mcu - my * (uint32_t)L.mcu_w;
        const uint32_t by = b / (uint32_t)L.hs, bx = b - by * (uint32_t)L.hs;
        return coef + 64L * ((long)(L.vs * my + by) * (L.hs * L.mcu_w) + L.hs * mx + bx);
    }
    return coef + 64L * (L.nl * L.mcus + (long)((int)b - L.nl) * L.mcus + mcu);
}

// Decodes the symbols that start in [start.p, boundary) from decoder state `start`; returns the end state.  WRITE: also
// stores the coefficients (DC: the difference) from global block g0 on, stops behind block total_blocks - 1 (the segment's
// last block) and reports
// corrupt data in *err.
template <bool WRITE>
RJ_HD uint64_t decode_span(const Layout& L, uint32_t stream_bytes, const TableSet& ts, const uint8_t* nat, const uint8_t* stream, uint64_t start,
                           uint32_t boundary, int16_t* coef, uint32_t g0, uint32_t total_blocks, int* err) {
    BitReader br;
    br.init_at(stream, stream_bytes, state_p(start));
    int k = state_k(start), b = state_b(start);
    uint32_t nblk = 0, g = g0;
    int16_t* blk = WRITE ? block_of(coef, L, g) : nullptr;
    while (br.pos() < boundary && (!WRITE || g < total_blocks)) {
        br.refill();
        const int comp = b < L.nl ? 0 : b - L.nl + 1;
        if (k == 0) {
            int s = decode_symbol(br, ts.dc[ts.comp_dc[comp]]);
            if (s < 0 || s > 16) { if (WRITE) *err = 1; s = 0; }
            if (s) {
                const uint32_t v = br.peek(s);
                br.skip(s);
                if (WRITE) blk[0] = (int16_t)extend(v, s);
            }
            k = 1;
        } else {
            int sym = decode_symbol(br, ts.ac[ts.comp_ac[comp]]);
            if (sym < 0) { if (WRITE) *err = 1; sym = 0; }
            const int r = sym >> 4, s = sym & 15;
            if (s) {
                k += r;
                if (k > 63) { if (WRITE) *err = 1; k = 63; }
                const uint32_t v = br.peek(s);
                br.skip(s);
                if (WRITE) blk[nat[k]] = (int16_t)extend(v, s);
                ++k;
            } else if (r == 15) {
                k += 16;
                if (k > 64) { if (WRITE) *err = 1; k = 64; }
            } else {
                k = 64;
            }
        }
        if (k >= 64) {
            k = 0;
            b = b == L.nb - 1 ? 0 : b + 1;
            ++nblk;
            ++g;
            if (WRITE) blk = block_of(coef, L, g < total_blocks ? g : total_blocks - 1);
        }
    }
    return span_state(br.pos(), nblk, k, b);
}

// ---- progressive files (SOF2): the four MCU decoders of jdphuff.c ------------------------------------------------------
// A progressive file codes the same quantised coefficients as its baseline twin in several scans: DC scans (Ss = Se = 0,
// one or more components, interleaved in MCUs when more than one) and AC scans (one component, band Ss..Se); a first scan
// (Ah = 0) codes the coefficients shifted right by Al, a refinement scan (Ah = Al + 1) one more bit of each.  Once every
// coefficient has been refined down to Al = 0 (the parser reports every other file) the coefficients are the baseline
// twin's, and so are the pixels (no block smoothing: libjpeg-turbo only smooths while coefficient bits are unknown).
// The scans are decoded into the same per-component block rasters as a baseline scan; the IDCT and colour stages are shared.
struct ScanRec {
    uint32_t image;
    uint8_t ncomp;               // components in the scan: 1 (non-interleaved: the component's own block raster) .. 3
    uint8_t comp[3];             // their indices 0 .. 2, in frame order
    uint8_t Ss, Se, Ah, Al;
    uint32_t out_block;          // refinement scans: first block of their results in the refinement output (RefineOut)
    int32_t dc_tab[3];           // index into the batch's HuffTab array per scan component (DC first scans), else -1
    int32_t ac_tab;              // AC scans, else -1
};

// One restart interval of a progressive scan (a scan without restart markers: one).  Bytes as in SegRec; a UNIT is an MCU
// of an interleaved scan and a block of a non-interleaved one.  EOBRUN and the DC predictions start from 0 in every one.
struct ScanSeg {
    uint64_t stream_off;
    uint32_t scan;
    uint32_t byte0;
    uint32_t stream_bytes;
    uint32_t first_unit;
    uint32_t n_units;
    uint32_t pad;
};

// What a refinement scan found for one block, kept apart from the coefficients so that the serial Huffman pass only
// decodes and a parallel pass applies it (apply_refinement): bit k = zigzag position k.
struct RefineOut {
    uint64_t corr;               // correction bit 1 (DC refinement: bit 0)
    uint64_t newpos;             // a new coefficient of magnitude 1 << Al
    uint64_t newneg;             // ... and it is negative
};

RJ_HD int ctz64(uint64_t x) {
#if defined(__CUDA_ARCH__)
    return __ffsll((long long)x) - 1;
#else
    return __builtin_ctzll(x);
#endif
}
RJ_HD int popc64(uint64_t x) {
#if defined(__CUDA_ARCH__)
    return __popcll(x);
#else
    return __builtin_popcountll(x);
#endif
}
RJ_HD uint64_t bits_from(int k) { return k >= 64 ? 0ull : ~0ull << k; }     // positions >= k
RJ_HD uint64_t bits_below(int k) { return k >= 64 ? ~0ull : (1ull << k) - 1; }   // positions < k

// blocks across / down of component comp in a non-interleaved scan: ceil(component size / 8) (jdinput.c), not padded to MCUs
RJ_HD int comp_blocks_w(const ImageRec& im, int comp) { return comp == 0 ? (im.w + 7) / 8 : ((im.w + im.hs - 1) / im.hs + 7) / 8; }
RJ_HD int comp_blocks_h(const ImageRec& im, int comp) { return comp == 0 ? (im.h + 7) / 8 : ((im.h + im.vs - 1) / im.vs + 7) / 8; }
RJ_HD uint32_t scan_units(const ImageRec& im, const ScanRec& sc) {
    return sc.ncomp > 1 ? (uint32_t)layout_of(im).mcus : (uint32_t)comp_blocks_w(im, sc.comp[0]) * (uint32_t)comp_blocks_h(im, sc.comp[0]);
}
RJ_HD uint32_t scan_blocks_per_unit(const ImageRec& im, const ScanRec& sc) {
    if (sc.ncomp == 1) return 1;
    uint32_t n = 0;
    for (int ci = 0; ci < sc.ncomp; ++ci) n += sc.comp[ci] == 0 ? (uint32_t)im.hs * im.vs : 1u;
    return n;
}
// block (by, bx) of component comp in an image's coefficient area (the rasters of block_of: luma hs * mcu_w blocks wide,
// chroma mcu_w).  Blocks a non-interleaved scan does not reach (right of / below ceil(size / 8)) keep zeros; they only
// feed plane samples at x >= w / y >= h (luma) or >= the real chroma size, which the colour stage never reads.
RJ_HD int16_t* comp_block(int16_t* coef, const Layout& L, int comp, uint32_t by, uint32_t bx) {
    if (comp == 0) return coef + 64L * ((long)by * (L.hs * L.mcu_w) + bx);
    return coef + 64L * (L.nl * L.mcus + (long)(comp - 1) * L.mcus + (long)by * L.mcu_w + bx);
}
// block j of a scan in coding order (unit j / blocks per unit; in an MCU the components' blocks in scan order)
RJ_HD int16_t* scan_block(int16_t* coef, const ImageRec& im, const ScanRec& sc, uint32_t j) {
    const Layout L = layout_of(im);
    if (sc.ncomp == 1) {
        const uint32_t bw = (uint32_t)comp_blocks_w(im, sc.comp[0]), by = j / bw;
        return comp_block(coef, L, sc.comp[0], by, j - by * bw);
    }
    const uint32_t bpu = scan_blocks_per_unit(im, sc), u = j / bpu;
    uint32_t b = j - u * bpu;
    const uint32_t my = u / (uint32_t)L.mcu_w, mx = u - my * (uint32_t)L.mcu_w;
    for (int ci = 0; ci < sc.ncomp; ++ci) {
        const int comp = sc.comp[ci];
        const uint32_t n = comp == 0 ? (uint32_t)(L.hs * L.vs) : 1u;
        if (b < n) {
            const uint32_t v = b / (uint32_t)(comp == 0 ? L.hs : 1), h = b - v * (uint32_t)(comp == 0 ? L.hs : 1);
            return comp == 0 ? comp_block(coef, L, 0, L.vs * my + v, L.hs * mx + h) : comp_block(coef, L, comp, my, mx);
        }
        b -= n;
    }
    return nullptr;
}

// the nonzero coefficients of a block as a mask over zigzag positions (what an AC refinement scan needs of the history)
RJ_HD uint64_t zigzag_nz_mask(const int16_t* blk, const uint8_t* nat) {
    uint64_t nat_mask = 0;
    for (int q = 0; q < 8; ++q) {   // eight 16-byte loads on the device (blocks are 128-byte aligned)
#if defined(__CUDA_ARCH__)
        const uint4 x = reinterpret_cast<const uint4*>(blk)[q];
        const uint32_t w[4] = {x.x, x.y, x.z, x.w};
#else
        uint32_t w[4];
        for (int j = 0; j < 4; ++j) w[j] = (uint16_t)blk[8 * q + 2 * j] | ((uint32_t)(uint16_t)blk[8 * q + 2 * j + 1] << 16);
#endif
        for (int j = 0; j < 4; ++j) {
            if (w[j] & 0xFFFFu) nat_mask |= 1ull << (8 * q + 2 * j);
            if (w[j] >> 16) nat_mask |= 1ull << (8 * q + 2 * j + 1);
        }
    }
    uint64_t m = 0;
    for (int k = 0; k < 64; ++k) m |= ((nat_mask >> nat[k]) & 1ull) << k;
    return m;
}

// jdphuff.c decode_mcu_AC_refine's correction bits: one per position of `positions` (ascending); returns the positions
// whose bit is 1
RJ_HD uint64_t read_corrections(BitReader& br, uint64_t positions) {
    uint64_t out = 0;
    while (positions) {
        br.refill();
        const int c = popc64(positions) < 32 ? popc64(positions) : 32;
        const uint32_t bits = br.peek(c);
        br.skip(c);
        for (int i = c - 1; i >= 0; --i) {
            const int pos = ctz64(positions);
            positions &= positions - 1;
            out |= (uint64_t)((bits >> i) & 1u) << pos;
        }
    }
    return out;
}

// One block of a progressive scan (jdphuff.c decode_mcu_DC_first / _AC_first / _DC_refine / _AC_refine); ci: the block's
// index in the scan's component list, *last_dc: that component's DC prediction.  First scans write the coefficients;
// refinement scans write *out (nz: the block's nonzero coefficients before the scan, zigzag_nz_mask).  Returns false on
// a corrupt stream.
RJ_HD bool decode_prog_block(BitReader& br, const ScanRec& sc, const HuffTab* tabs, const uint8_t* nat, int ci, int* last_dc,
                             uint32_t* eobrun, int16_t* blk, uint64_t nz, RefineOut* out) {
    const int Ss = sc.Ss, Se = sc.Se, Al = sc.Al;
    if (Ss == 0) {
        br.refill();
        if (sc.Ah == 0) {   // DC first: difference to the component's prediction, stored shifted left by Al
            const int s = decode_symbol(br, tabs[sc.dc_tab[ci]]);
            if (s < 0 || s > 16) return false;
            int diff = 0;
            if (s) {
                br.refill();
                diff = extend(br.peek(s), s);
                br.skip(s);
            }
            *last_dc += diff;
            blk[0] = (int16_t)(int)((uint32_t)*last_dc << Al);
        } else {            // DC refinement: one bit
            out->corr = br.peek(1);
            br.skip(1);
        }
        return true;
    }
    const HuffTab& ac = tabs[sc.ac_tab];
    if (sc.Ah == 0) {       // AC first: run-length / size symbols with end-of-band runs across blocks
        if (*eobrun > 0) { --*eobrun; return true; }
        for (int k = Ss; k <= Se; ++k) {
            br.refill();
            const int sym = decode_symbol(br, ac);
            if (sym < 0) return false;
            const int r = sym >> 4, s = sym & 15;
            if (s) {
                k += r;
                if (k > Se) return false;
                const int v = extend(br.peek(s), s);
                br.skip(s);
                blk[nat[k]] = (int16_t)(int)((uint32_t)v << Al);
            } else if (r == 15) {
                k += 15;
            } else {
                *eobrun = 1u << r;
                if (r) { *eobrun += br.peek(r); br.skip(r); }
                --*eobrun;
                break;
            }
        }
        return true;
    }
    // AC refinement on masks: a symbol's run of r zeros ends at the (r + 1)-th position of the band that is zero in the
    // history; every nonzero position passed on the way takes one correction bit (libjpeg walks them one at a time)
    const uint64_t band = bits_from(Ss) & bits_below(Se + 1);
    uint64_t corr = 0, newpos = 0, newneg = 0;
    int k = Ss;
    if (*eobrun == 0) {
        while (k <= Se) {
            br.refill();
            const int sym = decode_symbol(br, ac);
            if (sym < 0) return false;
            const int r = sym >> 4, s = sym & 15;
            bool neg = false;
            if (s) {
                if (s != 1) return false;
                neg = br.peek(1) == 0;
                br.skip(1);
            } else if (r != 15) {
                *eobrun = 1u << r;
                if (r) { br.refill(); *eobrun += br.peek(r); br.skip(r); }
                break;
            }
            uint64_t zeros = ~nz & band & bits_from(k);
            for (int i = 0; i < r && zeros; ++i) zeros &= zeros - 1;
            const int t = zeros ? ctz64(zeros) : Se + 1;   // the new coefficient's position (ZRL: the 16th zero)
            corr |= read_corrections(br, nz & band & bits_from(k) & bits_below(t));
            if (s) {
                if (t > Se) return false;
                newpos |= 1ull << t;
                if (neg) newneg |= 1ull << t;
            }
            k = t + 1;
        }
    }
    if (*eobrun > 0) {      // inside an end-of-band run: only the correction bits of the remaining nonzero coefficients
        corr |= read_corrections(br, nz & band & bits_from(k));
        --*eobrun;
    }
    out->corr = corr;
    out->newpos = newpos;
    out->newneg = newneg;
    return true;
}

// What decode_prog_block found for block blk of refinement scan sc, applied (the parallel pass after a level).
RJ_HD void apply_refinement(int16_t* blk, const ScanRec& sc, const RefineOut& o, const uint8_t* nat) {
    const int p1 = 1 << sc.Al, m1 = (int)(~0u << sc.Al);
    if (sc.Ss == 0) {
        if (o.corr) blk[0] = (int16_t)(blk[0] | p1);
        return;
    }
    for (uint64_t c = o.corr; c; c &= c - 1) {
        const int z = nat[ctz64(c)], v = blk[z];
        if ((v & p1) == 0) blk[z] = (int16_t)(v + (v >= 0 ? p1 : m1));
    }
    for (uint64_t n = o.newpos; n; n &= n - 1) {
        const int k = ctz64(n);
        blk[nat[k]] = (int16_t)(((o.newneg >> k) & 1u) ? m1 : p1);
    }
}

// One restart interval of a progressive scan, sequentially.  coef: the image's coefficient area; refinement scans read
// nz (the image's blocks' zigzag_nz_mask, same block order as coef) and write out (the scan's RefineOut, in coding
// order).  Returns 0, or 1 (corrupt code), 2 (ran past the end of the segment).
RJ_HD int decode_prog_segment(const ImageRec& im, const ScanRec& sc, const ScanSeg& sg, const HuffTab* tabs, const uint8_t* nat,
                              const uint8_t* streams, int16_t* coef, const uint64_t* nz, RefineOut* out) {
    const Layout L = layout_of(im);
    BitReader br;
    br.init_at(streams + sg.stream_off, sg.stream_bytes, 8u * sg.byte0);
    int dc0 = 0, dc1 = 0, dc2 = 0;   // the DC predictions of the scan's components (scalars: no local-memory array)
    uint32_t eobrun = 0;
    const bool ac_refine = sc.Ah != 0 && sc.Ss != 0;
    uint32_t j = sg.first_unit * scan_blocks_per_unit(im, sc);   // block index in coding order
    if (sc.ncomp == 1) {
        const int comp = sc.comp[0];
        const uint32_t bw = (uint32_t)comp_blocks_w(im, comp);
        for (uint32_t u = sg.first_unit; u < sg.first_unit + sg.n_units; ++u, ++j) {
            const uint32_t by = u / bw;
            int16_t* blk = comp_block(coef, L, comp, by, u - by * bw);
            if (!decode_prog_block(br, sc, tabs, nat, 0, &dc0, &eobrun, blk, ac_refine ? nz[(blk - coef) >> 6] : 0ull,
                                   out ? out + j : nullptr))
                return 1;
        }
    } else {   // interleaved: DC scans only (the parser checks), no history needed
        for (uint32_t u = sg.first_unit; u < sg.first_unit + sg.n_units; ++u) {
            const uint32_t my = u / (uint32_t)L.mcu_w, mx = u - my * (uint32_t)L.mcu_w;
            for (int ci = 0; ci < sc.ncomp; ++ci) {
                const int comp = sc.comp[ci];
                const int bh = comp == 0 ? L.vs : 1, bwid = comp == 0 ? L.hs : 1;
                int pred = ci == 0 ? dc0 : (ci == 1 ? dc1 : dc2);
                for (int v = 0; v < bh; ++v)
                    for (int h = 0; h < bwid; ++h, ++j)
                        if (!decode_prog_block(br, sc, tabs, nat, ci, &pred, &eobrun,
                                               comp_block(coef, L, comp, bh * my + v, bwid * mx + h), 0ull,
                                               out ? out + j : nullptr)) return 1;
                if (ci == 0) dc0 = pred; else if (ci == 1) dc1 = pred; else dc2 = pred;
            }
        }
    }
    return br.bits_used() > 8ull * sg.stream_bytes ? 2 : 0;
}

// jidctint.c jpeg_idct_islow: 64 quantised coefficients (natural order) x quantisation table -> 64 samples 0..255.
RJ_HD int idct_descale(int x, int n) { return (x + (1 << (n - 1))) >> n; }
RJ_HD uint8_t idct_limit(int v) {   // range_limit[(v) & RANGE_MASK] for in-range data: clamp(v + 128, 0, 255)
    v += 128;
    return (uint8_t)(v < 0 ? 0 : (v > 255 ? 255 : v));
}
RJ_HD void idct_1d(int d0, int d1, int d2, int d3, int d4, int d5, int d6, int d7, int even_shift, int* o) {
    // even part (d0, d4 enter shifted by CONST_BITS = 13)
    int z1 = (d2 + d6) * 4433;
    const int tmp2 = z1 + d6 * (-15137), tmp3 = z1 + d2 * 6270;
    const int tmp0 = (d0 + d4) * 8192, tmp1 = (d0 - d4) * 8192;
    const int tmp10 = tmp0 + tmp3, tmp13 = tmp0 - tmp3, tmp11 = tmp1 + tmp2, tmp12 = tmp1 - tmp2;
    // odd part
    int t0 = d7, t1 = d5, t2 = d3, t3 = d1;
    z1 = t0 + t3;
    int z2 = t1 + t2, z3 = t0 + t2, z4 = t1 + t3;
    const int z5 = (z3 + z4) * 9633;
    t0 *= 2446; t1 *= 16819; t2 *= 25172; t3 *= 12299;
    z1 *= -7373; z2 *= -20995; z3 *= -16069; z4 *= -3196;
    z3 += z5; z4 += z5;
    t0 += z1 + z3; t1 += z2 + z4; t2 += z2 + z3; t3 += z1 + z4;
    o[0] = idct_descale(tmp10 + t3, even_shift); o[7] = idct_descale(tmp10 - t3, even_shift);
    o[1] = idct_descale(tmp11 + t2, even_shift); o[6] = idct_descale(tmp11 - t2, even_shift);
    o[2] = idct_descale(tmp12 + t1, even_shift); o[5] = idct_descale(tmp12 - t1, even_shift);
    o[3] = idct_descale(tmp13 + t0, even_shift); o[4] = idct_descale(tmp13 - t0, even_shift);
}
RJ_HD void idct_islow(const int16_t* coef, const uint16_t* quant, uint8_t* out, long out_pitch) {
    int ws[64];
#if defined(__CUDA_ARCH__)
#pragma unroll
#endif
    for (int c = 0; c < 8; ++c) {   // pass 1: columns; results scaled up by 2^PASS1_BITS
        int d[8], o[8];
#if defined(__CUDA_ARCH__)
#pragma unroll
#endif
        for (int r = 0; r < 8; ++r) d[r] = (int)coef[8 * r + c] * (int)quant[8 * r + c];
        idct_1d(d[0], d[1], d[2], d[3], d[4], d[5], d[6], d[7], 13 - 2, o);
#if defined(__CUDA_ARCH__)
#pragma unroll
#endif
        for (int r = 0; r < 8; ++r) ws[8 * r + c] = o[r];
    }
#if defined(__CUDA_ARCH__)
#pragma unroll
#endif
    for (int r = 0; r < 8; ++r) {   // pass 2: rows; descale by 2^(CONST_BITS + PASS1_BITS + 3)
        int o[8];
        idct_1d(ws[8 * r], ws[8 * r + 1], ws[8 * r + 2], ws[8 * r + 3], ws[8 * r + 4], ws[8 * r + 5], ws[8 * r + 6],
                ws[8 * r + 7], 13 + 2 + 3, o);
        uint8_t* p = out + r * out_pitch;
#if defined(__CUDA_ARCH__)
#pragma unroll
#endif
        for (int c = 0; c < 8; ++c) p[c] = idct_limit(o[c]);
    }
}

// jdsample.c h2v2_fancy_upsample + jdmainct.c: the chroma sample of output pixel (x, y).  plane: the decoded half-resolution
// plane (pitch bytes per row); cw x ch = its REAL size, ceil(w / 2) x ceil(h / 2).  cw >= 3 (the parser rejects w < 5).
RJ_HD int upsample_h2v2(const uint8_t* plane, long pitch, int cw, int ch, int x, int y) {
    const int cy = y >> 1, cx = x >> 1;
    int ny = (y & 1) ? cy + 1 : cy - 1;          // the further row: below for odd output rows, above for even ones
    ny = ny < 0 ? 0 : (ny > ch - 1 ? ch - 1 : ny);
    const uint8_t* r0 = plane + (long)cy * pitch;
    const uint8_t* r1 = plane + (long)ny * pitch;
    const int cur = 3 * r0[cx] + r1[cx];
    if (x & 1) {
        if (cx == cw - 1) return (4 * cur + 7) >> 4;
        return (3 * cur + 3 * r0[cx + 1] + r1[cx + 1] + 7) >> 4;
    }
    if (cx == 0) return (4 * cur + 8) >> 4;
    return (3 * cur + 3 * r0[cx - 1] + r1[cx - 1] + 8) >> 4;
}

// jdsample.c h2v1_fancy_upsample (4:2:2): the filter along the row only.  cw >= 3.
RJ_HD int upsample_h2v1(const uint8_t* plane, long pitch, int cw, int x, int y) {
    const uint8_t* r0 = plane + (long)y * pitch;
    const int cx = x >> 1, cur = r0[cx];
    if (x & 1) return cx == cw - 1 ? cur : (3 * cur + r0[cx + 1] + 2) >> 2;
    return cx == 0 ? cur : (3 * cur + r0[cx - 1] + 1) >> 2;
}
// the chroma sample of output pixel (x, y) for luma sampling hs x vs
RJ_HD int chroma_at(const uint8_t* plane, long pitch, int hs, int vs, int cw, int ch, int x, int y) {
    if (hs == 2) return vs == 2 ? upsample_h2v2(plane, pitch, cw, ch, x, y) : upsample_h2v1(plane, pitch, cw, x, y);
    return plane[(long)y * pitch + x];
}

// The chroma samples of the four output pixels x0 .. x0 + 3 (x0 a multiple of 4) of row y in one go: the same values as four
// chroma_at calls, with the two or three plane columns they share read once.  Pixels at or beyond the image width get
// unspecified values.
RJ_HD void chroma_quad(const uint8_t* plane, long pitch, int hs, int vs, int cw, int ch, int x0, int y, int* o) {
    if (hs == 1) {
        const uint8_t* r = plane + (long)y * pitch + x0;   // (planes are padded to whole blocks: reading 4 bytes is safe)
        o[0] = r[0]; o[1] = r[1]; o[2] = r[2]; o[3] = r[3];
        return;
    }
    const int c0 = x0 >> 1;
    const int cl = c0 > 0 ? c0 - 1 : 0, c1 = c0 + 1 < cw ? c0 + 1 : cw - 1, c2 = c0 + 2 < cw ? c0 + 2 : cw - 1;
    if (vs == 2) {
        const int cy = y >> 1;
        int ny = (y & 1) ? cy + 1 : cy - 1;
        ny = ny < 0 ? 0 : (ny > ch - 1 ? ch - 1 : ny);
        const uint8_t* r0 = plane + (long)cy * pitch;
        const uint8_t* r1 = plane + (long)ny * pitch;
        const int sl = 3 * r0[cl] + r1[cl], s0 = 3 * r0[c0] + r1[c0], s1 = 3 * r0[c1] + r1[c1], s2 = 3 * r0[c2] + r1[c2];
        o[0] = c0 == 0 ? (4 * s0 + 8) >> 4 : (3 * s0 + sl + 8) >> 4;
        o[1] = c0 == cw - 1 ? (4 * s0 + 7) >> 4 : (3 * s0 + s1 + 7) >> 4;
        o[2] = (3 * s1 + s0 + 8) >> 4;
        o[3] = c0 + 1 >= cw - 1 ? (4 * s1 + 7) >> 4 : (3 * s1 + s2 + 7) >> 4;
        return;
    }
    const uint8_t* r0 = plane + (long)y * pitch;
    const int vl = r0[cl], v0 = r0[c0], v1 = r0[c1], v2 = r0[c2];
    o[0] = c0 == 0 ? v0 : (3 * v0 + vl + 1) >> 2;
    o[1] = c0 == cw - 1 ? v0 : (3 * v0 + v1 + 2) >> 2;
    o[2] = (3 * v1 + v0 + 1) >> 2;
    o[3] = c0 + 1 >= cw - 1 ? v1 : (3 * v1 + v2 + 2) >> 2;
}

// jdcolor.c ycc_rgb_convert (SCALEBITS 16), written as B, G, R
RJ_HD void ycc_to_bgr(int y, int cb, int cr, uint8_t* bgr) {
    cb -= 128; cr -= 128;
    const int r = y + ((91881 * cr + 32768) >> 16);
    const int g = y + ((-22554 * cb + 32768 - 46802 * cr) >> 16);
    const int b = y + ((116130 * cb + 32768) >> 16);
    bgr[0] = (uint8_t)(b < 0 ? 0 : (b > 255 ? 255 : b));
    bgr[1] = (uint8_t)(g < 0 ? 0 : (g > 255 ? 255 : g));
    bgr[2] = (uint8_t)(r < 0 ? 0 : (r > 255 ? 255 : r));
}

}  // namespace jpegdec
}  // namespace rod
