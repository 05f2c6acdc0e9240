// jpegdec_progressive_replay.cpp -- TEST INFRASTRUCTURE, built with g++ by tests/test_jpegdec_progressive.py; never linked
// into the product.
//
// replay_decode: the device decoder of csrc/jpegdec.cu replayed sequentially on the CPU from the same headers -- the parser
// (baseline and progressive files), the scan levels, the four progressive MCU decoders (one restart interval at a time, a
// level's segments in reverse order: they must not depend on each other), then the baseline IDCT and colour functions.
//
// replay_write: a small progressive entropy WRITER (libjpeg's jcphuff.c restated) that re-encodes the coefficients of a
// baseline file under a given scan script, so the decoder can be checked on scripts OpenCV and PIL never write.  It uses
// two "universal" Huffman tables (every symbol a scan can need, all codes of one length), in ascending or descending
// symbol order by scan, so that a decoder that kept a table of an earlier scan decodes garbage.
#include <string.h>

#include <vector>

#include "../../robust-object-detection_b200/csrc/rod_jpegdec_host.h"

using namespace rod::jpegdec;

namespace {

uint8_t g_nat[64];
void init_nat() {
    for (int z = 0; z < 64; ++z) g_nat[z] = (uint8_t)rod::jpeg::natural_order(z);
}

ImageRec image_of(const FileInfo& info) {
    ImageRec im;
    memset(&im, 0, sizeof(im));
    im.h = info.height; im.w = info.width;
    im.hs = (uint8_t)info.hs; im.vs = (uint8_t)info.vs; im.ncomp = (uint8_t)info.ncomp;
    return im;
}

// coefficients of a file (quantised, natural order, the device's block rasters); 0 or a device status (1, 2, 1x)
int decode_coefficients(const uint8_t* file, long n, int formats, FileInfo* info, TableSet* ts, std::vector<int16_t>* coef) {
    std::vector<uint8_t> stream((size_t)n + 64, 0);
    const ParseStatus st = parse_file(file, (size_t)n, info, ts, formats, stream.data());
    if (st != PARSE_OK) return 10 + (int)st;
    const ImageRec im = image_of(*info);
    const Layout L = layout_of(im);
    coef->assign((size_t)L.mcus * L.nb * 64, 0);
    if (!info->progressive) {
        std::vector<uint32_t> rst;
        const size_t sb = unstuff_scan(file, (size_t)n, info->scan_begin, stream.data(), &rst);
        if (sb == (size_t)-1) return 13;
        std::vector<SegRec> segs;
        if (!make_segments(im, 0, info->restart_interval, 0, sb, rst, &segs)) return 13;
        return decode_scan(im, segs.data(), (int)segs.size(), *ts, g_nat, stream.data(), coef->data());
    }
    std::vector<ScanRec> recs;
    std::vector<ScanSeg> segs;
    uint32_t out_blocks = 0;
    for (size_t s = 0; s < info->scans.size(); ++s) {
        ScanRec r = info->scans[s].rec;
        for (int j = 0; j < 3; ++j) r.dc_tab[j] = info->scans[s].dc_slot[j];
        r.ac_tab = info->scans[s].ac_slot;
        if (r.Ah != 0) {
            r.out_block = out_blocks;
            out_blocks += scan_units(im, r) * scan_blocks_per_unit(im, r);
        }
        recs.push_back(r);
        if (!make_scan_segments(im, info->scans[s], (uint32_t)s, 0, &segs)) return 13;
    }
    std::vector<int> level;
    const int n_levels = scan_levels(info->scans, &level);
    std::vector<RefineOut> out(out_blocks + 1);
    std::vector<uint64_t> nz(coef->size() / 64);
    int rc = 0;
    for (int lv = 0; lv < n_levels; ++lv) {   // the device's passes: history masks, Huffman decoding, refinements applied
        for (size_t b = 0; b < nz.size(); ++b) nz[b] = zigzag_nz_mask(coef->data() + 64 * b, g_nat);
        for (size_t q = segs.size(); q-- > 0;) {
            const ScanRec& sc = recs[segs[q].scan];
            if (level[segs[q].scan] != lv) continue;
            const int r = decode_prog_segment(im, sc, segs[q], info->huff.data(), g_nat, stream.data(), coef->data(), nz.data(),
                                              sc.Ah != 0 ? out.data() + sc.out_block : nullptr);
            if (r > rc) rc = r;
        }
        if (rc) return rc;
        for (size_t s = 0; s < recs.size(); ++s) {
            const ScanRec& sc = recs[s];
            if (level[s] != lv || sc.Ah == 0) continue;
            const uint32_t n = scan_units(im, sc) * scan_blocks_per_unit(im, sc);
            for (uint32_t j = 0; j < n; ++j) apply_refinement(scan_block(coef->data(), im, sc, j), sc, out[sc.out_block + j], g_nat);
        }
    }
    return rc;
}

}  // namespace

// Returns 0 and fills out (HWC BGR, pitch 3 * w) and hw[3] = (h, w, progressive); else the status the device decoder
// reports for the file (1 / 2 corrupt / truncated entropy data, 11 / 12 / 13 the host verdicts), or 20: out too small.
// poison: fill every coefficient block that no scan reaches (right of / below the image's blocks) with large values first
// -- the pixels must not change.
extern "C" int replay_decode(const uint8_t* file, long n, uint8_t* out, long out_cap, int* hw, int poison) {
    init_nat();
    FileInfo info;
    TableSet ts;
    std::vector<int16_t> coef;
    const int rc = decode_coefficients(file, n, kBaseline | kProgressive, &info, &ts, &coef);
    if (rc) return rc;
    const ImageRec im = image_of(info);
    const Layout L = layout_of(im);
    hw[0] = im.h; hw[1] = im.w; hw[2] = info.progressive ? 1 : 0;
    if ((long)im.h * im.w * 3 > out_cap) return 20;
    if (poison) {
        for (int c = 0; c < im.ncomp; ++c) {
            const int bw = comp_blocks_w(im, c), bh = comp_blocks_h(im, c);
            const int rw = c == 0 ? L.hs * L.mcu_w : L.mcu_w, rh = c == 0 ? L.vs * L.mcu_h : L.mcu_h;
            for (int by = 0; by < rh; ++by)
                for (int bx = 0; bx < rw; ++bx)
                    if (by >= bh || bx >= bw) {
                        int16_t* b = comp_block(coef.data(), L, c, (uint32_t)by, (uint32_t)bx);
                        for (int k = 0; k < 64; ++k) b[k] = (int16_t)((k * 37 + by * 11 + bx * 5) % 61 - 30);
                        b[0] = 90;
                    }
        }
    }
    const long ypitch = 8L * L.hs * L.mcu_w, cpitch = 8L * L.mcu_w;
    std::vector<uint8_t> yp((size_t)ypitch * 8 * L.vs * L.mcu_h), cbp((size_t)cpitch * 8 * L.mcu_h, 128), crp((size_t)cpitch * 8 * L.mcu_h, 128);
    for (int by = 0; by < L.vs * L.mcu_h; ++by)
        for (int bx = 0; bx < L.hs * L.mcu_w; ++bx)
            idct_islow(comp_block(coef.data(), L, 0, by, bx), ts.quant[0], yp.data() + 8L * by * ypitch + 8 * bx, ypitch);
    if (im.ncomp == 3)
        for (int by = 0; by < L.mcu_h; ++by)
            for (int bx = 0; bx < L.mcu_w; ++bx) {
                idct_islow(comp_block(coef.data(), L, 1, by, bx), ts.quant[1], cbp.data() + 8L * by * cpitch + 8 * bx, cpitch);
                idct_islow(comp_block(coef.data(), L, 2, by, bx), ts.quant[2], crp.data() + 8L * by * cpitch + 8 * bx, cpitch);
            }
    const int cw = (im.w + L.hs - 1) / L.hs, ch = (im.h + L.vs - 1) / L.vs;
    for (int y = 0; y < im.h; ++y)
        for (int x0 = 0; x0 < im.w; x0 += 4) {   // four pixels at a time, like a thread of jpegdec_color_kernel
            int cb[4] = {128, 128, 128, 128}, cr[4] = {128, 128, 128, 128};
            if (im.ncomp == 3) {
                chroma_quad(cbp.data(), cpitch, L.hs, L.vs, cw, ch, x0, y, cb);
                chroma_quad(crp.data(), cpitch, L.hs, L.vs, cw, ch, x0, y, cr);
            }
            for (int i = 0; i < 4 && x0 + i < im.w; ++i) {
                uint8_t* o = out + ((size_t)y * im.w + x0 + i) * 3;
                const int yy = yp[(size_t)y * ypitch + x0 + i];
                if (im.ncomp == 1) { o[0] = o[1] = o[2] = (uint8_t)yy; continue; }
                ycc_to_bgr(yy, cb[i], cr[i], o);
            }
        }
    return 0;
}

// ---- the writer ------------------------------------------------------------------------------------------------------
namespace {

struct Writer {
    std::vector<uint8_t>* out;
    uint32_t acc = 0;
    int n = 0;
    void bits(uint32_t v, int k) {   // MSB first, 0xFF stuffed
        for (int i = k - 1; i >= 0; --i) {
            acc = (acc << 1) | ((v >> i) & 1u);
            if (++n == 8) {
                out->push_back((uint8_t)acc);
                if ((uint8_t)acc == 0xFF) out->push_back(0);
                acc = 0; n = 0;
            }
        }
    }
    void flush() { while (n) bits(1, 1); }   // pad with ones
};

// universal tables: DC symbols 0..11 with 4-bit codes; AC: every (run, size <= 10) pair, EOBn (n <= 14) and ZRL, 8-bit codes
std::vector<uint8_t> dc_symbols(bool desc) {
    std::vector<uint8_t> v;
    for (int s = 0; s < 12; ++s) v.push_back((uint8_t)s);
    if (desc) std::vector<uint8_t>(v.rbegin(), v.rend()).swap(v);
    return v;
}
std::vector<uint8_t> ac_symbols(bool desc) {
    std::vector<uint8_t> v;
    for (int r = 0; r < 16; ++r) {
        if (r < 15) v.push_back((uint8_t)(r << 4));
        else v.push_back(0xF0);
        for (int s = 1; s <= 10; ++s) v.push_back((uint8_t)((r << 4) | s));
    }
    if (desc) std::vector<uint8_t>(v.rbegin(), v.rend()).swap(v);
    return v;
}

struct Enc {
    Writer w;
    int code_len;
    int code_of[256];
    void set(const std::vector<uint8_t>& syms, int len) {
        code_len = len;
        for (int i = 0; i < 256; ++i) code_of[i] = -1;
        for (size_t i = 0; i < syms.size(); ++i) code_of[syms[i]] = (int)i;   // canonical: one length, codes in table order
    }
    void sym(int s) { w.bits((uint32_t)code_of[s], code_len); }
};

int bitlen(int v) { int n = 0; while (v) { ++n; v >>= 1; } return n; }

void put_dht(std::vector<uint8_t>* f, int tc, int th, const std::vector<uint8_t>& syms, int len) {
    const size_t L = 2 + 17 + syms.size();
    f->insert(f->end(), {0xFF, 0xC4, (uint8_t)(L >> 8), (uint8_t)L, (uint8_t)((tc << 4) | th)});
    for (int l = 1; l <= 16; ++l) f->push_back(l == len ? (uint8_t)syms.size() : 0);
    f->insert(f->end(), syms.begin(), syms.end());
}

struct ScanState {   // jcphuff.c: EOBRUN and the correction bits buffered with it (BE)
    uint32_t eobrun = 0;
    std::vector<uint8_t> be;
};

void emit_eobrun(Enc& e, ScanState& s) {
    if (s.eobrun > 0) {
        const int nbits = bitlen((int)s.eobrun) - 1;
        e.sym(nbits << 4);
        if (nbits) e.w.bits(s.eobrun & ((1u << nbits) - 1), nbits);
        s.eobrun = 0;
        for (uint8_t b : s.be) e.w.bits(b, 1);
        s.be.clear();
    }
}

void encode_block(Enc& e, ScanState& s, const ScanRec& sc, const int16_t* blk, int ci, int* last_dc) {
    const int Ss = sc.Ss, Se = sc.Se, Al = sc.Al;
    if (Ss == 0) {
        if (sc.Ah == 0) {   // encode_mcu_DC_first
            const int t = blk[0] >> Al;
            int diff = t - last_dc[ci], d2 = diff;
            last_dc[ci] = t;
            if (diff < 0) { diff = -diff; --d2; }
            const int nb = bitlen(diff);
            e.sym(nb);
            if (nb) e.w.bits((uint32_t)d2 & ((1u << nb) - 1), nb);
        } else {            // encode_mcu_DC_refine
            e.w.bits((uint32_t)(blk[0] >> Al) & 1u, 1);
        }
        return;
    }
    if (sc.Ah == 0) {       // encode_mcu_AC_first
        int r = 0;
        for (int k = Ss; k <= Se; ++k) {
            int t = blk[g_nat[k]], t2;
            if (t == 0) { ++r; continue; }
            if (t < 0) { t = -t; t >>= Al; t2 = ~t; } else { t >>= Al; t2 = t; }
            if (t == 0) { ++r; continue; }
            emit_eobrun(e, s);
            while (r > 15) { e.sym(0xF0); r -= 16; }
            const int nb = bitlen(t);
            e.sym((r << 4) + nb);
            e.w.bits((uint32_t)t2 & ((1u << nb) - 1), nb);
            r = 0;
        }
        if (r > 0) {
            ++s.eobrun;
            if (s.eobrun == 0x7FFF) emit_eobrun(e, s);
        }
        return;
    }
    // encode_mcu_AC_refine
    int absv[64], eob = 0;
    for (int k = Ss; k <= Se; ++k) {
        int t = blk[g_nat[k]];
        if (t < 0) t = -t;
        absv[k] = t >> Al;
        if (absv[k] == 1) eob = k;
    }
    int r = 0;
    std::vector<uint8_t> br;
    for (int k = Ss; k <= Se; ++k) {
        const int t = absv[k];
        if (t == 0) { ++r; continue; }
        while (r > 15 && k <= eob) {
            emit_eobrun(e, s);
            e.sym(0xF0);
            r -= 16;
            for (uint8_t b : br) e.w.bits(b, 1);
            br.clear();
        }
        if (t > 1) { br.push_back((uint8_t)(t & 1)); continue; }
        emit_eobrun(e, s);
        e.sym((r << 4) + 1);
        e.w.bits(blk[g_nat[k]] < 0 ? 0u : 1u, 1);
        for (uint8_t b : br) e.w.bits(b, 1);
        br.clear();
        r = 0;
    }
    if (r > 0 || !br.empty()) {
        ++s.eobrun;
        s.be.insert(s.be.end(), br.begin(), br.end());
        if (s.eobrun == 0x7FFF || s.be.size() > 1000 - 64 + 1) emit_eobrun(e, s);
    }
}

}  // namespace

// script: n_scans records of 10 ints (ncomp, comp0, comp1, comp2, Ss, Se, Ah, Al, table slot 0..3, restart interval).
// Writes a progressive file with the coefficients of the baseline file into out; returns its length, or -1 (the input is
// not a baseline file this decoder takes), -2 (out too small).
extern "C" long replay_write(const uint8_t* file, long n, const int* script, int n_scans, uint8_t* out, long out_cap) {
    init_nat();
    FileInfo info;
    TableSet ts;
    std::vector<int16_t> coef;
    if (decode_coefficients(file, n, kBaseline, &info, &ts, &coef) != 0) return -1;
    const ImageRec im = image_of(info);
    const Layout L = layout_of(im);
    std::vector<uint8_t> f = {0xFF, 0xD8};
    // the baseline file's DQT and SOF segments (SOF0 -> SOF2); its DHT / DRI are replaced per scan
    for (size_t i = 2; i < info.scan_begin;) {
        const int m = file[i + 1];
        const size_t len = ((size_t)file[i + 2] << 8) | file[i + 3];
        if (m == 0xDB || m == 0xC0) {
            const size_t at = f.size();
            f.insert(f.end(), file + i, file + i + 2 + len);
            if (m == 0xC0) f[at + 1] = 0xC2;
        }
        i += 2 + len;
    }
    int cur_ri = 0;
    for (int q = 0; q < n_scans; ++q) {
        const int* d = script + 10 * q;
        ScanRec sc;
        memset(&sc, 0, sizeof(sc));
        sc.ncomp = (uint8_t)d[0];
        for (int j = 0; j < sc.ncomp; ++j) sc.comp[j] = (uint8_t)d[1 + j];
        sc.Ss = (uint8_t)d[4]; sc.Se = (uint8_t)d[5]; sc.Ah = (uint8_t)d[6]; sc.Al = (uint8_t)d[7];
        const int slot = d[8], ri = d[9];
        const bool desc = q & 1;
        Enc e;
        std::vector<uint8_t> data;
        e.w.out = &data;
        if (sc.Ss == 0 && sc.Ah == 0) { put_dht(&f, 0, slot, dc_symbols(desc), 4); e.set(dc_symbols(desc), 4); }
        if (sc.Ss > 0) { put_dht(&f, 1, slot, ac_symbols(desc), 8); e.set(ac_symbols(desc), 8); }
        if (ri != cur_ri) {
            f.insert(f.end(), {0xFF, 0xDD, 0, 4, (uint8_t)(ri >> 8), (uint8_t)ri});
            cur_ri = ri;
        }
        const size_t sl = 6 + 2 * (size_t)sc.ncomp;
        f.insert(f.end(), {0xFF, 0xDA, (uint8_t)(sl >> 8), (uint8_t)sl, sc.ncomp});
        for (int j = 0; j < sc.ncomp; ++j) {
            f.push_back((uint8_t)(info.ncomp == 3 ? sc.comp[j] + 1 : 1));   // the baseline file's component ids
            f.push_back((uint8_t)((slot << 4) | slot));
        }
        f.insert(f.end(), {sc.Ss, sc.Se, (uint8_t)((sc.Ah << 4) | sc.Al)});
        // the blocks in the decoder's order, restart markers every ri units
        ScanState st;
        int last_dc[3] = {0, 0, 0};
        const uint32_t units = scan_units(im, sc);
        int rst_no = 0;
        for (uint32_t u = 0; u < units; ++u) {
            if (ri > 0 && u > 0 && u % (uint32_t)ri == 0) {
                emit_eobrun(e, st);
                e.w.flush();
                data.push_back(0xFF);
                data.push_back((uint8_t)(0xD0 + (rst_no++ & 7)));
                last_dc[0] = last_dc[1] = last_dc[2] = 0;
            }
            if (sc.ncomp == 1) {
                const uint32_t bw = (uint32_t)comp_blocks_w(im, sc.comp[0]), by = u / bw;
                encode_block(e, st, sc, comp_block(coef.data(), L, sc.comp[0], by, u - by * bw), 0, last_dc);
            } else {
                const uint32_t my = u / (uint32_t)L.mcu_w, mx = u - my * (uint32_t)L.mcu_w;
                for (int ci = 0; ci < sc.ncomp; ++ci) {
                    const int c = sc.comp[ci], bh = c == 0 ? L.vs : 1, bwid = c == 0 ? L.hs : 1;
                    for (int v = 0; v < bh; ++v)
                        for (int h = 0; h < bwid; ++h)
                            encode_block(e, st, sc, comp_block(coef.data(), L, c, bh * my + v, bwid * mx + h), ci, last_dc);
                }
            }
        }
        emit_eobrun(e, st);
        e.w.flush();
        f.insert(f.end(), data.begin(), data.end());
    }
    f.push_back(0xFF);
    f.push_back(0xD9);
    if ((long)f.size() > out_cap) return -2;
    memcpy(out, f.data(), f.size());
    return (long)f.size();
}
