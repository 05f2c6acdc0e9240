// rod_jpegdec_host.h -- host side of the JPEG decoder: walk a file's markers, build the decoding tables
// (jdhuff.c jpeg_make_d_derived_tbl) and copy the entropy-coded segment without its 0xFF00 stuffing.
// Used by jpegdec.cu (results uploaded to the device) and by tests/emu (CPU check against cv2.imdecode).
#pragma once
#include <string.h>

#include <vector>

#include "rod_jpegdec.h"

namespace rod {
namespace jpegdec {

enum ParseStatus {
    PARSE_OK = 0,
    PARSE_NOT_JPEG = 1,          // no SOI / broken marker structure / truncated header
    PARSE_UNSUPPORTED = 2,       // a valid JPEG of another layout (progressive when not asked for, other sampling, CMYK,
                                 // EXIF rotation, a progression that leaves coefficient bits unknown ...)
    PARSE_NO_EOI = 3,            // a progressive file whose scans do not end in EOI (truncated)
};

// formats a caller takes (include/rod_b200.h ROD_JPEGDEC_BASELINE / ROD_JPEGDEC_PROGRESSIVE)
constexpr int kBaseline = 1, kProgressive = 2;

// One scan of a progressive file as the parser found it.  rec.image and the table indices are the caller's to fill in:
// dc_slot / ac_slot index FileInfo::huff (the tables in force at the scan's SOS).
struct ScanInfo {
    ScanRec rec;
    int dc_slot[3], ac_slot;
    int restart_interval;        // DRI in force at the scan's SOS
    size_t data_off, data_bytes; // the unstuffed data: out + data_off
    std::vector<uint32_t> rst;   // restart marker positions, relative to data_off
};

struct FileInfo {
    int height = 0, width = 0;
    int hs = 0, vs = 0, ncomp = 0;   // luma sampling (chroma 1 x 1), 3 components or 1
    int restart_interval = 0;        // MCUs per restart interval (DRI), 0: none
    size_t scan_begin = 0;       // first byte of the entropy-coded segment
    bool progressive = false;    // SOF2: scans, huff and the quantisation tables of the TableSet describe the file
    std::vector<ScanInfo> scans;
    std::vector<HuffTab> huff;
    size_t stream_bytes = 0;     // progressive: unstuffed bytes of all scans together
};

// true when an APP1 segment is an Exif block whose orientation tag is present and not 1 (cv2.imread would rotate the image)
inline bool exif_rotates(const uint8_t* p, size_t n) {
    if (n < 14 || memcmp(p, "Exif\0\0", 6) != 0) return false;
    const uint8_t* t = p + 6;
    const size_t tn = n - 6;
    const bool le = t[0] == 'I' && t[1] == 'I';
    if (!le && !(t[0] == 'M' && t[1] == 'M')) return true;   // malformed: leave the file to the host codec
    auto u16 = [&](size_t o) -> unsigned { return le ? (t[o] | (t[o + 1] << 8)) : ((t[o] << 8) | t[o + 1]); };
    auto u32 = [&](size_t o) -> size_t {
        return le ? ((size_t)t[o] | ((size_t)t[o + 1] << 8) | ((size_t)t[o + 2] << 16) | ((size_t)t[o + 3] << 24))
                  : (((size_t)t[o] << 24) | ((size_t)t[o + 1] << 16) | ((size_t)t[o + 2] << 8) | (size_t)t[o + 3]);
    };
    const size_t ifd = u32(4);
    if (ifd + 2 > tn) return true;
    const unsigned cnt = u16(ifd);
    for (unsigned i = 0; i < cnt; ++i) {
        const size_t e = ifd + 2 + 12u * i;
        if (e + 12 > tn) return true;
        if (u16(e) == 0x0112) return u16(e + 8) != 1;
    }
    return false;
}

inline void derive_table(const uint8_t* bits /* [16] */, const uint8_t* vals, int nvals, HuffTab* t) {
    memset(t, 0, sizeof(*t));
    memcpy(t->huffval, vals, (size_t)nvals);
    int code = 0, k = 0;
    for (int l = 1; l <= 16; ++l) {
        if (bits[l - 1]) {
            t->valoffset[l] = k - code;
            for (int i = 0; i < bits[l - 1]; ++i, ++k, ++code) {
                if (l <= kLook) {
                    const int first = code << (kLook - l), cnt = 1 << (kLook - l);
                    for (int q = 0; q < cnt; ++q) t->look[first + q] = (uint16_t)((l << 8) | vals[k]);
                }
            }
            t->maxcode[l] = code - 1;
        } else {
            t->maxcode[l] = -1;
        }
        code <<= 1;
    }
    t->maxcode[17] = 0xFFFFF;
    t->maxcode[0] = -1;
}

// Copies the entropy-coded data f[begin ..] into out (nullptr: only walks it) without the stuffed zero bytes and without the
// restart markers, whose positions in `out` (= the starts of the following intervals) are appended to *rst, up to the first
// other marker; *marker receives its position (n when the data runs to the end of the file).  out must hold n - begin + 16
// bytes; the 16 bytes behind the returned length are zeroed.  Returns the length.
inline size_t unstuff_segment(const uint8_t* f, size_t n, size_t begin, uint8_t* out, std::vector<uint32_t>* rst, size_t* marker) {
    size_t o = 0, i = begin;
    *marker = n;
    while (i < n) {
        const uint8_t* q = static_cast<const uint8_t*>(memchr(f + i, 0xFF, n - i));
        const size_t run = q ? (size_t)(q - (f + i)) : n - i;
        if (out) memcpy(out + o, f + i, run);
        o += run;
        i += run;
        if (!q) break;
        if (i + 1 >= n) break;
        const uint8_t m = f[i + 1];
        if (m == 0x00) { if (out) out[o] = 0xFF; ++o; i += 2; continue; }
        if (m == 0xFF) { ++i; continue; }   // fill byte
        if (m >= 0xD0 && m <= 0xD7) { if (rst) rst->push_back((uint32_t)o); i += 2; continue; }
        *marker = i;
        break;
    }
    if (out) memset(out + o, 0, 16);
    return o;
}

// The one scan of a baseline file: as unstuff_segment; returns (size_t)-1 when the data does not end in EOI (further
// scans, truncated file).
inline size_t unstuff_scan(const uint8_t* f, size_t n, size_t begin, uint8_t* out, std::vector<uint32_t>* rst) {
    size_t marker;
    const size_t o = unstuff_segment(f, n, begin, out, rst, &marker);
    return marker + 1 < n && f[marker + 1] == 0xD9 ? o : (size_t)-1;
}

// Walks the markers.  Baseline file: up to SOS; on PARSE_OK `ts` is complete and info->scan_begin points behind the SOS
// segment.  Progressive file (only when `formats` has kProgressive): up to EOI; every scan is checked the way jdphuff.c
// start_pass_phuff_decoder does (but reported, not warned about), its data unstuffed into out + info->stream_bytes (out:
// n + 16 bytes, or nullptr to only check the file), and `ts` receives the quantisation tables as libjpeg latches them at
// each component's first scan.
inline ParseStatus parse_file(const uint8_t* f, size_t n, FileInfo* info, TableSet* ts, int formats = kBaseline, uint8_t* out = nullptr) {
    memset(ts, 0, sizeof(*ts));
    *info = FileInfo();
    if (n < 4 || f[0] != 0xFF || f[1] != 0xD8) return PARSE_NOT_JPEG;
    uint16_t qt[4][64];
    bool have_q[4] = {false, false, false, false}, high_slot = false;
    int cur_dc[4] = {-1, -1, -1, -1}, cur_ac[4] = {-1, -1, -1, -1};   // the table in each slot: index into info->huff
    int tq[3] = {0, 0, 0}, comp_id[3] = {0, 0, 0};
    bool have_sof = false, adobe = false;
    int coef_bits[3][64];        // progressive: the Al each coefficient was last coded with, -1 before its first scan
    bool latched[3] = {false, false, false};
    for (int c = 0; c < 3; ++c)
        for (int k = 0; k < 64; ++k) coef_bits[c][k] = -1;
    info->huff.reserve(8);
    size_t i = 2;
    for (;;) {
        if (i >= n || f[i] != 0xFF) return PARSE_NOT_JPEG;
        while (i + 1 < n && f[i + 1] == 0xFF) ++i;   // fill bytes
        if (i + 2 > n) return PARSE_NOT_JPEG;
        const int m = f[i + 1];
        if (m == 0xD9) {   // (ends a progressive file; a baseline one ends its walk at SOS)
            if (info->scans.empty()) return PARSE_NOT_JPEG;
            // every coefficient complete: otherwise libjpeg would block-smooth or leave bits unknown
            for (int c = 0; c < info->ncomp; ++c)
                for (int k = 0; k < 64; ++k)
                    if (coef_bits[c][k] != 0) return PARSE_UNSUPPORTED;
            return PARSE_OK;
        }
        if (i + 4 > n) return PARSE_NOT_JPEG;
        if (m == 0xD8 || (m >= 0xD0 && m <= 0xD7) || m == 0x01) { i += 2; continue; }
        const size_t L = ((size_t)f[i + 2] << 8) | f[i + 3];
        if (L < 2 || i + 2 + L > n) return PARSE_NOT_JPEG;
        const uint8_t* p = f + i + 4;
        const size_t pl = L - 2;
        if (m == 0xDB) {
            size_t o = 0;
            while (o < pl) {
                const int pq = p[o] >> 4, t = p[o] & 15;
                if (t > 3) return PARSE_NOT_JPEG;
                if (pq != 0) return PARSE_UNSUPPORTED;   // 16-bit tables
                if (o + 65 > pl) return PARSE_NOT_JPEG;
                // libjpeg latched the table at the first scan of its components: a redefinition is not taken
                for (int c = 0; c < info->ncomp; ++c)
                    if (latched[c] && tq[c] == t) return PARSE_UNSUPPORTED;
                for (int z = 0; z < 64; ++z) qt[t][rod::jpeg::natural_order(z)] = p[o + 1 + z];
                have_q[t] = true;
                o += 65;
            }
        } else if (m == 0xC0 || (m == 0xC2 && (formats & kProgressive))) {
            if (have_sof) return PARSE_UNSUPPORTED;
            if (pl < 6) return PARSE_NOT_JPEG;
            if (p[0] != 8 || (p[5] != 3 && p[5] != 1) || pl < 6 + 3u * p[5]) return PARSE_UNSUPPORTED;
            info->height = (p[1] << 8) | p[2];
            info->width = (p[3] << 8) | p[4];
            info->ncomp = p[5];
            info->progressive = m == 0xC2;
            for (int c = 0; c < info->ncomp; ++c) {
                const int id = p[6 + 3 * c], hs = p[7 + 3 * c] >> 4, vs = p[7 + 3 * c] & 15;
                comp_id[c] = id;
                if (info->ncomp == 3 && id != c + 1) return PARSE_UNSUPPORTED;   // libjpeg's YCbCr guess: ids 1, 2, 3 (or a JFIF marker)
                if (c == 0) { info->hs = hs; info->vs = vs; }
                else if (hs != 1 || vs != 1) return PARSE_UNSUPPORTED;
                tq[c] = p[8 + 3 * c];
                if (tq[c] > 3) return PARSE_NOT_JPEG;
            }
            if (info->ncomp == 1) info->hs = info->vs = 1;   // a single-component scan is not interleaved: one block per MCU
            if (!((info->hs == 2 && info->vs == 2) || (info->hs == 2 && info->vs == 1) || (info->hs == 1 && info->vs == 1)))
                return PARSE_UNSUPPORTED;
            // one or two chroma columns: libjpeg-turbo's upsampler reads its padding there
            if (info->height < 1 || info->width < (info->hs == 2 ? 5 : 1)) return PARSE_UNSUPPORTED;
            have_sof = true;
        } else if (m >= 0xC1 && m <= 0xCF && m != 0xC4 && m != 0xC8 && m != 0xCC) {
            return PARSE_UNSUPPORTED;   // extended, progressive (when not asked for), lossless, arithmetic
        } else if (m == 0xC4) {
            size_t o = 0;
            while (o < pl) {
                if (o + 17 > pl) return PARSE_NOT_JPEG;
                const int tc = p[o] >> 4, th = p[o] & 15;
                if (tc > 1 || th > 3) return PARSE_NOT_JPEG;
                if (th > 1) {   // baseline files keep to slots 0 and 1; progressive ones may use all four
                    if (!(formats & kProgressive)) return PARSE_UNSUPPORTED;
                    high_slot = true;
                }
                int total = 0;
                for (int l = 0; l < 16; ++l) total += p[o + 1 + l];
                if (total > 256 || o + 17 + total > pl) return PARSE_NOT_JPEG;
                info->huff.emplace_back();
                derive_table(p + o + 1, p + o + 17, total, &info->huff.back());
                (tc == 0 ? cur_dc : cur_ac)[th] = (int)info->huff.size() - 1;
                o += 17 + (size_t)total;
            }
        } else if (m == 0xDD) {
            if (pl < 2) return PARSE_NOT_JPEG;
            info->restart_interval = (p[0] << 8) | p[1];
        } else if (m == 0xE1) {
            if (exif_rotates(p, pl)) return PARSE_UNSUPPORTED;
        } else if (m == 0xEE) {
            if (pl >= 12 && memcmp(p, "Adobe", 5) == 0) adobe = true;
        } else if (m == 0xDA && !info->progressive) {
            if (!have_sof) return PARSE_NOT_JPEG;
            const int nc = info->ncomp;
            if (pl < 4 + 2u * nc || p[0] != nc) return PARSE_UNSUPPORTED;   // one scan with all components
            if (high_slot) return PARSE_UNSUPPORTED;
            for (int c = 0; c < nc; ++c) {
                if (p[1 + 2 * c] != comp_id[c]) return PARSE_UNSUPPORTED;
                ts->comp_dc[c] = p[2 + 2 * c] >> 4;
                ts->comp_ac[c] = p[2 + 2 * c] & 15;
                if (ts->comp_dc[c] > 1 || ts->comp_ac[c] > 1) return PARSE_UNSUPPORTED;
                if (cur_dc[ts->comp_dc[c]] < 0 || cur_ac[ts->comp_ac[c]] < 0 || !have_q[tq[c]]) return PARSE_NOT_JPEG;
                memcpy(ts->quant[c], qt[tq[c]], sizeof(qt[0]));
            }
            if (p[1 + 2 * nc] != 0 || p[2 + 2 * nc] != 63 || p[3 + 2 * nc] != 0) return PARSE_UNSUPPORTED;
            if (adobe) return PARSE_UNSUPPORTED;   // Adobe marker: the colour transform is the marker's, not JFIF's
            info->scan_begin = i + 2 + L;
            // only the slots in use are copied: tables of unused slots must not make two equal files look different
            for (int c = 0; c < nc; ++c) {
                ts->dc[ts->comp_dc[c]] = info->huff[cur_dc[ts->comp_dc[c]]];
                ts->ac[ts->comp_ac[c]] = info->huff[cur_ac[ts->comp_ac[c]]];
            }
            info->huff.clear();
            return PARSE_OK;
        } else if (m == 0xDA) {   // a scan of a progressive file
            if (adobe) return PARSE_UNSUPPORTED;
            const int ns = pl >= 1 ? p[0] : 0;
            if (ns < 1 || ns > 3 || pl != 4 + 2u * ns) return PARSE_NOT_JPEG;
            ScanInfo sc;
            memset(&sc.rec, 0, sizeof(sc.rec));
            sc.rec.ncomp = (uint8_t)ns;
            const int Ss = p[1 + 2 * ns], Se = p[2 + 2 * ns], Ah = p[3 + 2 * ns] >> 4, Al = p[3 + 2 * ns] & 15;
            sc.rec.Ss = (uint8_t)Ss; sc.rec.Se = (uint8_t)Se; sc.rec.Ah = (uint8_t)Ah; sc.rec.Al = (uint8_t)Al;
            bool bad = Ss == 0 ? Se != 0 : (Ss > Se || Se > 63 || ns != 1);
            if (Ah != 0 && Al != Ah - 1) bad = true;
            if (Al > 13) bad = true;
            if (bad) return PARSE_UNSUPPORTED;
            sc.ac_slot = -1;
            int prev = -1;
            for (int j = 0; j < ns; ++j) {
                int c = 0;
                while (c < info->ncomp && comp_id[c] != p[1 + 2 * j]) ++c;
                if (c == info->ncomp) return PARSE_NOT_JPEG;
                if (c <= prev) return PARSE_UNSUPPORTED;   // components in frame order, each once
                prev = c;
                sc.rec.comp[j] = (uint8_t)c;
                const int td = p[2 + 2 * j] >> 4, ta = p[2 + 2 * j] & 15;
                if (td > 3 || ta > 3) return PARSE_NOT_JPEG;
                sc.dc_slot[j] = (Ss == 0 && Ah == 0) ? cur_dc[td] : -1;
                if (Ss == 0 && Ah == 0 && sc.dc_slot[j] < 0) return PARSE_NOT_JPEG;
                if (Ss > 0) {
                    sc.ac_slot = cur_ac[ta];
                    if (sc.ac_slot < 0) return PARSE_NOT_JPEG;
                }
                int* bits = coef_bits[c];
                if (Ss > 0 && bits[0] < 0) return PARSE_UNSUPPORTED;   // AC before the component's first DC scan
                for (int k = Ss; k <= Se; ++k) {
                    if (Ah != (bits[k] < 0 ? 0 : bits[k])) return PARSE_UNSUPPORTED;   // bogus progression
                    bits[k] = Al;
                }
                if (!latched[c]) {
                    if (!have_q[tq[c]]) return PARSE_NOT_JPEG;
                    memcpy(ts->quant[c], qt[tq[c]], sizeof(qt[0]));
                    latched[c] = true;
                }
            }
            for (int j = ns; j < 3; ++j) sc.dc_slot[j] = -1;
            sc.restart_interval = info->restart_interval;
            sc.data_off = info->stream_bytes;
            size_t marker;
            sc.data_bytes = unstuff_segment(f, n, i + 2 + L, out ? out + info->stream_bytes : nullptr, &sc.rst, &marker);
            info->stream_bytes += sc.data_bytes;
            if (marker == n) return PARSE_NO_EOI;
            info->scans.push_back(std::move(sc));
            i = marker;
            continue;
        }
        i += 2 + L;
    }
}

}  // namespace jpegdec
}  // namespace rod

namespace rod {
namespace jpegdec {

// The restart intervals of one image as segment records.  slot: 4-byte aligned offset of the image's unstuffed scan in the
// stream buffer, sb its length, rst the interval starts found by unstuff_scan.  false: the markers do not match the DRI.
inline bool make_segments(const ImageRec& im, uint32_t image, int restart_interval, uint64_t slot, size_t sb,
                          const std::vector<uint32_t>& rst, std::vector<SegRec>* out) {
    const Layout L = layout_of(im);
    const long ri = restart_interval > 0 ? restart_interval : L.mcus;
    const long n_seg = (L.mcus + ri - 1) / ri;
    if ((long)rst.size() != n_seg - 1) return false;
    for (long q = 0; q < n_seg; ++q) {
        const uint64_t b0 = q == 0 ? 0 : rst[q - 1], b1 = q + 1 < n_seg ? rst[q] : sb;
        if (b1 < b0) return false;
        SegRec sg;
        const uint64_t abs0 = slot + b0;
        sg.stream_off = abs0 & ~(uint64_t)3;
        sg.byte0 = (uint32_t)(abs0 & 3);
        sg.stream_bytes = sg.byte0 + (uint32_t)(b1 - b0);
        sg.image = image;
        sg.first_block = (uint32_t)(q * ri * L.nb);
        sg.n_blocks = (uint32_t)((q + 1 < n_seg ? ri : L.mcus - q * ri) * L.nb);
        sg.pad = 0;
        out->push_back(sg);
    }
    return true;
}

// The restart intervals of one progressive scan as segment records (units: MCUs of an interleaved scan, blocks of a
// non-interleaved one; the DRI counts those).  slot: offset of the image's unstuffed scans in the stream buffer.  false:
// the markers do not match the DRI.
inline bool make_scan_segments(const ImageRec& im, const ScanInfo& si, uint32_t scan, uint64_t slot, std::vector<ScanSeg>* out) {
    const long units = (long)scan_units(im, si.rec);
    const long ri = si.restart_interval > 0 ? si.restart_interval : units;
    const long n_seg = (units + ri - 1) / ri;
    if ((long)si.rst.size() != n_seg - 1) return false;
    for (long q = 0; q < n_seg; ++q) {
        const uint64_t b0 = q == 0 ? 0 : si.rst[q - 1], b1 = q + 1 < n_seg ? si.rst[q] : si.data_bytes;
        if (b1 < b0) return false;
        ScanSeg sg;
        const uint64_t abs0 = slot + si.data_off + b0;
        sg.stream_off = abs0 & ~(uint64_t)3;
        sg.byte0 = (uint32_t)(abs0 & 3);
        sg.stream_bytes = sg.byte0 + (uint32_t)(b1 - b0);
        sg.scan = scan;
        sg.first_unit = (uint32_t)(q * ri);
        sg.n_units = (uint32_t)(q + 1 < n_seg ? ri : units - q * ri);
        sg.pad = 0;
        out->push_back(sg);
    }
    return true;
}

// Dependency levels of a progressive file's scans: a scan runs after every earlier scan that shares a component and a
// coefficient with it (a refinement reads what they wrote).  Scans of disjoint bands or components share a level, so
// libjpeg's default script takes three: the first scans; the DC, chroma and luma Al 2 -> 1 refinements; the last luma one.
inline int scan_levels(const std::vector<ScanInfo>& scans, std::vector<int>* level) {
    level->assign(scans.size(), 0);
    int n_levels = 0;
    for (size_t s = 0; s < scans.size(); ++s) {
        const ScanRec& b = scans[s].rec;
        for (size_t t = 0; t < s; ++t) {
            const ScanRec& a = scans[t].rec;
            if (a.Se < b.Ss || b.Se < a.Ss) continue;
            bool shared = false;
            for (int i = 0; i < a.ncomp; ++i)
                for (int j = 0; j < b.ncomp; ++j) shared |= a.comp[i] == b.comp[j];
            if (shared && (*level)[t] + 1 > (*level)[s]) (*level)[s] = (*level)[t] + 1;
        }
        if ((*level)[s] + 1 > n_levels) n_levels = (*level)[s] + 1;
    }
    return n_levels;
}

}  // namespace jpegdec
}  // namespace rod
