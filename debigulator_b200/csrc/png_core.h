// png_core.h -- device code for the PNG container path (sm_100a), one warp per
// image. Replaces the data-touching parts of the reference's decode_png()
// (decode_png.c:683-1567):
//
//   png_scan_warp      signature + chunk walk (:730-1355) with the reference's
//                      own bookkeeping, per-chunk CRC-32 (update_crc :313-333,
//                      table :29-286) computed by 32 lanes over 8 KiB tiles and
//                      recombined in GF(2), IHDR / PLTE / zlib-header
//                      validation (:900-1277) and the IDAT concatenation
//                      (:1285-1291) into a compact per-image zlib stream.
//   png_unfilter_warp  scanline reconstruction (:1381-1507, undo_PNG_filter
//                      :497-541, Paeth :441-487) as a 32-row skewed wavefront:
//                      lane j owns row r0+j and runs j pixels behind lane j-1,
//                      taking `b`/`c` from its neighbour by shuffle; tiles are
//                      staged through shared memory so global loads and stores
//                      stay row-contiguous. Palette expansion (:1538-1564) and
//                      RGB->RGBA are fused into the tile write-out.
//
// The reference's bookkeeping quirks are kept (Q11: IHDR/PLTE/zlib-header bytes
// are not subtracted from the remaining-size counter; ancillary test is a
// signed `char > 'Z'`), with real bounds checks added so nothing is read
// outside the file. Known, documented divergences: D1 (the reference corrupts
// the last <=771 stream bytes when a late deflate block starts, see DESIGN.md),
// D3 (the reference's RGB expansion is broken; this one is correct).
#pragma once
#include "inflate_core.h"
#include "simt.h"

#ifdef DBG_SIMT_EMU
static inline uint32_t atomicAdd(uint32_t *p, uint32_t v) { uint32_t o = *p; *p = o + v; return o; }
static inline uint32_t atomicXor(uint32_t *p, uint32_t v) { uint32_t o = *p; *p = o ^ v; return o; }
struct uint4 { uint32_t x, y, z, w; };
#endif

namespace dbg {

enum : uint32_t {
    ST_PNG_CRC = 13,
    ST_PNG_FILTER = 14,
    ST_PNG_SHORT = 15,
};

struct PngInfo {
    uint32_t w, h;
    uint32_t bpp;        // bytes per pixel in the filtered stream: 4 (ct 6), 3 (ct 2), 1 (ct 3)
    uint32_t plte_off;   // file offset of the PLTE payload (ct 3)
    uint32_t plte_size;  // entries
    uint32_t pad[3];
};

// ------------------------------------------------------------------ CRC-32 ----
constexpr uint32_t CRC_POLY = 0xedb88320u;  // decode_png.c:289-304
constexpr uint32_t CRC_SLICE = 256;         // bytes per lane per tile
constexpr uint32_t CRC_TILE = 32 * CRC_SLICE;

struct CrcTables {
    uint32_t t[4][256];  // slicing-by-4: t[k][b] = CRC state of byte b followed by k zero bytes
};

// a(x) * b(x) mod P in the reflected representation (bit 31 = x^0).
DBG_DEV uint32_t gf2_mulmod(uint32_t a, uint32_t b)
{
    uint32_t p = 0;
    for (int i = 31; i >= 0; i--) {
        p ^= (0u - ((a >> i) & 1u)) & b;
        b = (b >> 1) ^ (CRC_POLY & (0u - (b & 1u)));
    }
    return p;
}
// x^(8*nbytes) mod P
DBG_DEV uint32_t gf2_xpow_bytes(uint32_t nbytes)
{
    uint32_t sq = 0x00800000u;  // x^8
    uint32_t r = 0x80000000u;   // x^0
    while (nbytes) {
        if (nbytes & 1) r = gf2_mulmod(sq, r);
        sq = gf2_mulmod(sq, sq);
        nbytes >>= 1;
    }
    return r;
}

// Fill the slicing tables; `tid`/`nthreads` enumerate the cooperating threads.
DBG_DEV void crc_tables_init(CrcTables *T, int tid, int nthreads)
{
    for (int i = tid; i < 256; i += nthreads) {
        uint32_t c = (uint32_t)i;
        for (int k = 0; k < 8; k++) c = (c >> 1) ^ (CRC_POLY & (0u - (c & 1u)));
        uint32_t c1 = c, c2, c3;
        // appending one zero byte to state s: (s >> 8) ^ t0[s & 255]; t0 itself
        // is still being written by other threads, so recompute it locally.
        uint32_t lo = c1 & 255, z = lo;
        for (int k = 0; k < 8; k++) z = (z >> 1) ^ (CRC_POLY & (0u - (z & 1u)));
        c2 = (c1 >> 8) ^ z;
        lo = c2 & 255, z = lo;
        for (int k = 0; k < 8; k++) z = (z >> 1) ^ (CRC_POLY & (0u - (z & 1u)));
        c3 = (c2 >> 8) ^ z;
        lo = c3 & 255, z = lo;
        for (int k = 0; k < 8; k++) z = (z >> 1) ^ (CRC_POLY & (0u - (z & 1u)));
        uint32_t c4 = (c3 >> 8) ^ z;
        T->t[0][i] = c1;
        T->t[1][i] = c2;
        T->t[2][i] = c3;
        T->t[3][i] = c4;
    }
}

DBG_DEV uint32_t crc_slice(const CrcTables *T, uint32_t c, const uint8_t *p, uint32_t len)
{
    while (len && ((uintptr_t)p & 3)) {
        c = T->t[0][(c ^ *p) & 255] ^ (c >> 8);
        p++;
        len--;
    }
    while (len >= 4) {
        c ^= *(const uint32_t *)p;
        c = T->t[3][c & 255] ^ T->t[2][(c >> 8) & 255] ^ T->t[1][(c >> 16) & 255] ^ T->t[0][c >> 24];
        p += 4;
        len -= 4;
    }
    while (len) {
        c = T->t[0][(c ^ *p) & 255] ^ (c >> 8);
        p++;
        len--;
    }
    return c;
}

// CRC-32 (init and final xor 0xFFFFFFFF, decode_png.c:766,873) of p[0..n), n >= 1,
// computed by the whole warp. `lane_k` must hold x^(8*CRC_SLICE*(31-lane)).
// The region is cut into 8 KiB tiles counted from its END, so only the first
// tile is partial and every lane's "bytes after my slice" count is a constant.
// Raw CRC register after feeding p[0..n) to a register that starts at `init` (no final xor): the
// building block for regions that are split over several warps.
DBG_DEV uint32_t crc_state_warp(const CrcTables *T, uint32_t lane_k, const uint8_t *p, uint64_t n, uint32_t init)
{
    const uint32_t ln = (uint32_t)simt::lane();
    uint32_t head = (uint32_t)(n % CRC_TILE);
    uint32_t running = init;
    bool first = true;
    uint64_t done = 0;
    while (done < n) {
        uint32_t tlen = (first && head) ? head : CRC_TILE;  // real bytes in this tile
        uint32_t vstart = CRC_TILE - tlen;                  // virtual offset of the first real byte
        uint32_t s0 = ln * CRC_SLICE, s1 = s0 + CRC_SLICE;  // my virtual slice
        uint32_t c = 0;
        if (s1 > vstart) {
            uint32_t b0 = s0 > vstart ? s0 : vstart;
            bool has_first = (b0 == vstart);
            if (has_first) c = running;
            c = crc_slice(T, c, p + done + (b0 - vstart), s1 - b0);
            c = gf2_mulmod(lane_k, c);
        }
        for (int d = 16; d; d >>= 1) c ^= simt::shfl_xor(c, d);
        running = c;
        done += tlen;
        first = false;
    }
    return running;
}

DBG_DEV uint32_t crc32_warp(const CrcTables *T, uint32_t lane_k, const uint8_t *p, uint64_t n)
{
    return crc_state_warp(T, lane_k, p, n, 0xffffffffu) ^ 0xffffffffu;
}

// Work that one warp per image would serialise (a 150 MB IDAT chunk) is handed to a second
// kernel as 64 KiB segment tasks: CRC-32 segments (recombined in GF(2): the contribution of a
// segment is its raw register times x^(8 * bytes after it), XOR-accumulated per chunk) and
// IDAT copy segments.
constexpr uint32_t SCAN_SEG = 65536;
constexpr uint32_t SCAN_NONE = 0xffffffffu;
struct ScanTask {
    const uint8_t *src;
    uint8_t *dst;          // nullptr: CRC only
    uint32_t len;
    uint32_t bytes_after;  // bytes of the CRC region after this segment
    uint32_t big;          // accumulator index, SCAN_NONE: copy only
    uint32_t first;        // 1: the register starts at 0xFFFFFFFF
};
struct BigChunk {
    uint32_t img, expected, acc, armed;  // armed: `expected` is valid (the walk got as far as the stored CRC)
};
struct ScanQueues {
    ScanTask *tasks;
    uint32_t *ntasks;
    uint32_t task_cap;
    BigChunk *big;
    uint32_t *nbig;
    uint32_t big_cap;
};

// Enqueues segment tasks for region p[0..n) (uniform call). Returns false when the queue is full.
DBG_DEV bool scan_enqueue(ScanQueues *q, const uint8_t *p, uint64_t n, uint8_t *dst, uint32_t big)
{
    const uint32_t ln = (uint32_t)simt::lane();
    const uint32_t nseg = (uint32_t)((n + SCAN_SEG - 1) / SCAN_SEG);
    uint32_t base = 0;
    if (ln == 0) base = atomicAdd(q->ntasks, nseg);
    base = simt::shfl(base, 0);
    if (base + nseg > q->task_cap) {  // no room: the caller does the work itself; the slots that exist are marked empty
        for (uint32_t k = base + ln; k < q->task_cap; k += 32) q->tasks[k].len = 0;  // (the scratch is reused: no stale records)
        return false;
    }
    for (uint32_t k = ln; k < nseg; k += 32) {
        ScanTask t;
        uint64_t o = (uint64_t)k * SCAN_SEG;
        t.src = p + o;
        t.dst = dst ? dst + o : nullptr;
        t.len = (uint32_t)(n - o < SCAN_SEG ? n - o : SCAN_SEG);
        t.bytes_after = (uint32_t)(n - o - t.len);
        t.big = big;
        t.first = k == 0;
        q->tasks[base + k] = t;
    }
    return true;
}

// One segment task (png_tasks_kernel, uniform call): its contribution to the CRC of its chunk, XOR-ed into the chunk's
// accumulator, and its copy.
DBG_DEV void scan_task_run(const CrcTables *T, uint32_t lane_k, const ScanTask &k, BigChunk *big)
{
    const uint32_t ln = (uint32_t)simt::lane();
    if (k.big != SCAN_NONE) {
        uint32_t st = crc_state_warp(T, lane_k, k.src, k.len, k.first ? 0xffffffffu : 0u);
        st = gf2_mulmod(gf2_xpow_bytes(k.bytes_after), st);
        if (ln == 0) atomicXor(&big[k.big].acc, st);
    }
    if (k.dst) {
        if ((((uintptr_t)k.src | (uintptr_t)k.dst) & 15) == 0) {
            const uint4 *s4 = (const uint4 *)k.src;
            uint4 *d4 = (uint4 *)k.dst;
            for (uint32_t i = ln; i < k.len / 16; i += 32) d4[i] = s4[i];
            for (uint32_t i = (k.len & ~15u) + ln; i < k.len; i += 32) k.dst[i] = k.src[i];
        } else {
            for (uint32_t i = ln; i < k.len; i += 32) k.dst[i] = k.src[i];
        }
    }
}

// png_verify_kernel: the recombined CRC of a large chunk against the stored one (decode_png.c:1341-1348), once every
// segment task has run. A chunk the walk never got to the end of is not armed and fails on its own account.
DBG_DEV bool big_chunk_crc_bad(const BigChunk &c) { return c.armed && (c.acc ^ 0xffffffffu) != c.expected; }

// --------------------------------------------------------------- chunk walk ----
DBG_DEV uint32_t be32(const uint8_t *p)
{
    return ((uint32_t)p[0] << 24) | ((uint32_t)p[1] << 16) | ((uint32_t)p[2] << 8) | (uint32_t)p[3];
}
DBG_DEV bool tag_is(const uint8_t *p, char a, char b, char c, char d)
{
    return p[0] == (uint8_t)a && p[1] == (uint8_t)b && p[2] == (uint8_t)c && p[3] == (uint8_t)d;
}

// Walks one PNG file. Uniform across the warp. On success returns ST_OK, fills
// `info`, and has copied the concatenated IDAT payload (minus the 2-byte zlib
// header) to `zdst`; *z_size is the deflate size handed to inflate
// (payload - 4, decode_png.c:816).
// With a single IDAT chunk (every stb-written PNG) nothing is copied: *z_ptr points into the file.
// `q` (may be null) receives the CRC / copy work of chunks larger than SCAN_SEG.
DBG_DEV uint32_t png_scan_warp(const CrcTables *T, uint32_t lane_k, const uint8_t *file, uint64_t size,
                               uint64_t rgba_size, uint8_t *zdst, uint64_t zcap, PngInfo *info, uint64_t *z_size,
                               const uint8_t **z_ptr, ScanQueues *q, uint32_t img)
{
    const uint32_t ln = (uint32_t)simt::lane();
    *z_size = 0;
    *z_ptr = zdst;
    uint64_t first_off = 0, first_len = 0;  // the first IDAT payload, not copied until a second one shows up
    uint32_t n_idat = 0;
    if (size < 8 || size >= (1ull << 32)) return ST_CONTAINER;
    if (!(file[1] == 'P' && file[2] == 'N' && file[3] == 'G')) return ST_CONTAINER;  // decode_png.c:730-753
    uint64_t pos = 8;
    uint64_t left = size - 8;
    bool found_idat = false, ran_inflate = false, found_ihdr = false, found_iend = false;
    uint64_t zlen = 0, zlen_at_run = 0;
    uint32_t w = 0, h = 0, ct = 0;
    info->plte_off = 0;
    info->plte_size = 0;
    while (left >= 8 && !found_iend) {  // decode_png.c:755-758
        if (pos + 8 > size) return ST_CONTAINER;
        const uint8_t *hdr = file + pos;
        uint64_t length = be32(hdr);
        const uint8_t *type = hdr + 4;
        pos += 8;
        left -= 8;
        bool is_idat = tag_is(type, 'I', 'D', 'A', 'T');
        if (!is_idat && found_idat) {  // decode_png.c:775-860: the point where the reference inflates
            ran_inflate = true;
            zlen_at_run = zlen;
        }
        if (length >= left) return ST_CONTAINER;            // decode_png.c:886
        if (pos + length + 4 > size) return ST_CONTAINER;   // real bounds (Q11 makes `left` optimistic)
        uint32_t crc = 0, big = SCAN_NONE;                      // decode_png.c:862-874
        if (q && 4 + length > SCAN_SEG) {
            uint32_t bi = 0;
            if (ln == 0) bi = atomicAdd(q->nbig, 1u);
            bi = simt::shfl(bi, 0);
            if (bi < q->big_cap) {
                if (ln == 0) {
                    BigChunk bc;
                    bc.img = img;
                    bc.expected = 0;
                    bc.acc = 0;
                    bc.armed = 0;
                    q->big[bi] = bc;
                }
                simt::syncwarp();
                if (scan_enqueue(q, type, 4 + length, nullptr, bi)) big = bi;
            }
        }
        if (big == SCAN_NONE) crc = crc32_warp(T, lane_k, type, 4 + length);
        if (tag_is(type, 'P', 'L', 'T', 'E')) {             // decode_png.c:900-950
            if (!found_ihdr) return ST_CONTAINER;
            if (length % 3 != 0) return ST_CONTAINER;
            info->plte_off = (uint32_t)pos;
            info->plte_size = (uint32_t)(length / 3);
            pos += length;
        } else if (tag_is(type, 'I', 'H', 'D', 'R')) {      // decode_png.c:951-1138
            found_ihdr = true;
            if (pos + 13 > size) return ST_CONTAINER;
            const uint8_t *b = file + pos;
            pos += 13;
            w = be32(b);
            h = be32(b + 4);
            uint32_t depth = b[8];
            ct = b[9];
            uint32_t filter_method = b[11];
            if ((uint64_t)w * h * 4 != rgba_size) return ST_CONTAINER;       // :970
            if ((uint64_t)w * h * 4 + h + 1 >= (1ull << 32)) return ST_TOO_LARGE;
            if (!(ct == 2 || ct == 3 || ct == 6)) return ST_CONTAINER;       // :987-1038
            if (w < 1 || h < 1) return ST_CONTAINER;                         // :1044
            if (depth != 8) return ST_CONTAINER;                             // :1088
            if (filter_method != 0) return ST_CONTAINER;                     // :1118
            if (left < 4) return ST_CONTAINER;                               // :1127
        } else if (is_idat) {                               // decode_png.c:1140-1292
            if (!found_ihdr) return ST_CONTAINER;
            uint64_t data_len = length;
            if (!found_idat) {
                found_idat = true;
                if (length < 2) return ST_CONTAINER;
                uint32_t cmf = file[pos], flg = file[pos + 1];
                pos += 2;
                data_len -= 2;
                if ((cmf & 15) != 8) return ST_CONTAINER;                    // :1186
                uint32_t chk = (cmf << 8) | flg;
                if (chk == 0 || chk % 31 != 0) return ST_CONTAINER;          // :1214-1220
                if ((flg >> 5) & 1) return ST_CONTAINER;                     // FDICT :1262-1265
            }
            if (zlen + data_len > zcap) return ST_CONTAINER;
            n_idat++;
            if (n_idat == 1) {
                first_off = pos;
                first_len = data_len;
            } else {                                                         // :1285-1291
                for (int pass = n_idat == 2 ? 0 : 1; pass < 2; pass++) {     // second IDAT: the first one moves too
                    const uint8_t *src = pass == 0 ? file + first_off : file + pos;
                    uint8_t *dst = pass == 0 ? zdst : zdst + zlen;
                    uint64_t cl = pass == 0 ? first_len : data_len;
                    if (!(q && cl > SCAN_SEG && scan_enqueue(q, src, cl, dst, SCAN_NONE)))
                        for (uint64_t i = ln; i < cl; i += 32) dst[i] = src[i];
                }
            }
            zlen += data_len;
            pos += data_len;
            left -= data_len;
        } else if (tag_is(type, 'I', 'E', 'N', 'D')) {      // :1293-1302
            found_iend = true;
        } else if ((int8_t)type[0] > (int8_t)'Z') {         // :1303-1308 ancillary (signed char compare)
            pos += length;
            left -= length;
        } else {
            return ST_CONTAINER;                            // :1309-1319 unknown critical chunk
        }
        if (left < 4) return ST_CONTAINER;                  // :1321
        if (pos + 4 > size) return ST_CONTAINER;
        uint32_t stored = be32(file + pos);
        pos += 4;
        left -= 4;
        if (big != SCAN_NONE) {                             // verified once the segment tasks have run
            if (ln == 0) {
                q->big[big].expected = stored;
                q->big[big].armed = 1;
            }
        } else if (stored != crc) return ST_PNG_CRC;        // :1341-1348
    }
    if (!ran_inflate) return ST_CONTAINER;                  // :1357
    if (zlen_at_run < 4 + 5) {
        // the reference hands (payload - 4) to inflate, which rejects < 5 bytes
        // (and the subtraction wraps below 4) -- inflate.c:836
        return zlen_at_run < 4 ? ST_CONTAINER : ST_INPUT_TOO_SMALL;
    }
    info->w = w;
    info->h = h;
    info->bpp = ct == 6 ? 4 : ct == 2 ? 3 : 1;              // :1401-1414
    if (n_idat == 1) *z_ptr = file + first_off;
    *z_size = zlen_at_run - 4;
    return ST_OK;
}

// ---------------------------------------------------------------- un-filter ----
constexpr int UNF_RS = 68;  // ring row stride in words: (UNF_RS - 1) odd keeps the skewed accesses of the wavefront conflict-free
struct UnfilterSmem {
    union {
        uint32_t tile[32][33];      // palette / RGB images (png_unfilter_band)
        uint32_t ring[33][UNF_RS];  // RGBA8 images (png_unfilter_band4): row 0 = last row of the band above, rows 1..32 = the
                                    // band, column = pixel x & 63 (two 32-pixel blocks: the one being staged / computed and the
                                    // one the skewed lanes are still finishing)
    };
};

DBG_DEV uint32_t swar_add4(uint32_t a, uint32_t b)
{
    return ((a & 0x7f7f7f7fu) + (b & 0x7f7f7f7fu)) ^ ((a ^ b) & 0x80808080u);
}
DBG_DEV uint32_t swar_havg4(uint32_t a, uint32_t b)  // per-byte floor((a+b)/2), decode_png.c:512-515
{
    return (a & b) + (((a ^ b) & 0xfefefefeu) >> 1);
}
DBG_DEV uint32_t paeth4(uint32_t a, uint32_t b, uint32_t c)  // decode_png.c:441-487, ties a -> b -> c
{
    uint32_t r = 0;
    for (int k = 0; k < 32; k += 8) {
        int ia = (int)((a >> k) & 255), ib = (int)((b >> k) & 255), ic = (int)((c >> k) & 255);
        int pa = ib - ic, pb = ia - ic, pc = ia + ib - 2 * ic;
        pa = pa < 0 ? -pa : pa;
        pb = pb < 0 ? -pb : pb;
        pc = pc < 0 ? -pc : pc;
        int pr = (pa <= pb && pa <= pc) ? ia : (pb <= pc ? ib : ic);
        r |= (uint32_t)pr << k;
    }
    return r;
}

// Four bytes at once. absdiff4 is one VABSDIFF4 on sm_100a; ge4_hi leaves x >= y in bit 7 of every byte (the other bits
// are garbage): bit 7 of the per-byte rounded-up average of x and 255 - y; sign_mask4 spreads bit 7 over its byte (PRMT).
#ifndef DBG_SIMT_EMU
DBG_DEV uint32_t absdiff4(uint32_t a, uint32_t b) { return __vabsdiffu4(a, b); }
DBG_DEV uint32_t sign_mask4(uint32_t v)  // __byte_perm() drops the selector's replicate-sign bit, the instruction does not
{
    uint32_t r;
    asm("prmt.b32 %0, %1, %1, 0xba98;" : "=r"(r) : "r"(v));
    return r;
}
#else
DBG_DEV uint32_t absdiff4(uint32_t a, uint32_t b)
{
    uint32_t r = 0;
    for (int k = 0; k < 32; k += 8) {
        int x = (int)((a >> k) & 255) - (int)((b >> k) & 255);
        r |= (uint32_t)(x < 0 ? -x : x) << k;
    }
    return r;
}
DBG_DEV uint32_t sign_mask4(uint32_t v) { return ((v >> 7) & 0x01010101u) * 255u; }
#endif
DBG_DEV uint32_t ge4_hi(uint32_t x, uint32_t y)
{
    const uint32_t ny = ~y;
    return (x | ny) - (((x ^ ny) >> 1) & 0x7f7f7f7fu);
}
// Paeth predictor of four channels without leaving the 32-bit word (decode_png.c:441-487: pa = |b - c|, pb = |a - c|,
// pc = |a + b - 2c|, ties a -> b -> c). pc does not fit a byte, but it is never needed as a number: with x = b - c and
// y = a - c it is |x + y|, i.e. pa + pb (>= both, so c loses every comparison) when x and y have the same sign, and
// |pa - pb| when they do not; both forms agree when either is zero.
DBG_DEV uint32_t paeth4_swar(uint32_t a, uint32_t b, uint32_t c)
{
    const uint32_t pa = absdiff4(b, c), pb = absdiff4(a, c), pcd = absdiff4(pa, pb);
    const uint32_t same = ~(ge4_hi(b, c) ^ ge4_hi(a, c));
    const uint32_t sel_a = ge4_hi(pb, pa) & (same | ge4_hi(pcd, pa));
    const uint32_t sel_b = ~sel_a & (same | ge4_hi(pcd, pb));
    const uint32_t ma = sign_mask4(sel_a), mb = sign_mask4(sel_b);
    return (a & ma) | (~ma & ((b & mb) | (c & ~mb)));
}

template <int BPP>
DBG_DEV uint32_t load_px(const uint8_t *p)
{
    if (BPP == 4) {
        uintptr_t a = (uintptr_t)p;
        const uint32_t *q = (const uint32_t *)(a & ~(uintptr_t)3);
        uint32_t sh = (uint32_t)(a & 3) * 8;
        uint32_t lo = q[0];
        if (sh == 0) return lo;
        return simt::funnel_r(lo, q[1], sh);
    }
    uint32_t v = 0;
    for (int k = 0; k < BPP; k++) v |= (uint32_t)p[k] << (8 * k);
    return v;
}

// Up-row pixel written by ANOTHER warp (the band above): read it from L2, not from a
// possibly stale L1 line.
template <int BPP>
DBG_DEV uint32_t load_px_l2(const uint8_t *p)
{
    if (BPP == 4) return simt::ldcg_u32((const uint32_t *)p);  // RGBA output rows are 4-byte aligned
    uint32_t v = 0;
    for (int k = 0; k < BPP; k++) v |= simt::ldcg_u8(p + k) << (8 * k);
    return v;
}

enum { BAND_ROWS = 32, BAND_SLOTS = 128 };
constexpr uint32_t UNF4_MAX_W = 1u << 30;  // png_unfilter_band4 counts pixels in 32-bit signed integers

// Reconstructs band `band` (rows 32*band .. 32*band+31) of one image. `scan`
// holds h rows of (1 filter byte + w*BPP bytes); it is overwritten in place
// with reconstructed bytes when BPP != 4 (those rows are the "previous
// scanline" of the next band). RGBA pixels go to `out`.
//
// Bands of one image are processed by different warps as a pipeline: band b
// may work on tile k once band b-1 has finished tile k+1 (its last row is this
// band's `b`/`c` input). Progress is handed over through `prog`, a ring of
// BAND_SLOTS 64-bit words per image: slot (b % BAND_SLOTS) = (b+1) << 32 | tiles
// done. Work items are issued in (image, band) order, so the band above is
// always already running when a band waits for it. A slot is shared by bands b
// and b + BAND_SLOTS; band b therefore starts only after band b - (BAND_SLOTS-1)
// -- the last reader of the slot it is about to overwrite -- has finished, which
// bounds the pipeline depth at BAND_SLOTS - 1 bands.
template <int BPP>
DBG_DEV void png_unfilter_band(UnfilterSmem *sm, uint8_t *scan, uint32_t w, uint32_t h, uint8_t *out, const uint8_t *plte,
                               uint32_t plte_size, uint32_t band, uint64_t *prog)
{
    const uint32_t ln = (uint32_t)simt::lane();
    const uint64_t stride = (uint64_t)w * BPP + 1;
    const uint32_t mask = BPP == 4 ? 0xffffffffu : ((1u << (8 * (BPP & 3))) - 1);
    const uint32_t ntiles = (w + 31 + 31) / 32;
    uint32_t *out32 = (uint32_t *)out;
    const uint32_t r0 = band * BAND_ROWS;
    const uint32_t r = r0 + ln;
    const bool row_ok = r < h;
    const uint32_t ft = row_ok ? scan[(uint64_t)r * stride] : 0;
    uint32_t prev_out = 0, prev_b = 0;
    if (prog && band >= BAND_SLOTS - 1) {
        const uint32_t q = band - (BAND_SLOTS - 1);
        const uint64_t done = ((uint64_t)(q + 1) << 32) | ntiles;
        const uint64_t *slot = prog + (q & (BAND_SLOTS - 1));
        while (simt::ld_acquire_u64(slot) < done) simt::backoff();
        simt::syncwarp();
    }
    for (uint32_t k = 0; k < ntiles; k++) {
        // stage the skewed tile: row jj holds pixels [32k - jj, 32k - jj + 32)
        for (uint32_t jj = 0; jj < 32; jj++) {
            int64_t x = (int64_t)32 * k - jj + ln;
            uint32_t v = 0;
            if (r0 + jj < h && x >= 0 && x < (int64_t)w)
                v = load_px<BPP>(scan + (uint64_t)(r0 + jj) * stride + 1 + (uint64_t)x * BPP);
            sm->tile[jj][ln] = v;
        }
        // the band above must have finished the tiles that hold pixels [32k, 32k+32) of its last row
        uint32_t up_px = 0;
        if (r0 > 0) {
            if (prog) {
                const uint64_t need = ((uint64_t)band << 32) | (k + 2 < ntiles ? k + 2 : ntiles);
                const uint64_t *slot = prog + ((band - 1) & (BAND_SLOTS - 1));
                while (simt::ld_acquire_u64(slot) < need) simt::backoff();
                simt::syncwarp();
            }
            uint32_t x = 32 * k + ln;
            if (x < w) {
                if (BPP == 4) up_px = load_px_l2<4>((const uint8_t *)(out32 + (uint64_t)(r0 - 1) * w + x));
                else up_px = load_px_l2<BPP>(scan + (uint64_t)(r0 - 1) * stride + 1 + (uint64_t)x * BPP);
            }
        }
        simt::syncwarp();
        for (uint32_t i = 0; i < 32; i++) {
            int64_t x = (int64_t)32 * k + i - ln;
            uint32_t b_in = simt::shfl_up(prev_out, 1);
            uint32_t b0 = simt::shfl(up_px, (int)i);
            if (ln == 0) b_in = b0;
            bool px_ok = row_ok && x >= 0 && x < (int64_t)w;
            uint32_t cur = sm->tile[ln][i];
            uint32_t a = x > 0 ? prev_out : 0;
            uint32_t c = x > 0 ? prev_b : 0;
            uint32_t b = b_in;
            uint32_t o;
            switch (ft) {  // undo_PNG_filter decode_png.c:497-541
                case 0: o = cur; break;
                case 1: o = swar_add4(cur, a); break;
                case 2: o = swar_add4(cur, b); break;
                case 3: o = swar_add4(cur, swar_havg4(a, b)); break;
                case 4: o = swar_add4(cur, paeth4(a, b, c)); break;
                default: o = 0; break;  // :528-540 unknown filter -> 0 in the no-assert build
            }
            o &= mask;
            if (px_ok) {
                sm->tile[ln][i] = o;
                prev_out = o;
            } else {
                prev_out = 0;
            }
            prev_b = b_in;
        }
        simt::syncwarp();
        for (uint32_t jj = 0; jj < 32; jj++) {
            int64_t x = (int64_t)32 * k - jj + ln;
            if (r0 + jj < h && x >= 0 && x < (int64_t)w) {
                uint32_t v = sm->tile[jj][ln];
                uint64_t pix = (uint64_t)(r0 + jj) * w + (uint64_t)x;
                if (BPP == 4) {
                    out32[pix] = v;
                } else {
                    uint8_t *q = scan + (uint64_t)(r0 + jj) * stride + 1 + (uint64_t)x * BPP;
                    for (int kk = 0; kk < BPP; kk++) q[kk] = (uint8_t)(v >> (8 * kk));
                    if (BPP == 3) {
                        out32[pix] = v | 0xff000000u;
                    } else {  // palette, alpha forced to 255 (decode_png.c:1552-1560)
                        uint32_t rgb = 0;
                        if (v < plte_size) {
                            const uint8_t *e = plte + 3 * v;
                            rgb = (uint32_t)e[0] | ((uint32_t)e[1] << 8) | ((uint32_t)e[2] << 16);
                        }
                        out32[pix] = rgb | 0xff000000u;
                    }
                }
            }
        }
        simt::syncwarp();  // every lane's rows of this tile are written ...
        if (prog && ln == 0) {  // ... and published to the band below
            simt::threadfence();
            simt::st_release_u64(prog + (band & (BAND_SLOTS - 1)), ((uint64_t)(band + 1) << 32) | (k + 1));
        }
    }
}

// ------------------------------------------------ un-filter of RGBA8 bands by row class ----
// (decode_png.c:497-541; BASELINE configs 3 and 4.) A band's 32 filter bytes decide how it is reconstructed:
//   * None / Up rows only: every column is independent -- one lane per pixel column walks down the rows straight from the
//     scanlines to the RGBA output (elementwise, no shared memory, coalesced both ways);
//   * None / Sub rows only: every row is independent of the rows above -- one lane per row, running per-channel sum along the
//     row, and the band neither waits for the band above nor reads its last row;
//   * anything with Average or Paeth rows (or a mix of Sub and Up): the skewed wavefront -- lane j = row j, j pixels behind
//     lane j-1, `b` by shuffle, `c` = the previous `b`; all four channels of a pixel in one 32-bit word (paeth4_swar), the row's
//     filter applied through per-lane masks so that a band of mixed rows does not diverge. The Paeth arithmetic is compiled
//     in only for bands that have a Paeth row.
// The row-per-lane forms work on a shared-memory ring of two 32-pixel blocks per row: block k is staged (coalesced reads,
// the scanline's odd byte offset removed by a funnel shift), the lanes run their 32 steps, and block k-1 -- finished by every
// lane by then -- is written out with coalesced stores. Progress towards the band below is published in the same units
// as png_unfilter_band: t tiles done = pixels [0, 32 (t-1)) of every row are in `out`.
DBG_DEV void unf4_publish(uint64_t *prog, uint32_t band, uint32_t tiles)
{
    simt::syncwarp();  // orders the other lanes' stores before lane 0's release (which is a fence of its own: no __threadfence())
    if (prog && simt::lane() == 0) simt::st_release_u64(prog + (band & (BAND_SLOTS - 1)), ((uint64_t)(band + 1) << 32) | tiles);
}
DBG_DEV void unf4_wait_above(const uint64_t *prog, uint32_t band, uint32_t tiles)
{
    if (prog) {
        const uint64_t need = ((uint64_t)band << 32) | tiles;
        const uint64_t *slot = prog + ((band - 1) & (BAND_SLOTS - 1));
        while (simt::ld_acquire_u64(slot) < need) simt::backoff();
        simt::syncwarp();
    }
}

// Pixels [32k, 32k + 32) of the band's rows into registers, one row per register: one aligned word per lane, the next word
// from the lane above it (lane 31 loads its own), the scanline's byte offset (1 filter byte + 4 * pixels: any alignment)
// removed by a funnel shift. All loads are issued before the first is used.
DBG_DEV void unf4_load_block(const uint8_t *scan, uint64_t stride, uint32_t r0, uint32_t rows, uint32_t x_blk, uint32_t w,
                             uint32_t (&v)[32])
{
    const uint32_t ln = (uint32_t)simt::lane();
    uint32_t hi31[32];
#pragma unroll
    for (uint32_t jj = 0; jj < 32; jj++) {
        v[jj] = 0;
        hi31[jj] = 0;
        if (jj < rows) {
            const uintptr_t p = (uintptr_t)(scan + (uint64_t)(r0 + jj) * stride + 1 + (uint64_t)x_blk * 4);
            const uint32_t *q = (const uint32_t *)(p & ~(uintptr_t)3);
            if (x_blk <= w) v[jj] = q[0];  // the word after the last pixel's holds its last 1..3 bytes
            if (ln == 31 && x_blk < w && (p & 3)) hi31[jj] = q[1];
        }
    }
#pragma unroll
    for (uint32_t jj = 0; jj < 32; jj++) {
        if (jj < rows) {
            const uint32_t sh = (uint32_t)((uintptr_t)(scan + (uint64_t)(r0 + jj) * stride + 1) & 3) * 8;
            uint32_t hi = simt::shfl_down(v[jj], 1);
            if (ln == 31) hi = hi31[jj];
            v[jj] = simt::funnel_r(v[jj], hi, sh);
        }
    }
}

// MODE 0: None / Sub rows; 1: general without Paeth rows; 2: general
template <int MODE>
DBG_DEV void unf4_rows(UnfilterSmem *sm, const uint8_t *scan, uint32_t w, uint32_t h, uint32_t *out32, uint32_t band, uint64_t *prog,
                       uint32_t ft, bool needs_up)
{
    const uint32_t ln = (uint32_t)simt::lane();
    const uint64_t stride = (uint64_t)w * 4 + 1;
    const uint32_t r0 = band * BAND_ROWS;
    const uint32_t rows = h - r0 < BAND_ROWS ? h - r0 : BAND_ROWS;
    const bool row_ok = ln < rows;
    const uint32_t nblk = (w + 31) / 32, ntiles = nblk + 1;
    const uint32_t m_sub = ft == 1 ? ~0u : 0u, m_up = ft == 2 ? ~0u : 0u, m_avg = ft == 3 ? ~0u : 0u, m_paeth = ft == 4 ? ~0u : 0u;
    const uint32_t keep = ft <= 4 ? ~0u : 0u;  // :528-540 unknown filter -> 0 in the no-assert build
    const uint32_t w_eff = row_ok ? w : 0;
    uint32_t *my = sm->ring[1 + ln];
    uint32_t prev_out = 0, prev_b = 0;
    // Lanes j > 0 begin j pixels left of the image: there the ring (the half block 0 does not use), hence every input and
    // every result, is zero, which is what the first pixel's `a` and `c` have to be.
    for (uint32_t jj = 0; jj < 33; jj++) sm->ring[jj][32 + ln] = 0;
    uint32_t v[32], up = 0;
    unf4_load_block(scan, stride, r0, rows, ln, w, v);
    if (MODE != 0 && needs_up) {
        unf4_wait_above(prog, band, 2 < ntiles ? 2 : ntiles);
        if (ln < w) up = simt::ldcg_u32(out32 + (uint64_t)(r0 - 1) * w + ln);
    }
    for (uint32_t k = 0; k < ntiles; k++) {
        if (k < nblk) {
            const uint32_t col = (32 * k + ln) & 63;
#pragma unroll
            for (uint32_t jj = 0; jj < 32; jj++)
                if (jj < rows) sm->ring[1 + jj][col] = v[jj];
            if (MODE != 0) sm->ring[0][col] = up;
        }
        simt::syncwarp();
#pragma unroll 4
        for (uint32_t i = 0; i < 32; i++) {
            const uint32_t x = 32 * k + i - ln;  // "negative" left of the image
            const uint32_t cx = x & 63;
            uint32_t b = 0;
            if (MODE != 0) {
                b = simt::shfl_up(prev_out, 1);
                if (ln == 0) b = sm->ring[0][cx];
            }
            const uint32_t cur = my[cx];
            const uint32_t a = prev_out;
            uint32_t pred = a & m_sub;
            if (MODE != 0) {
                pred |= (b & m_up) | (swar_havg4(a, b) & m_avg);
                if (MODE == 2) pred |= paeth4_swar(a, b, prev_b) & m_paeth;
            }
            const uint32_t o = swar_add4(cur, pred) & keep;
            if (x < w_eff) my[cx] = o;
            prev_out = o;  // past the end of the row it is read by no one
            prev_b = b;
        }
        simt::syncwarp();
        // the next block's loads are in flight while the finished block is written out and published
        if (k + 1 < nblk) unf4_load_block(scan, stride, r0, rows, 32 * (k + 1) + ln, w, v);
        if (k >= 1) {
            const uint32_t x_out = 32 * (k - 1) + ln, oc = x_out & 63;
            if (x_out < w) {
#pragma unroll 8
                for (uint32_t jj = 0; jj < rows; jj++) out32[(uint64_t)(r0 + jj) * w + x_out] = sm->ring[1 + jj][oc];
            }
        }
        unf4_publish(prog, band, k + 1);
        if (MODE != 0 && needs_up && k + 1 < nblk) {
            unf4_wait_above(prog, band, k + 3 < ntiles ? k + 3 : ntiles);
            const uint32_t xn = 32 * (k + 1) + ln;
            up = xn < w ? simt::ldcg_u32(out32 + (uint64_t)(r0 - 1) * w + xn) : 0;
        }
    }
}

// None / Up rows only: lane = pixel column
DBG_DEV void unf4_columns(const uint8_t *scan, uint32_t w, uint32_t h, uint32_t *out32, uint32_t band, uint64_t *prog, uint32_t ft,
                          bool needs_up)
{
    const uint32_t ln = (uint32_t)simt::lane();
    const uint64_t stride = (uint64_t)w * 4 + 1;
    const uint32_t r0 = band * BAND_ROWS;
    const uint32_t rows = h - r0 < BAND_ROWS ? h - r0 : BAND_ROWS;
    const uint32_t nblk = (w + 31) / 32, ntiles = nblk + 1;
    const uint32_t up_rows = simt::ballot(ft == 2);
    uint32_t v[32];
    for (uint32_t k = 0; k < nblk; k++) {
        const uint32_t x = 32 * k + ln;
        unf4_load_block(scan, stride, r0, rows, x, w, v);
        uint32_t acc = 0;
        if (needs_up) {
            unf4_wait_above(prog, band, k + 2 < ntiles ? k + 2 : ntiles);
            if (x < w) acc = simt::ldcg_u32(out32 + (uint64_t)(r0 - 1) * w + x);
        }
#pragma unroll
        for (uint32_t jj = 0; jj < 32; jj++) {
            if (jj < rows) {
                acc = (up_rows >> jj) & 1 ? swar_add4(v[jj], acc) : v[jj];
                if (x < w) out32[(uint64_t)(r0 + jj) * w + x] = acc;
            }
        }
        unf4_publish(prog, band, k + 2 < ntiles ? k + 2 : ntiles);
    }
    if (nblk == 0) unf4_publish(prog, band, ntiles);
}

DBG_DEV void png_unfilter_band4(UnfilterSmem *sm, const uint8_t *scan, uint32_t w, uint32_t h, uint8_t *out, uint32_t band,
                                uint64_t *prog)
{
    const uint32_t ln = (uint32_t)simt::lane();
    const uint64_t stride = (uint64_t)w * 4 + 1;
    const uint32_t r0 = band * BAND_ROWS;
    const uint32_t r = r0 + ln;
    const uint32_t ft = r < h ? scan[(uint64_t)r * stride] : 0;
    const uint32_t ntiles = (w + 31) / 32 + 1;
    // This band publishes in the slot band - BAND_SLOTS used: that band must have finished (a band whose first row is None or
    // Sub does not wait for the band above, so "the band BAND_SLOTS - 1 above is done" would not imply it, and a late
    // publication of the old band would take the slot backwards under this band's readers). Its only reader, one band further
    // down, then finds a larger value than it waits for, which is right: everything it wants is there.
    if (prog && band >= BAND_SLOTS) {
        const uint64_t done = ((uint64_t)(band - BAND_SLOTS + 1) << 32) | ntiles;
        const uint64_t *slot = prog + (band & (BAND_SLOTS - 1));
        while (simt::ld_acquire_u64(slot) < done) simt::backoff();
        simt::syncwarp();
    }
    const bool has_sub = simt::any(ft == 1), has_up = simt::any(ft == 2), has_avg = simt::any(ft == 3), has_paeth = simt::any(ft == 4),
               has_bad = simt::any(ft > 4);
    const uint32_t ft0 = simt::shfl(ft, 0);
    const bool needs_up = r0 > 0 && ft0 >= 2 && ft0 <= 4;  // only the band's first row looks at the band above
    uint32_t *out32 = (uint32_t *)out;
    if (!has_avg && !has_paeth && !has_bad && !has_up) unf4_rows<0>(sm, scan, w, h, out32, band, prog, ft, false);
    else if (!has_avg && !has_paeth && !has_bad && !has_sub) unf4_columns(scan, w, h, out32, band, prog, ft, needs_up);
    else if (!has_paeth) unf4_rows<1>(sm, scan, w, h, out32, band, prog, ft, needs_up);
    else unf4_rows<2>(sm, scan, w, h, out32, band, prog, ft, needs_up);
}

// Whole image by one warp (bands in order, no hand-off needed).
template <int BPP>
DBG_DEV void png_unfilter_warp(UnfilterSmem *sm, uint8_t *scan, uint32_t w, uint32_t h, uint8_t *out, const uint8_t *plte,
                               uint32_t plte_size)
{
    for (uint32_t band = 0; band * BAND_ROWS < h; band++) {
        if (BPP == 4 && w <= UNF4_MAX_W) png_unfilter_band4(sm, scan, w, h, out, band, nullptr);
        else png_unfilter_band<BPP>(sm, scan, w, h, out, plte, plte_size, band, nullptr);
        simt::syncwarp();
    }
}

}  // namespace dbg
