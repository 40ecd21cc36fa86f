// tests/simt_emu/emu.cpp -- TEST SCAFFOLDING, not product code.
//
// A single-threaded 32-lane SIMT emulator (ucontext coroutines) that compiles
// the *device* kernel bodies from debigulator_b200/csrc/*_core.h for the host,
// so their logic can be checked against the oracle on a CPU-only box before
// GPU minutes are spent. Warp collectives are rendezvous points: a lane runs
// until its next collective, then the next lane runs, so a missing
// __syncwarp() between a store and another lane's load shows up as a wrong
// answer in at least one of the two lane orders (`reverse`).
//
// Nothing here is linked into libdebigulator_b200.so and no product entry
// point can reach it; the product fails loudly without a GPU.
#define DBG_SIMT_EMU 1
#include <stdint.h>
#include <stdlib.h>
#include <vector>
#include <string.h>
#include <ucontext.h>

#include "../../debigulator_b200/csrc/simt.h"

namespace simt {
int g_lane = 0;
uint32_t g_slot[32];
static ucontext_t g_ctx[32], g_main;
static bool g_done[32];
static int g_order[32], g_rank[32];

static int next_alive(int cur)
{
    int r = g_rank[cur];
    for (int k = 1; k <= 32; k++) {
        int cand = g_order[(r + k) & 31];
        if (!g_done[cand]) return cand;
    }
    return -1;
}
void emu_barrier()
{
    int cur = g_lane;
    int nxt = next_alive(cur);
    if (nxt < 0 || nxt == cur) return;
    g_lane = nxt;
    swapcontext(&g_ctx[cur], &g_ctx[nxt]);
    g_lane = cur;
}
static void (*g_body)(void *);
static void *g_arg;
static void trampoline()
{
    g_body(g_arg);
    int cur = g_lane;
    g_done[cur] = true;
    int nxt = next_alive(cur);
    if (nxt < 0) {
        setcontext(&g_main);
    } else {
        g_lane = nxt;
        setcontext(&g_ctx[nxt]);
    }
}
static void run_warp(void (*body)(void *), void *arg, int reverse)
{
    static char *stacks = nullptr;
    const size_t STK = 512 * 1024;
    if (!stacks) stacks = (char *)malloc(32 * STK);
    g_body = body;
    g_arg = arg;
    for (int i = 0; i < 32; i++) {
        g_order[i] = reverse ? 31 - i : i;
        g_rank[g_order[i]] = i;
        g_done[i] = false;
    }
    for (int i = 0; i < 32; i++) {
        getcontext(&g_ctx[i]);
        g_ctx[i].uc_stack.ss_sp = stacks + i * STK;
        g_ctx[i].uc_stack.ss_size = STK;
        g_ctx[i].uc_link = nullptr;
        makecontext(&g_ctx[i], trampoline, 0);
    }
    g_lane = g_order[0];
    swapcontext(&g_main, &g_ctx[g_lane]);
}
}  // namespace simt

#include "../../debigulator_b200/csrc/inflate_core.h"

struct InflateArgs {
    uint32_t *scratch;  // token scratch of the lane-parallel rounds (nullptr: plain symbol walk)
    dbg::InflateSmem *sm;
    const uint8_t *in;
    uint64_t in_size;
    uint8_t *out;
    uint64_t cap;
    uint64_t final_size[32];
    uint32_t status[32];
};
static void inflate_body(void *p)
{
    InflateArgs *a = (InflateArgs *)p;
    int l = simt::lane();
    a->status[l] = dbg::inflate_warp(a->sm, a->in, a->in_size, a->out, a->cap, &a->final_size[l], a->scratch);
}

// Returns the status (or 0x1000 | lane if the lanes disagree, which would be a
// uniformity bug in the kernel body).
extern "C" uint32_t emu_inflate(const uint8_t *in, uint64_t in_size, uint8_t *out, uint64_t cap, uint64_t *final_size,
                                int misalign, int reverse)
{
    // stage the input at the requested misalignment inside a 16-byte aligned,
    // padded arena whose surroundings are poisoned (0xA5) up to the 16 B rule.
    size_t arena_sz = (size_t)in_size + 64 + 32;
    uint8_t *arena = (uint8_t *)aligned_alloc(16, (arena_sz + 15) & ~(size_t)15);
    memset(arena, 0xA5, (arena_sz + 15) & ~(size_t)15);
    uint8_t *src = arena + 16 + (misalign & 15);
    memcpy(src, in, in_size);
    memset(src + in_size, 0, 16);  // what the host API puts behind every item (and the reference binding behind its input)
    dbg::InflateSmem *sm = (dbg::InflateSmem *)aligned_alloc(16, sizeof(dbg::InflateSmem));
    memset(sm, 0xCD, sizeof(*sm));
    InflateArgs a;
    a.scratch = (misalign & 16) ? nullptr : (uint32_t *)malloc(dbg::LB_ROUND_TOKENS * 4);  // bit 4 of `misalign`: rounds off
    a.sm = sm;
    a.in = src;
    a.in_size = in_size;
    a.out = out;
    a.cap = cap;
    simt::run_warp(inflate_body, &a, reverse);
    uint32_t st = a.status[0];
    for (int i = 1; i < 32; i++)
        if (a.status[i] != st || a.final_size[i] != a.final_size[0]) st = 0x1000 | i;
    *final_size = a.final_size[0];
    free(a.scratch);
    free(sm);
    free(arena);
    return st;
}

// ------------------------------------------------- lane-serial fixed-block path ----
#include "../../debigulator_b200/csrc/bsplit_core.h"
#include "../../debigulator_b200/csrc/fx_core.h"

struct FxHeadArgs {
    const dbg::FxLuts *luts;
    const uint8_t *in;
    uint64_t in_size;
    uint32_t chunk, chunk_bytes;
    uint32_t *hyp, *surv_start;
    uint32_t nsurv[32];
};
static void fx_head_body(void *p)
{
    FxHeadArgs *a = (FxHeadArgs *)p;
    a->nsurv[simt::lane()] = dbg::fx_head_warp(a->luts, a->in, a->in_size, a->chunk, a->chunk_bytes, a->hyp, a->surv_start);
}
struct FxExpandArgs {
    const uint32_t *tok;
    uint32_t ntok;
    uint16_t *cells;
    uint64_t abs_base;
    uint32_t st[32], ob[32];
};
static void fx_expand_body(void *p)
{
    FxExpandArgs *a = (FxExpandArgs *)p;
    const int l = simt::lane();
    a->st[l] = dbg::expand_tokens_warp(a->tok, a->ntok, a->cells, a->abs_base, &a->ob[l]);
}

// The whole lane-serial pipeline of fx_kernels.cuh (head, sizes, chain, tokens, expansion per group, resolve)
// run through the emulator. Returns the status; 0x2000 = not a single fixed block, 0x3000 = the passes
// disagree (cannot happen), 0x4000 = the chain needed a survivor that has no work item. *max_surv = the largest
// number of survivors any chunk had, *n_chunks = chunks on the real chain.
extern "C" uint32_t emu_fx_inflate(const uint8_t *in, uint64_t in_size, uint8_t *out, uint64_t cap, uint64_t *final_size,
                                   int misalign, int reverse, uint32_t chunk_bytes, uint32_t group_chunks, uint32_t *max_surv,
                                   uint32_t *n_chunks)
{
    size_t arena_sz = ((size_t)in_size + 64 + 32 + 15) & ~(size_t)15;
    uint8_t *arena = (uint8_t *)aligned_alloc(16, arena_sz);
    memset(arena, 0xA5, arena_sz);
    uint8_t *src = arena + 16 + (misalign & 15);
    memcpy(src, in, in_size);
    memset(src + in_size, 0, 16);  // what the host API puts behind every item (and the reference binding behind its input)
    *final_size = 0;
    *max_surv = 0;
    *n_chunks = 0;
    if (!dbg::is_single_fixed_block(src)) { free(arena); return 0x2000; }
    dbg::FxLuts luts;
    dbg::fx_build_luts(&luts, 0, 1);
    const uint32_t nch = (uint32_t)((in_size + chunk_bytes - 1) / chunk_bytes);
    uint32_t *hyp = (uint32_t *)calloc((size_t)(nch + 1) * 32, 4), *sstart = (uint32_t *)calloc((size_t)nch * 32, 4);
    uint32_t *nsurv = (uint32_t *)calloc(nch, 4);
    dbg::FxRec *rec = (dbg::FxRec *)calloc((size_t)nch * 32, sizeof(dbg::FxRec));
    uint32_t status = 0;
    FxHeadArgs h;
    h.luts = &luts; h.in = src; h.in_size = in_size; h.chunk_bytes = chunk_bytes;
    for (uint32_t c = 0; c < nch; c++) {
        h.chunk = c; h.hyp = hyp + (size_t)c * 32; h.surv_start = sstart + (size_t)c * 32;
        simt::run_warp(fx_head_body, &h, reverse);
        for (int i = 1; i < 32; i++) if (h.nsurv[i] != h.nsurv[0]) status = 0x1000 | i;
        nsurv[c] = h.nsurv[0];
        if (nsurv[c] > *max_surv) *max_surv = nsurv[c];
    }
    for (uint32_t c = 0; c < nch && !status; c++)
        for (uint32_t sv = 0; sv < nsurv[c]; sv++)
            rec[(size_t)c * 32 + sv] = dbg::fx_sizes_lane(&luts, src, in_size, c, chunk_bytes, sstart[(size_t)c * 32 + sv], hyp + (size_t)(c + 1) * 32);
    // chain
    uint32_t *csv = (uint32_t *)calloc(nch, 4), *ooff = (uint32_t *)calloc(nch + 1, 4), *toff = (uint32_t *)calloc(nch + 1, 4);
    uint64_t pos = 0, tok = 0;
    uint32_t e = 0, used = 0, end_flag = dbg::CH_RUN;
    bool ended = false;
    for (uint32_t c = 0; c < nch && !status && !ended; c++) {
        if (e >= nsurv[c]) { status = 0x4000; break; }
        const dbg::FxRec r = rec[(size_t)c * 32 + e];
        csv[c] = e; ooff[c] = (uint32_t)pos; toff[c] = (uint32_t)tok;
        pos += r.out_bytes; tok += r.ntok; used++;
        if ((r.link & 0xff) != dbg::CH_RUN) { ended = true; end_flag = r.link & 0xff; }
        e = r.link >> 8;
    }
    if (!status && !ended) status = dbg::ST_TRUNCATED;
    if (!status && end_flag >= dbg::CH_ERR) status = end_flag - dbg::CH_ERR;
    if (!status && pos > cap) status = dbg::ST_OUT_OVERFLOW;
    *n_chunks = used;
    if (!status) {
        uint32_t *tokens = (uint32_t *)malloc((tok + 16) * 4);
        for (uint32_t c = 0; c < used && !status; c++) {
            const dbg::FxRec r = rec[(size_t)c * 32 + csv[c]];
            uint32_t ob = 0, nt = 0;
            dbg::fx_tokens_lane(&luts, src, in_size, c, chunk_bytes, sstart[(size_t)c * 32 + csv[c]], r.exit_rel, tokens + toff[c], &ob, &nt);
            if (ob != r.out_bytes || nt != r.ntok) status = 0x3000;
        }
        uint16_t *cells = (uint16_t *)malloc((pos + 16) * 2);
        ooff[used] = (uint32_t)pos; toff[used] = (uint32_t)tok;
        for (uint32_t c = 0; c < used && !status; c += group_chunks) {
            const uint32_t ce = c + group_chunks < used ? c + group_chunks : used;
            FxExpandArgs x;
            x.tok = tokens + toff[c]; x.ntok = toff[ce] - toff[c]; x.cells = cells + ooff[c]; x.abs_base = ooff[c];
            simt::run_warp(fx_expand_body, &x, reverse);
            if (x.st[0]) status = x.st[0];
            else if (x.ob[0] != ooff[ce] - ooff[c]) status = 0x3000;
            // resolve this group (markers point at most 32 KiB before the group)
            for (uint32_t i = ooff[c]; i < ooff[ce] && !status; i++) {
                const uint32_t v = cells[i];
                out[i] = v < 256 ? (uint8_t)v : out[ooff[c] + (int64_t)v - 33024];
            }
        }
        free(cells); free(tokens);
        if (!status) *final_size = pos;
    }
    free(hyp); free(sstart); free(nsurv); free(rec); free(csv); free(ooff); free(toff); free(arena);
    return status;
}

// ------------------------------------------------------------ block split ----

struct BsArgs {
    dbg::InflateSmem *sm;
    dbg::SearchSmem *q;
    const uint16_t *kraft;
    const uint8_t *in;
    uint64_t in_size;
    int mode;  // 0 search, 1 count, 2 decode, 3 expand tokens, 4 cut the token run into pieces
    uint32_t piece_tok, npieces[32];
    uint64_t out0, *p_off;
    uint32_t *p_len;
    uint32_t *tok;
    uint32_t tok_cap, ntok, exp_bytes[32], exp_st[32];
    int lanes;
    uint64_t lo, hi, start, stop;
    uint16_t *cells;
    uint32_t cell_cap;
    uint64_t abs_base;
    uint64_t found[32];
    dbg::ChunkResult res[32];
};
static void bs_body(void *p)
{
    BsArgs *a = (BsArgs *)p;
    int l = simt::lane();
    if (a->mode == 0) a->found[l] = dbg::find_block_start(a->q, a->kraft, a->in, a->in_size, a->lo, a->hi);
    else if (a->mode == 1 && a->tok)
        a->res[l] = dbg::decode_block_chunk<dbg::SINK_TOKENS>(a->sm, a->in, a->in_size, a->start, a->stop, nullptr, 0, 0, a->tok, a->tok_cap, a->lanes != 0);
    else if (a->mode == 1) a->res[l] = dbg::decode_block_chunk<dbg::SINK_COUNT>(a->sm, a->in, a->in_size, a->start, a->stop, nullptr, 0, 0);
    else if (a->mode == 3) a->exp_st[l] = dbg::expand_tokens_warp(a->tok, a->ntok, a->cells, a->abs_base, &a->exp_bytes[l]);
    else if (a->mode == 4) a->npieces[l] = dbg::cut_token_pieces(a->tok, a->ntok, a->piece_tok, a->out0, a->p_off, a->p_len);
    else a->res[l] = dbg::decode_block_chunk<dbg::SINK_U16>(a->sm, a->in, a->in_size, a->start, a->stop, a->cells, a->cell_cap, a->abs_base);
}

// The block-split pipeline (search, count, chain, 16-bit decode, resolve) of bsplit_kernels.cuh run
// region by region through the emulator. Returns the status; 0x4000 = the chain did not close (the
// product would hand the stream back to the warp-per-stream kernel). *n_chunks = hinted regions used.
// max_pieces > 1: a chunk's tokens are expanded as up to that many pieces, each a marker domain of its own (cut_token_pieces)
static uint32_t bsplit_inflate_impl(const uint8_t *in, uint64_t in_size, uint8_t *out, uint64_t cap, uint64_t *final_size,
                                    int misalign, int reverse, uint32_t region_bytes, uint32_t *n_chunks, uint32_t tok_per_byte,
                                    int lanes, uint32_t max_pieces)
{
    size_t arena_sz = ((size_t)in_size + 64 + 32 + 15) & ~(size_t)15;
    uint8_t *arena = (uint8_t *)aligned_alloc(16, arena_sz);
    memset(arena, 0xA5, arena_sz);
    uint8_t *src = arena + 16 + (misalign & 15);
    memcpy(src, in, in_size);
    memset(src + in_size, 0, 16);  // what the host API puts behind every item (and the reference binding behind its input)
    dbg::InflateSmem *sm = (dbg::InflateSmem *)aligned_alloc(16, sizeof(dbg::InflateSmem));
    dbg::SearchSmem q;
    static uint16_t kraft[4096];
    dbg::build_kraft12(kraft, 0, 1);
    *final_size = 0;
    *n_chunks = 0;
    const uint32_t nreg = (uint32_t)((in_size + region_bytes - 1) / region_bytes);
    uint64_t *cand = (uint64_t *)calloc(nreg, 8), *exitb = (uint64_t *)calloc(nreg, 8), *ooff = (uint64_t *)calloc(nreg, 8);
    uint32_t *olen = (uint32_t *)calloc(nreg, 4), *flag = (uint32_t *)calloc(nreg, 4), *ntok = (uint32_t *)calloc(nreg, 4);
    uint32_t *tokens = tok_per_byte ? (uint32_t *)malloc(((size_t)tok_per_byte * in_size + 16) * 4) : nullptr;
    BsArgs a;
    a.sm = sm; a.q = &q; a.kraft = kraft; a.in = src; a.in_size = in_size; a.cells = nullptr; a.tok = nullptr; a.tok_cap = 0;
    a.lanes = lanes;
    uint32_t status = 0;
    for (uint32_t c = 0; c < nreg; c++) {
        cand[c] = 0;
        if (!c) continue;
        a.mode = 0; a.lo = (uint64_t)c * region_bytes * 8; a.hi = (uint64_t)(c + 1) * region_bytes * 8;
        simt::run_warp(bs_body, &a, reverse);
        for (int i = 1; i < 32; i++) if (a.found[i] != a.found[0]) status = 0x1000 | i;
        cand[c] = a.found[0];
    }
    auto next_hint = [&](uint32_t c) { for (uint32_t u = c + 1; u < nreg; u++) if (cand[u] != dbg::BS_NONE) return cand[u]; return dbg::BS_NONE; };
    for (uint32_t c = 0; c < nreg && !status; c++) {
        if (cand[c] == dbg::BS_NONE) continue;
        a.mode = 1; a.start = cand[c]; a.stop = next_hint(c);
        if (tokens) {
            a.tok = tokens + (size_t)tok_per_byte * (cand[c] >> 3);
            a.tok_cap = (uint32_t)(tok_per_byte * ((a.stop == dbg::BS_NONE ? in_size : a.stop >> 3) - (cand[c] >> 3)));
        }
        simt::run_warp(bs_body, &a, reverse);
        exitb[c] = a.res[0].exit_bits; olen[c] = a.res[0].out_bytes; flag[c] = a.res[0].flag; ntok[c] = a.res[0].ntok;
    }
    uint64_t pos = 0, expected = 0;
    bool ended = false, fail = false;
    for (uint32_t c = 0; c < nreg && !status; c++) {
        ooff[c] = pos;
        if (cand[c] == dbg::BS_NONE || ended || fail) { flag[c] = dbg::CH_IDLE; continue; }
        if (cand[c] < expected) { flag[c] = dbg::CH_IDLE; continue; }  // a hint the previous chunk stepped over: dropped
        if (cand[c] != expected) { fail = true; flag[c] = dbg::CH_IDLE; continue; }
        (*n_chunks)++;
        if (flag[c] >= dbg::CH_ERR) { status = pos + olen[c] > cap ? (uint32_t)dbg::ST_OUT_OVERFLOW : flag[c] - dbg::CH_ERR; ended = true; flag[c] = dbg::CH_IDLE; continue; }
        pos += olen[c];
        if (pos > cap) { status = dbg::ST_OUT_OVERFLOW; ended = true; }
        else if (flag[c] != dbg::CH_RUN) ended = true;
        else expected = exitb[c];
    }
    if (!status && (fail || !ended)) status = 0x4000;
    if (!status) {
        uint16_t *cells = (uint16_t *)malloc((pos + 16) * 2);
        for (uint32_t c = 0; c < nreg && !status; c++) {
            if (flag[c] == dbg::CH_IDLE) continue;
            a.mode = 2; a.start = cand[c]; a.stop = flag[c] == dbg::CH_RUN ? exitb[c] : dbg::BS_NONE;
            a.cells = cells + ooff[c]; a.cell_cap = olen[c]; a.abs_base = ooff[c];
            uint64_t nh = next_hint(c);
            uint32_t cap_c = tokens ? (uint32_t)(tok_per_byte * ((nh == dbg::BS_NONE ? in_size : nh >> 3) - (cand[c] >> 3))) : 0;
            if (tokens && ntok[c] <= cap_c && max_pieces > 1 && ntok[c]) {
                // the product's piece scheme: cut, expand every piece on its own, resolve the pieces in order
                uint32_t *ctok = tokens + (size_t)tok_per_byte * (cand[c] >> 3);
                uint32_t pt = (ntok[c] + max_pieces - 1) / max_pieces;
                pt = (pt + 127) & ~127u;
                std::vector<uint64_t> poff(max_pieces + 1);
                std::vector<uint32_t> plen(max_pieces + 1);
                a.mode = 4; a.tok = ctok; a.ntok = ntok[c]; a.piece_tok = pt; a.out0 = ooff[c]; a.p_off = poff.data(); a.p_len = plen.data();
                simt::run_warp(bs_body, &a, reverse);
                const uint32_t np = a.npieces[0];
                if (np == 0 || np > max_pieces) { status = 0x3001; continue; }
                uint64_t sum = 0;
                for (uint32_t j = 0; j < np && !status; j++) {
                    if (poff[j] != ooff[c] + sum) status = 0x3002;
                    sum += plen[j];
                    a.mode = 3; a.tok = ctok + (size_t)j * pt; a.ntok = j + 1 < np ? pt : ntok[c] - j * pt;
                    a.cells = cells + poff[j]; a.abs_base = poff[j];
                    simt::run_warp(bs_body, &a, reverse);
                    if (a.exp_st[0]) status = a.exp_st[0];
                    else if (a.exp_bytes[0] != plen[j]) status = 0x3000;
                    for (uint32_t i = 0; i < plen[j] && !status; i++) {  // resolve this piece (its markers point before it)
                        uint32_t v = cells[poff[j] + i];
                        out[poff[j] + i] = v < 256 ? (uint8_t)v : out[poff[j] + (int64_t)v - 33024];
                    }
                }
                if (!status && sum != olen[c]) status = 0x3003;
                flag[c] = dbg::CH_IDLE;  // resolved already
                (*n_chunks) += 0x10000;
                continue;
            }
            if (tokens && ntok[c] <= cap_c) {
                a.mode = 3; a.tok = tokens + (size_t)tok_per_byte * (cand[c] >> 3); a.ntok = ntok[c];
                simt::run_warp(bs_body, &a, reverse);
                if (a.exp_st[0]) status = a.exp_st[0];
                else if (a.exp_bytes[0] != olen[c]) status = 0x3000;
                (*n_chunks) += 0x10000;  // high half: chunks expanded from tokens
            } else {
                simt::run_warp(bs_body, &a, reverse);
                if (a.res[0].flag >= dbg::CH_ERR) status = a.res[0].flag - dbg::CH_ERR;
                else if (a.res[0].out_bytes != olen[c] || a.res[0].flag != flag[c]) status = 0x3000;
            }
            if (max_pieces > 1 && !status) {  // pieces are resolved as they come, so everything before them must be bytes already
                for (uint32_t i = 0; i < olen[c]; i++) {
                    uint32_t v = cells[ooff[c] + i];
                    out[ooff[c] + i] = v < 256 ? (uint8_t)v : out[ooff[c] + (int64_t)v - 33024];
                }
                flag[c] = dbg::CH_IDLE;
            }
        }
        for (uint32_t c = 0; c < nreg && !status; c++) {
            if (flag[c] == dbg::CH_IDLE) continue;
            for (uint32_t i = 0; i < olen[c]; i++) {
                uint32_t v = cells[ooff[c] + i];
                out[ooff[c] + i] = v < 256 ? (uint8_t)v : out[ooff[c] + (int64_t)v - 33024];
            }
        }
        free(cells);
        if (!status) *final_size = pos;
    }
    free(cand); free(exitb); free(ooff); free(olen); free(flag); free(ntok); free(tokens); free(sm); free(arena);
    return status;
}

extern "C" uint32_t emu_bsplit_inflate(const uint8_t *in, uint64_t in_size, uint8_t *out, uint64_t cap, uint64_t *final_size,
                                       int misalign, int reverse, uint32_t region_bytes, uint32_t *n_chunks, uint32_t tok_per_byte,
                                       int lanes)
{
    return bsplit_inflate_impl(in, in_size, out, cap, final_size, misalign, reverse, region_bytes, n_chunks, tok_per_byte, lanes, 1);
}
extern "C" uint32_t emu_bsplit_inflate_pieces(const uint8_t *in, uint64_t in_size, uint8_t *out, uint64_t cap, uint64_t *final_size,
                                              int misalign, int reverse, uint32_t region_bytes, uint32_t *n_chunks,
                                              uint32_t tok_per_byte, int lanes, uint32_t max_pieces)
{
    return bsplit_inflate_impl(in, in_size, out, cap, final_size, misalign, reverse, region_bytes, n_chunks, tok_per_byte, lanes, max_pieces);
}

extern "C" void emu_lane_block_stats(uint32_t *tried, uint32_t *done, int reset)
{
    *tried = dbg::g_lb_tried;
    *done = dbg::g_lb_done + dbg::g_lb_partial;
    if (reset) dbg::g_lb_tried = dbg::g_lb_done = dbg::g_lb_partial = 0;
}

// ------------------------------------------------------------------- PNG -----
#include "../../debigulator_b200/csrc/png_core.h"

struct PngArgs {
    const uint8_t *file;
    uint64_t size;
    uint8_t *out;
    uint64_t rgba_size;
    dbg::CrcTables *tables;
    dbg::InflateSmem *ism;
    dbg::UnfilterSmem *usm;
    uint8_t *zbuf;
    uint64_t zcap;
    uint8_t *scan;
    uint32_t status[32];
    uint32_t crc_only;   // when set: just CRC `size` bytes of `file`
    uint32_t crc[32];
    dbg::ScanQueues *q;  // non-null: the walk defers large chunks (phase 0), the tasks run one by one (phase 1), then
    uint32_t phase;      // inflate + un-filter (phase 2), as png_scan_kernel / png_tasks_kernel / the later passes do
    dbg::ScanTask task;
    dbg::PngInfo info;
    uint64_t zs;
    const uint8_t *zp;
};
static void png_decode_rest(PngArgs *a, uint32_t &st)
{
    const dbg::PngInfo info = a->info;
    uint64_t est = (uint64_t)info.w * info.h * 4 + info.h + 1, ssize = 0;
    st = dbg::inflate_warp(a->ism, a->zp, a->zs, a->scan, est, &ssize);
    simt::syncwarp();  // a kernel boundary in the product: the last deferred match store of one lane is read by another below
    if (st == dbg::ST_OK) {
        uint64_t need = (uint64_t)info.h * ((uint64_t)info.w * info.bpp + 1);
        if (a->scan[0] > 4) st = dbg::ST_PNG_FILTER;
        else if (ssize < need) st = dbg::ST_PNG_SHORT;
        else if (info.bpp == 4) dbg::png_unfilter_warp<4>(a->usm, a->scan, info.w, info.h, a->out, nullptr, 0);
        else if (info.bpp == 3) dbg::png_unfilter_warp<3>(a->usm, a->scan, info.w, info.h, a->out, nullptr, 0);
        else dbg::png_unfilter_warp<1>(a->usm, a->scan, info.w, info.h, a->out, a->file + info.plte_off, info.plte_size);
    }
}
static void png_body(void *p)
{
    PngArgs *a = (PngArgs *)p;
    int l = simt::lane();
    dbg::crc_tables_init(a->tables, l, 32);
    simt::syncwarp();
    uint32_t lane_k = dbg::gf2_xpow_bytes(dbg::CRC_SLICE * (31 - l));
    if (a->crc_only) {
        a->crc[l] = dbg::crc32_warp(a->tables, lane_k, a->file, a->size);
        return;
    }
    uint32_t st = dbg::ST_OK;
    if (a->phase == 1) {
        dbg::scan_task_run(a->tables, lane_k, a->task, a->q->big);
        return;
    }
    if (a->phase == 0) {
        dbg::PngInfo info;
        info.w = info.h = info.bpp = 0;
        uint64_t zs = 0;
        const uint8_t *zp = a->zbuf;
        st = dbg::png_scan_warp(a->tables, lane_k, a->file, a->size, a->rgba_size, a->zbuf, a->zcap, &info, &zs, &zp, a->q, 0);
        simt::syncwarp();
        if (l == 0) {
            a->info = info;
            a->zs = zs;
            a->zp = zp;
        }
        simt::syncwarp();
    }
    if (st == dbg::ST_OK && (a->phase == 2 || !a->q)) png_decode_rest(a, st);
    a->status[l] = st;
}

static uint32_t png_decode_impl(const uint8_t *file, uint64_t size, uint8_t *out, uint64_t rgba_size, int misalign, int reverse,
                                dbg::ScanQueues *q)
{
    PngArgs a;
    memset(&a, 0, sizeof(a));
    const uint64_t arena = (size + 64 + 16 + 15) & ~(uint64_t)15;
    uint8_t *fcopy = (uint8_t *)aligned_alloc(16, arena);
    memset(fcopy, 0xA5, arena);
    memcpy(fcopy + (misalign & 15), file, size);
    a.file = fcopy + (misalign & 15);
    a.size = size;
    a.out = out;
    a.rgba_size = rgba_size;
    a.tables = (dbg::CrcTables *)aligned_alloc(16, sizeof(dbg::CrcTables));
    a.ism = (dbg::InflateSmem *)aligned_alloc(16, sizeof(dbg::InflateSmem));
    a.usm = (dbg::UnfilterSmem *)aligned_alloc(16, (sizeof(dbg::UnfilterSmem) + 15) & ~(size_t)15);
    a.zcap = (size + 16 + 15) & ~(uint64_t)15;
    a.zbuf = (uint8_t *)aligned_alloc(16, a.zcap + 16);
    memset(a.zbuf, 0x5A, a.zcap + 16);
    uint64_t scan_cap = (rgba_size + rgba_size / 4 + 64 + 15) & ~(uint64_t)15;
    a.scan = (uint8_t *)aligned_alloc(16, scan_cap);
    memset(a.scan, 0x77, scan_cap);
    a.q = q;
    simt::run_warp(png_body, &a, reverse);
    uint32_t st = a.status[0];
    for (int i = 1; i < 32; i++)
        if (a.status[i] != st) st = 0x1000 | i;
    if (q && st < 0x1000) {
        // png_tasks_kernel, then png_verify_kernel: the verdict of the walk is raised to 13 by a bad large chunk
        const uint32_t total = *q->ntasks < q->task_cap ? *q->ntasks : q->task_cap;
        a.phase = 1;
        for (uint32_t t = 0; t < total; t++) {
            a.task = q->tasks[reverse ? total - 1 - t : t];
            if (a.task.len) simt::run_warp(png_body, &a, reverse);
        }
        const uint32_t nbig = *q->nbig < q->big_cap ? *q->nbig : q->big_cap;
        for (uint32_t i = 0; i < nbig; i++)
            if (dbg::big_chunk_crc_bad(q->big[i]) && st < dbg::ST_PNG_CRC) st = dbg::ST_PNG_CRC;
        if (st == dbg::ST_OK) {
            a.phase = 2;
            simt::run_warp(png_body, &a, reverse);
            st = a.status[0];
            for (int i = 1; i < 32; i++)
                if (a.status[i] != st) st = 0x1000 | i;
        }
    }
    free(fcopy); free(a.tables); free(a.ism); free(a.usm); free(a.zbuf); free(a.scan);
    return st;
}

extern "C" uint32_t emu_png_decode(const uint8_t *file, uint64_t size, uint8_t *out, uint64_t rgba_size, int reverse)
{
    return png_decode_impl(file, size, out, rgba_size, 0, reverse, nullptr);
}

// The same with the walk's segment queues (png_task_cap / png_big_cap of a batch of this one file unless the caps are
// given), the file at `misalign` bytes past a 16-byte boundary. The tasks run in queue order, or in reverse order with
// the lanes. *ntasks / *nbig: what the walk enqueued.
extern "C" uint32_t emu_png_decode_queued(const uint8_t *file, uint64_t size, uint8_t *out, uint64_t rgba_size, int misalign,
                                          int reverse, uint32_t task_cap, uint32_t big_cap, uint32_t *ntasks, uint32_t *nbig)
{
    if (!task_cap) task_cap = (uint32_t)(4 * (size / dbg::SCAN_SEG) + 64);
    if (!big_cap) big_cap = (uint32_t)(size / dbg::SCAN_SEG + 16);
    std::vector<dbg::ScanTask> tasks(task_cap);
    std::vector<dbg::BigChunk> big(big_cap);
    uint32_t counters[2] = {0, 0};
    dbg::ScanQueues q{tasks.data(), &counters[0], task_cap, big.data(), &counters[1], big_cap};
    const uint32_t st = png_decode_impl(file, size, out, rgba_size, misalign, reverse, &q);
    *ntasks = counters[0];
    *nbig = counters[1];
    return st;
}

extern "C" uint32_t emu_crc32(const uint8_t *p, uint64_t n, int reverse)
{
    PngArgs a;
    memset(&a, 0, sizeof(a));
    a.file = p;
    a.size = n;
    a.crc_only = 1;
    a.tables = (dbg::CrcTables *)aligned_alloc(16, sizeof(dbg::CrcTables));
    simt::run_warp(png_body, &a, reverse);
    uint32_t c = a.crc[0];
    for (int i = 1; i < 32; i++)
        if (a.crc[i] != c) c = 0xDEADBEEF;
    free(a.tables);
    return c;
}

// paeth4_swar (png_core.h) against the scalar definition (decode_png.c:441-487) for every byte triple, four different
// triples per word so that the byte lanes are seen not to leak into each other. Returns the number of mismatches.
extern "C" uint64_t emu_paeth4_mismatches()
{
    auto paeth = [](int a, int b, int c) {
        int pa = b - c, pb = a - c, pc = a + b - 2 * c;
        pa = pa < 0 ? -pa : pa; pb = pb < 0 ? -pb : pb; pc = pc < 0 ? -pc : pc;
        return (pa <= pb && pa <= pc) ? a : (pb <= pc ? b : c);
    };
    uint64_t bad = 0;
    for (int a = 0; a < 256; a++)
        for (int b = 0; b < 256; b++)
            for (int c = 0; c < 256; c++) {
                const uint32_t A = (uint32_t)a | ((uint32_t)b << 8) | ((uint32_t)c << 16) | ((uint32_t)(255 - a) << 24);
                const uint32_t B = (uint32_t)b | ((uint32_t)c << 8) | ((uint32_t)a << 16) | ((uint32_t)b << 24);
                const uint32_t Cw = (uint32_t)c | ((uint32_t)a << 8) | ((uint32_t)b << 16) | ((uint32_t)(c ^ 0x55) << 24);
                const uint32_t want = (uint32_t)paeth(a, b, c) | ((uint32_t)paeth(b, c, a) << 8) | ((uint32_t)paeth(c, a, b) << 16) |
                                      ((uint32_t)paeth(255 - a, b, c ^ 0x55) << 24);
                if (dbg::paeth4_swar(A, B, Cw) != want) bad++;
            }
    return bad;
}
