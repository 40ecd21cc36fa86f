// png_kernels.cuh -- __global__ wrappers and launch helpers for the PNG path.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "png_core.h"

namespace dbg {

// Scratch carved out of one device allocation (dbg_ctx::d_png_scratch).
struct PngLayout {
    uint64_t *z_off, *z_size;          // per image: compacted deflate stream (offset into idat, size)
    uint64_t *s_off, *s_cap, *s_size;  // per image: filtered scanline buffer (offset into scan, capacity, inflated size)
    uint32_t *inf_status, *pre_status;
    PngInfo *info;
    uint32_t *band_base;  // n + 1: first un-filter work item (32-row band) of every image
    uint64_t *band_prog;  // BAND_SLOTS per image: band pipeline hand-off
    uint32_t *band_counter;  // [0] work-queue head, [1] number of fetches, [2] band levels (0: items in image order)
    ScanQueues queues;     // deferred CRC / copy segments of large chunks
    uint32_t *task_counter;
    uint8_t *idat;  // compacted IDAT payloads
    uint8_t *scan;  // inflated, still filtered scanlines
    uint64_t idat_bytes, scan_bytes;
};

struct PngBatch {
    const uint8_t *in_base;
    const uint64_t *in_off;
    const uint64_t *in_size;
    const uint64_t *rgba_size;
    uint32_t n;
    PngLayout lay;
};

__host__ __device__ static inline uint64_t png_align(uint64_t v, uint64_t a) { return (v + a - 1) / a * a; }

// est = w*h*4 + h + 1 <= rgba + rgba/4 + 1 (decode_png.c:965-968); 32 bytes of
// slack per image cover alignment and the word-granular reads of load_px<4>.
static inline uint64_t png_idat_bytes(uint64_t n, uint64_t total_in) { return png_align(total_in + 32 * n + 64, 256); }
static inline uint64_t png_scan_bytes(uint64_t n, uint64_t total_rgba)
{
    return png_align(total_rgba + total_rgba / 4 + 48 * n + 64, 256);
}
static inline uint64_t png_meta_bytes(uint64_t n)
{
    return png_align(n * (5 * 8 + 2 * 4 + sizeof(PngInfo) + 4 + 8 * BAND_SLOTS) + 256, 256);
}
// at most total_in / SCAN_SEG chunks exceed SCAN_SEG, each cut into ceil(len / SCAN_SEG) segments,
// CRC and copy counted separately
static inline uint64_t png_task_cap(uint64_t n, uint64_t total_in) { return 4 * (total_in / SCAN_SEG) + 64; }
static inline uint64_t png_big_cap(uint64_t n, uint64_t total_in) { return total_in / SCAN_SEG + 16; }
static inline uint64_t png_queue_bytes(uint64_t n, uint64_t total_in)
{
    return png_align(png_task_cap(n, total_in) * sizeof(ScanTask) + png_big_cap(n, total_in) * sizeof(BigChunk) + 256, 256);
}
static inline uint64_t png_scratch_bytes(uint64_t n, uint64_t total_in, uint64_t total_rgba)
{
    return png_meta_bytes(n) + png_queue_bytes(n, total_in) + png_idat_bytes(n, total_in) + png_scan_bytes(n, total_rgba);
}
static inline PngLayout png_layout(uint8_t *base, uint64_t n, uint64_t total_in, uint64_t total_rgba)
{
    PngLayout l;
    uint64_t *u = (uint64_t *)base;
    l.z_off = u;
    l.z_size = u + n;
    l.s_off = u + 2 * n;
    l.s_cap = u + 3 * n;
    l.s_size = u + 4 * n;
    l.info = (PngInfo *)(u + 5 * n);
    l.band_prog = (uint64_t *)(l.info + n);
    l.inf_status = (uint32_t *)(l.band_prog + n * BAND_SLOTS);
    l.pre_status = l.inf_status + n;
    l.band_base = l.pre_status + n;
    l.band_counter = l.band_base + n + 1;
    uint8_t *qb = base + png_meta_bytes(n);
    l.queues.tasks = (ScanTask *)(qb + 256);
    l.queues.task_cap = (uint32_t)png_task_cap(n, total_in);
    l.queues.big = (BigChunk *)(l.queues.tasks + l.queues.task_cap);
    l.queues.big_cap = (uint32_t)png_big_cap(n, total_in);
    l.queues.ntasks = (uint32_t *)qb;
    l.queues.nbig = l.queues.ntasks + 1;
    l.task_counter = l.queues.ntasks + 2;
    l.idat = qb + png_queue_bytes(n, total_in);
    l.idat_bytes = png_idat_bytes(n, total_in);
    l.scan = l.idat + l.idat_bytes;
    l.scan_bytes = png_scan_bytes(n, total_rgba);
    return l;
}

// Pass A (one CTA): per-image buffer sizes and their exclusive prefix sums. The
// scanline buffer is sized for any IHDR whose w*h*4 is the caller's rgba size:
// the walk accepts every such IHDR and the last one sets the inflate capacity
// (decode_png.c:965-968), so png_scan_kernel sets s_cap once the walk is done;
// w >= 1 bounds h by rgba/4.
constexpr int PLAN_THREADS = 1024;
__global__ void __launch_bounds__(PLAN_THREADS) png_plan_kernel(PngBatch b)
{
    __shared__ uint64_t sh_z[PLAN_THREADS], sh_s[PLAN_THREADS];
    __shared__ uint64_t carry_z, carry_s;
    const int t = threadIdx.x;
    if (t == 0) {
        carry_z = 0;
        carry_s = 0;
        *b.lay.queues.ntasks = 0;
        *b.lay.queues.nbig = 0;
        *b.lay.task_counter = 0;
    }
    __syncthreads();
    for (uint32_t base = 0; base < b.n; base += PLAN_THREADS) {
        uint32_t i = base + t;
        uint64_t zc = 0, sc = 0, est = 0;
        if (i < b.n) {
            zc = png_align(b.in_size[i] + 16, 16);
            const uint64_t rgba = b.rgba_size[i];
            if (rgba >= 4 && rgba < (1ull << 32)) {
                est = rgba + rgba / 4 + 1;
                sc = png_align(est + 16, 16);
            }
        }
        sh_z[t] = zc;
        sh_s[t] = sc;
        __syncthreads();
        for (int d = 1; d < PLAN_THREADS; d <<= 1) {
            uint64_t vz = t >= d ? sh_z[t - d] : 0, vs = t >= d ? sh_s[t - d] : 0;
            __syncthreads();
            sh_z[t] += vz;
            sh_s[t] += vs;
            __syncthreads();
        }
        if (i < b.n) {
            // The scratch was sized from the caller's totals (device API: total_in_bytes / total_rgba_bytes). An item that
            // would reach past it gets no room: a null stream address fails it in png_scan_kernel, a scanline buffer of
            // capacity 0 fails its inflate.
            const bool z_fits = carry_z + sh_z[t] <= b.lay.idat_bytes, s_fits = carry_s + sh_s[t] <= b.lay.scan_bytes;
            b.lay.z_off[i] = z_fits ? (uint64_t)(uintptr_t)(b.lay.idat + (carry_z + sh_z[t] - zc)) : 0ull;  // absolute address
            b.lay.s_off[i] = s_fits ? carry_s + sh_s[t] - sc : 0ull;
            b.lay.s_cap[i] = s_fits ? est : 0ull;  // room; png_scan_kernel narrows it to inflate's recipient_size
            b.lay.z_size[i] = 0;
            b.lay.s_size[i] = 0;
            b.lay.inf_status[i] = 0;
        }
        __syncthreads();
        if (t == PLAN_THREADS - 1) {
            carry_z += sh_z[t];
            carry_s += sh_s[t];
        }
        __syncthreads();
    }
}

// Pass B: one warp per image -- chunk walk, CRC-32, IDAT gather.
constexpr int SCAN_WARPS = 8;
__global__ void __launch_bounds__(SCAN_WARPS * 32) png_scan_kernel(PngBatch b)
{
    __shared__ CrcTables tables;
    crc_tables_init(&tables, threadIdx.x, blockDim.x);
    __syncthreads();
    const uint32_t ln = (uint32_t)simt::lane();
    const uint32_t lane_k = gf2_xpow_bytes(CRC_SLICE * (31 - ln));
    const uint32_t warps = gridDim.x * SCAN_WARPS;
    for (uint32_t i = blockIdx.x * SCAN_WARPS + (threadIdx.x >> 5); i < b.n; i += warps) {
        uint8_t *zdst = (uint8_t *)(uintptr_t)b.lay.z_off[i];
        uint64_t zcap = png_align(b.in_size[i] + 16, 16);
        uint64_t zs = 0;
        const uint8_t *zp = zdst;
        PngInfo info;
        info.w = info.h = info.bpp = 0;
        ScanQueues q = b.lay.queues;
        uint32_t st = ST_TOO_LARGE;  // no room in the scratch (under-reported totals, see png_plan_kernel)
        if (zdst)
            st = png_scan_warp(&tables, lane_k, b.in_base + b.in_off[i], b.in_size[i], b.rgba_size[i], zdst, zcap, &info, &zs, &zp,
                               &q, i);
        if (ln == 0) {
            b.lay.z_off[i] = (uint64_t)(uintptr_t)zp;
            b.lay.z_size[i] = zs;
            b.lay.pre_status[i] = st;
            b.lay.info[i] = info;
            // recipient_size from the last IHDR the walk accepted (decode_png.c:803-804, 965-968)
            if (st == ST_OK && b.lay.s_cap[i]) b.lay.s_cap[i] = (uint64_t)info.w * info.h * 4 + info.h + 1;
        }
        simt::syncwarp();
    }
}

// Pass B2: the deferred segments (persistent warps, queue filled by pass B).
__global__ void __launch_bounds__(SCAN_WARPS * 32) png_tasks_kernel(PngBatch b)
{
    __shared__ CrcTables tables;
    crc_tables_init(&tables, threadIdx.x, blockDim.x);
    __syncthreads();
    const uint32_t ln = (uint32_t)simt::lane();
    const uint32_t lane_k = gf2_xpow_bytes(CRC_SLICE * (31 - ln));
    uint32_t total = *b.lay.queues.ntasks;
    if (total > b.lay.queues.task_cap) total = b.lay.queues.task_cap;
    for (;;) {
        uint32_t t = 0;
        if (ln == 0) t = atomicAdd(b.lay.task_counter, 1u);
        t = simt::shfl(t, 0);
        if (t >= total) break;
        const ScanTask k = b.lay.queues.tasks[t];
        if (k.len == 0) continue;
        scan_task_run(&tables, lane_k, k, b.lay.queues.big);
        simt::syncwarp();
    }
}

// Pass B3: compare the recombined CRCs of the large chunks with the stored ones (decode_png.c:1341-1348).
__global__ void png_verify_kernel(PngBatch b)
{
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    uint32_t nbig = *b.lay.queues.nbig;
    if (nbig > b.lay.queues.big_cap) nbig = b.lay.queues.big_cap;
    if (i >= nbig) return;
    const BigChunk c = b.lay.queues.big[i];
    if (big_chunk_crc_bad(c)) atomicMax(&b.lay.pre_status[c.img], (uint32_t)ST_PNG_CRC);
}

// Pass C2 (one CTA): un-filter work items. An image that decoded so far gets one item per 32-row
// band, any other image a single item (which only reports its status).
__global__ void __launch_bounds__(PLAN_THREADS) png_bands_kernel(PngBatch b)
{
    __shared__ uint32_t sh[PLAN_THREADS];
    __shared__ uint32_t carry, max_nb;
    const int t = threadIdx.x;
    if (t == 0) {
        carry = 0;
        max_nb = 0;
        *b.lay.band_counter = 0;
    }
    __syncthreads();
    for (uint32_t base = 0; base < b.n; base += PLAN_THREADS) {
        uint32_t i = base + t, nb = 0;
        if (i < b.n) {
            bool ok = b.lay.pre_status[i] == ST_OK && b.lay.inf_status[i] == ST_OK;
            nb = ok ? (b.lay.info[i].h + BAND_ROWS - 1) / BAND_ROWS : 1;
            for (int k = 0; k < BAND_SLOTS; k += 8)  // reset this image's hand-off ring (8 words per step)
                for (int j = 0; j < 8; j++) b.lay.band_prog[(uint64_t)i * BAND_SLOTS + k + j] = 0;
        }
        sh[t] = nb;
        if (nb) atomicMax(&max_nb, nb);
        __syncthreads();
        for (int d = 1; d < PLAN_THREADS; d <<= 1) {
            uint32_t v = t >= d ? sh[t - d] : 0;
            __syncthreads();
            sh[t] += v;
            __syncthreads();
        }
        if (i < b.n) b.lay.band_base[i] = carry + sh[t] - nb;
        __syncthreads();
        if (t == PLAN_THREADS - 1) carry += sh[t];
        __syncthreads();
    }
    if (t == 0) {
        b.lay.band_base[b.n] = carry;
        // Order of the work items. Band-major -- band 0 of every image, then band 1 of every image, ... (fetch f = band f / n of
        // image f % n, skipped when the image is not that tall) -- keeps the resident warps busy: by the time a warp takes band
        // k of an image, band k-1 is well ahead. In image order the 32-row bands of one image start two tiles apart, so with
        // a few thousand warps resident most of them would sit waiting for the band above. When the heights differ so much that
        // most fetches would be skips, items go in image order.
        const uint64_t fetches = (uint64_t)b.n * max_nb;
        const bool by_band = fetches <= 8ull * carry + 4096 && fetches < (1ull << 31);
        b.lay.band_counter[1] = by_band ? (uint32_t)fetches : carry;
        b.lay.band_counter[2] = by_band ? max_nb : 0;
    }
}

// Pass D: scanline reconstruction into RGBA. Persistent warps take (image, band) items in order (see
// png_bands_kernel) from a global counter; the bands of one image form a pipeline (png_unfilter_band), so a single large image
// keeps hundreds of warps busy instead of one.
constexpr int UNF_WARPS = 4;
__global__ void __launch_bounds__(UNF_WARPS * 32, 6) png_unfilter_kernel(PngBatch b, uint8_t *out_base, const uint64_t *out_off,
                                                                     uint32_t *status)
{
    __shared__ UnfilterSmem sm_all[UNF_WARPS];
    UnfilterSmem *sm = &sm_all[threadIdx.x >> 5];
    const uint32_t ln = (uint32_t)simt::lane();
    const uint32_t total = b.lay.band_counter[1], levels = b.lay.band_counter[2];
    for (;;) {
        uint32_t t = 0;
        if (ln == 0) t = atomicAdd(b.lay.band_counter, 1u);
        t = simt::shfl(t, 0);
        if (t >= total) break;
        uint32_t i, band;
        if (levels) {  // band-major order
            band = t / b.n;
            i = t - band * b.n;
            if (band >= b.lay.band_base[i + 1] - b.lay.band_base[i]) continue;
        } else {  // image of work item t: last i with band_base[i] <= t
            uint32_t lo = 0, hi = b.n;
            while (hi - lo > 1) {
                uint32_t mid = (lo + hi) >> 1;
                if (b.lay.band_base[mid] <= t) lo = mid;
                else hi = mid;
            }
            i = lo;
            band = t - b.lay.band_base[i];
        }
        uint32_t st = b.lay.pre_status[i];
        if (st == ST_OK) st = b.lay.inf_status[i];
        if (st == ST_OK) {
            PngInfo info = b.lay.info[i];
            uint8_t *scan = b.lay.scan + b.lay.s_off[i];
            uint64_t need = (uint64_t)info.h * ((uint64_t)info.w * info.bpp + 1);
            // the first filter byte is read through L2: band 0 of a palette / RGB image rewrites nothing
            // at offset 0, but keep every band's verdict identical and cache-independent
            if (simt::ldcg_u8(scan) > 4) st = ST_PNG_FILTER;          // decode_png.c:847-858
            else if (b.lay.s_size[i] < need) st = ST_PNG_SHORT;       // Q13: the reference reads stale memory here
            else {
                uint8_t *out = out_base + out_off[i];
                const uint8_t *file = b.in_base + b.in_off[i];
                uint64_t *prog = b.lay.band_prog + (uint64_t)i * BAND_SLOTS;
                if (info.bpp == 4 && info.w <= UNF4_MAX_W) png_unfilter_band4(sm, scan, info.w, info.h, out, band, prog);
                else if (info.bpp == 4) png_unfilter_band<4>(sm, scan, info.w, info.h, out, nullptr, 0, band, prog);
                else if (info.bpp == 3) png_unfilter_band<3>(sm, scan, info.w, info.h, out, nullptr, 0, band, prog);
                else png_unfilter_band<1>(sm, scan, info.w, info.h, out, file + info.plte_off, info.plte_size, band, prog);
            }
        }
        if (ln == 0 && band == 0) status[i] = st;
        simt::syncwarp();
    }
}

// Opt-in integrity check for gzip members (SURVEY.md 8f-3; the reference reads the trailer but never
// checks it, decode_gz.c:281-297): CRC-32 of the decoded payload and ISIZE against the 8-byte trailer.
// One warp per member, same slicing / GF(2) recombination as the PNG chunk CRCs.
constexpr uint32_t ST_CHECKSUM = 16;
__global__ void __launch_bounds__(SCAN_WARPS * 32) gz_verify_kernel(const uint8_t *in_base, const uint64_t *in_off,
                                                                   const uint64_t *in_size, const uint8_t *out_base,
                                                                   const uint64_t *out_off, const uint64_t *out_size,
                                                                   uint32_t *status, uint32_t n)
{
    __shared__ CrcTables tables;
    crc_tables_init(&tables, threadIdx.x, blockDim.x);
    __syncthreads();
    const uint32_t ln = (uint32_t)simt::lane();
    const uint32_t lane_k = gf2_xpow_bytes(CRC_SLICE * (31 - ln));
    const uint32_t warps = gridDim.x * SCAN_WARPS;
    for (uint32_t i = blockIdx.x * SCAN_WARPS + (threadIdx.x >> 5); i < n; i += warps) {
        if (status[i] != ST_OK) continue;
        const uint8_t *t = in_base + in_off[i] + in_size[i] - 8;
        const uint32_t want_crc = (uint32_t)t[0] | ((uint32_t)t[1] << 8) | ((uint32_t)t[2] << 16) | ((uint32_t)t[3] << 24);
        const uint32_t want_size = (uint32_t)t[4] | ((uint32_t)t[5] << 8) | ((uint32_t)t[6] << 16) | ((uint32_t)t[7] << 24);
        const uint64_t len = out_size[i];
        uint32_t crc = len ? crc32_warp(&tables, lane_k, out_base + out_off[i], len) : 0u;
        if (ln == 0 && (crc != want_crc || (uint32_t)len != want_size)) status[i] = ST_CHECKSUM;
        simt::syncwarp();
    }
}

// Opt-in: Adler-32 of the inflated scanline stream against the zlib trailer (the reference drops those four
// bytes unread, decode_png.c:816). One warp per image; 2 KiB tiles, 64 bytes per lane, warp reductions.
__global__ void __launch_bounds__(SCAN_WARPS * 32) png_adler_kernel(PngBatch b)
{
    const uint32_t ln = (uint32_t)simt::lane();
    const uint32_t warps = gridDim.x * SCAN_WARPS;
    for (uint32_t i = blockIdx.x * SCAN_WARPS + (threadIdx.x >> 5); i < b.n; i += warps) {
        if (b.lay.pre_status[i] != ST_OK || b.lay.inf_status[i] != ST_OK) continue;
        const uint8_t *p = b.lay.scan + b.lay.s_off[i];
        const uint64_t n = b.lay.s_size[i];
        uint64_t s1 = 1, s2 = 0;
        for (uint64_t t0 = 0; t0 < n; t0 += 2048) {
            const uint32_t tl = (uint32_t)(n - t0 < 2048 ? n - t0 : 2048);
            uint32_t a = 0, w = 0;
            const uint32_t lo = ln * 64;
            for (uint32_t j = lo; j < lo + 64 && j < tl; j++) {
                uint32_t v = p[t0 + j];
                a += v;
                w += (tl - j) * v;
            }
            for (int d = 16; d; d >>= 1) {
                a += simt::shfl_xor(a, d);
                w += simt::shfl_xor(w, d);
            }
            s2 = (s2 + (uint64_t)tl * s1 + w) % 65521u;
            s1 = (s1 + a) % 65521u;
        }
        const uint8_t *z = (const uint8_t *)(uintptr_t)b.lay.z_off[i] + b.lay.z_size[i];
        const uint32_t want = ((uint32_t)z[0] << 24) | ((uint32_t)z[1] << 16) | ((uint32_t)z[2] << 8) | z[3];
        if (ln == 0 && want != (uint32_t)((s2 << 16) | s1)) b.lay.inf_status[i] = ST_CHECKSUM;
        simt::syncwarp();
    }
}

static inline void png_configure_kernels() {}

// returns 0 or a cudaError_t value
static inline int png_launch_scan(const PngBatch &b, int sm_count, cudaStream_t s)
{
    png_plan_kernel<<<1, PLAN_THREADS, 0, s>>>(b);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return (int)e;
    uint32_t ctas = (b.n + SCAN_WARPS - 1) / SCAN_WARPS;
    uint32_t cap = (uint32_t)sm_count * 8;
    png_scan_kernel<<<ctas < cap ? ctas : cap, SCAN_WARPS * 32, 0, s>>>(b);
    e = cudaGetLastError();
    if (e != cudaSuccess) return (int)e;
    png_tasks_kernel<<<(uint32_t)sm_count * 4, SCAN_WARPS * 32, 0, s>>>(b);
    uint32_t big_cap = b.lay.queues.big_cap;
    png_verify_kernel<<<(big_cap + 255) / 256, 256, 0, s>>>(b);
    return (int)cudaGetLastError();
}

static inline int png_launch_unfilter(const PngBatch &b, uint8_t *out_base, const uint64_t *out_off, uint32_t *status,
                                      int sm_count, cudaStream_t s)
{
    png_bands_kernel<<<1, PLAN_THREADS, 0, s>>>(b);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return (int)e;
    // persistent grid: every CTA must be resident (bands wait for the band above, which is always
    // an earlier work item): 80 registers x 128 threads and 17 KB of shared memory allow 6 per SM
    png_unfilter_kernel<<<(uint32_t)sm_count * 6, UNF_WARPS * 32, 0, s>>>(b, out_base, out_off, status);
    return (int)cudaGetLastError();
}

}  // namespace dbg
