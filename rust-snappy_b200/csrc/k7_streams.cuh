// k7_streams.cuh -- K7: batches of raw streams of any size (units above 64KB) around K1 / K2.
//
// Compress: unit u becomes exactly Encoder::compress(unit) (reference src/compress.rs:99-154), all units of the
// batch in one launch sequence and laid out back to back:
//   k7_plan        : thread per unit: sum of the lengths, first refused unit, exclusive scan (inside 1024-unit
//                    tiles) of the unit's item count max(1, ceil(n/65536))
//   scan_tiles     : tile totals -> first item of every unit, total item count
//   k7_expand      : thread per item slot: the owning unit (binary search over the first items), K1's input
//                    pointer and length for block k of that unit (slots past the item count get length 0)
//   K1             : every item into a kSlotStride slot, block bodies only (flags = 0)
//   k7_item_scan   : item size = body + (unit's first item ? varint length of n : 0), scanned in tiles
//   scan_tiles     : item offsets, total
//   k7_gather      : per unit its offset and status; per item (warp) varint + body to the final offset
// A unit refused by max_compress_len (== 0) has one item of size 0 and status TooBig{n, 2^32-1}; an empty unit has
// one zero-length item whose stream is the one byte 0x00 (src/compress.rs:104-124).
//
// Decompress: every unit is one raw stream; its output size is its varint header (0 when the header is unusable)
//   k7_dplan       : header parse + exclusive 64-bit scan of the sizes in tiles
//   scan_tiles     : dense output offsets, total
//   k7_dfill       : K2's per-unit output pointer / capacity / input length
//   K2             : unchanged, the only place that produces the reference's errors
//   k7_dfinish     : statuses K2 cannot give (call-level BufferTooSmall, inputs above 2^32-1 bytes), first failure
//   k7_dresult     : the result record
#pragma once
#include "common.cuh"
#include "k2_decompress.cuh"
#include "k4_frame.cuh"

namespace sbk {

struct StreamsCtl {
    unsigned long long sum_in;   // sum of the unit lengths (compress)
    uint32_t first_bad;          // lowest unit index with a non-Ok status (0xFFFFFFFF: none)
    uint32_t _pad;
};

struct StreamsPlan {
    const uint8_t* const* in_ptrs;  // unit inputs (device)
    const uint64_t* in_lens;
    uint32_t count;
    uint32_t max_items;             // item slots: count + total_in / 65536
    uint64_t total_in;              // caller's bound on the sum of the lengths
    uint64_t* ufirst;               // per unit: first item, tile-relative (scan)
    uint64_t* utiles;               // unit scan tiles; utiles[ntiles] = item count
    const uint8_t** item_ptr;       // per item: K1 input
    uint32_t* item_len;
    uint32_t* item_unit;            // owning unit (>= count: unused slot)
    uint8_t* slots;                 // K1 output slots, stride kSlotStride
    uint32_t* clens;                // K1 output lengths
    uint64_t* ioffs;                // per item: offset, tile-relative (scan)
    uint64_t* itiles;               // item scan tiles; itiles[ntiles] = total bytes
    uint8_t* out;
    uint64_t cap;
    uint64_t* out_offs;             // count + 1 entries
    sb_error* statuses;             // may be null
    sb_frame_result* result;
    StreamsCtl* ctl;
};

// ---- workspace (host side: shared by the library and the emulator harness; every array 256-byte aligned)
inline uint64_t k7_up256(uint64_t v) { return (v + 255) / 256 * 256; }
inline uint64_t k7_meta_bytes(uint64_t count, uint64_t max_items) {
    return 3 * k7_up256(max_items * 4 + 4) + 2 * k7_up256(max_items * 8 + 8) + k7_up256((max_items / K4_TILE + 3) * 8) +
           k7_up256(count * 8 + 8) + k7_up256((count / K4_TILE + 3) * 8) + k7_up256(sizeof(StreamsCtl)) +
           k7_up256(sizeof(sb_frame_result)) + 256;
}
// carves everything but the slots and the caller's arrays; returns the device result record's place
inline sb_frame_result* k7_carve_meta(StreamsPlan& p, void* meta) {
    uint8_t* q = (uint8_t*)k7_up256((uint64_t)(uintptr_t)meta);
    const uint64_t m = p.max_items, c = p.count;
    p.item_len = (uint32_t*)q; q += k7_up256(m * 4 + 4);
    p.item_unit = (uint32_t*)q; q += k7_up256(m * 4 + 4);
    p.clens = (uint32_t*)q; q += k7_up256(m * 4 + 4);
    p.item_ptr = (const uint8_t**)q; q += k7_up256(m * 8 + 8);
    p.ioffs = (uint64_t*)q; q += k7_up256(m * 8 + 8);
    p.itiles = (uint64_t*)q; q += k7_up256((m / K4_TILE + 3) * 8);
    p.ufirst = (uint64_t*)q; q += k7_up256(c * 8 + 8);
    p.utiles = (uint64_t*)q; q += k7_up256((c / K4_TILE + 3) * 8);
    p.ctl = (StreamsCtl*)q; q += k7_up256(sizeof(StreamsCtl));
    return (sb_frame_result*)q;
}

struct StreamsDecPlan {
    const uint8_t* const* in_ptrs;
    const uint64_t* in_lens;
    uint32_t count;
    uint8_t* out;
    uint64_t cap;
    uint64_t* out_offs;             // count + 1 entries: tile-relative after k7_dplan, absolute after k7_dfill
    uint64_t* tiles;
    uint32_t* k2_in_lens;           // K2's batch arrays
    uint8_t** k2_out_ptrs;
    uint32_t* k2_out_caps;
    uint32_t* k2_out_lens;
    sb_error* statuses;
    sb_frame_result* result;
    StreamsCtl* ctl;
};
inline uint64_t k7_dec_bytes(uint64_t count) {
    return k7_up256((count / K4_TILE + 3) * 8) + 3 * k7_up256(count * 4 + 4) + k7_up256(count * 8 + 8) +
           k7_up256(sizeof(StreamsCtl)) + 256;
}
inline void k7_carve_dec(StreamsDecPlan& p, void* scratch) {
    uint8_t* q = (uint8_t*)k7_up256((uint64_t)(uintptr_t)scratch);
    const uint64_t c = p.count;
    p.tiles = (uint64_t*)q; q += k7_up256((c / K4_TILE + 3) * 8);
    p.k2_in_lens = (uint32_t*)q; q += k7_up256(c * 4 + 4);
    p.k2_out_caps = (uint32_t*)q; q += k7_up256(c * 4 + 4);
    p.k2_out_lens = (uint32_t*)q; q += k7_up256(c * 4 + 4);
    p.k2_out_ptrs = (uint8_t**)q; q += k7_up256(c * 8 + 8);
    p.ctl = (StreamsCtl*)q;
}

// ---- compress
// max_compress_len(n) == 0 (src/compress.rs:42-53, :104-117)
SB_DEVICE bool k7_refused(uint64_t n) { return n > kMaxInput || 32 + n + n / 6 > kMaxInput; }
SB_DEVICE uint32_t k7_items(uint64_t n) { return (k7_refused(n) || n == 0) ? 1u : (uint32_t)((n + kMaxBlock - 1) / kMaxBlock); }
SB_DEVICE uint32_t k7_varint_len(uint64_t n) { uint32_t l = 1; while (n >= 0x80) { n >>= 7; l++; } return l; }
SB_DEVICE uint64_t k7_first_item(const StreamsPlan& p, uint32_t u) { return p.utiles[u / K4_TILE] + p.ufirst[u]; }
SB_DEVICE uint64_t k7_item_count(const StreamsPlan& p) { return p.utiles[(p.count + K4_TILE - 1) / K4_TILE]; }
SB_DEVICE bool k7_valid(const StreamsPlan& p) { return p.ctl->sum_in <= p.total_in && k7_item_count(p) <= p.max_items; }
// bytes in front of item i's body: the unit's varint when i is the first item of a unit that is not refused
SB_DEVICE uint32_t k7_head_len(const StreamsPlan& p, uint32_t i) {
    const uint32_t u = p.item_unit[i];
    if (u >= p.count || k7_first_item(p, u) != i) return 0;
    const uint64_t n = p.in_lens[u];
    return k7_refused(n) ? 0 : k7_varint_len(n);
}

// 1024 threads per CTA (the scan's tile). ctl zeroed, first_bad = 0xFFFFFFFF before the launch.
SB_DEVICE void k7_plan_body(const StreamsPlan& p) {
    const uint64_t u = (uint64_t)block_idx() * K4_TILE + thread_idx();
    const uint64_t n = u < p.count ? p.in_lens[u] : 0;
    if (u < p.count && k7_refused(n)) atomic_min(&p.ctl->first_bad, (uint32_t)u);
    uint64_t s = n;
#pragma unroll
    for (unsigned k = 16; k >= 1; k >>= 1) s += shfl(s, lane_id() ^ k);
    if (lane_id() == 0 && s) atomic_add(&p.ctl->sum_in, (unsigned long long)s);
    scan_local_body(p.count, [&](uint32_t i) { return k7_items(p.in_lens[i]); }, p.ufirst, p.utiles);
}
SB_DEVICE void k7_unit_tiles_body(const StreamsPlan& p) { scan_tiles_body(p.count, 0, p.utiles); }

SB_DEVICE void k7_expand_body(const StreamsPlan& p) {
    const uint64_t nthreads = (uint64_t)grid_dim() * block_dim();
    const bool valid = k7_valid(p);
    const uint64_t items = k7_item_count(p);
    for (uint64_t s = (uint64_t)block_idx() * block_dim() + thread_idx(); s < p.max_items; s += nthreads) {
        if (!valid || s >= items) { p.item_ptr[s] = nullptr; p.item_len[s] = 0; p.item_unit[s] = 0xFFFFFFFFu; continue; }
        uint32_t lo = 0, hi = p.count - 1;                 // last unit whose first item is <= s (every unit has one)
        while (lo < hi) {
            const uint32_t mid = lo + (hi - lo + 1) / 2;
            if (k7_first_item(p, mid) <= s) lo = mid; else hi = mid - 1;
        }
        const uint64_t k = s - k7_first_item(p, lo), n = p.in_lens[lo];
        const uint64_t at = k * kMaxBlock;
        const uint64_t left = (k7_refused(n) || n <= at) ? 0 : n - at;
        p.item_ptr[s] = p.in_ptrs[lo] + at;
        p.item_len[s] = left > kMaxBlock ? kMaxBlock : (uint32_t)left;
        p.item_unit[s] = lo;
    }
}

SB_DEVICE void k7_item_scan_body(const StreamsPlan& p) {
    scan_local_body(p.max_items, [&](uint32_t i) { return p.clens[i] + k7_head_len(p, i); }, p.ioffs, p.itiles);
}
SB_DEVICE void k7_item_tiles_body(const StreamsPlan& p) { scan_tiles_body(p.max_items, 0, p.itiles); }

SB_DEVICE void k7_gather_body(const StreamsPlan& p) {
    const uint64_t total = p.itiles[(p.max_items + K4_TILE - 1) / K4_TILE];
    const bool valid = k7_valid(p), fits = valid && total <= p.cap;
    const uint64_t sum = p.ctl->sum_in;
    const uint32_t bad = p.ctl->first_bad;
    // per unit: offset of its first item and its status
    const uint64_t tid = (uint64_t)block_idx() * block_dim() + thread_idx(), nthreads = (uint64_t)grid_dim() * block_dim();
    for (uint64_t u = tid; u < p.count; u += nthreads) {
        const uint64_t f = k7_first_item(p, (uint32_t)u);
        p.out_offs[u] = f < p.max_items ? p.itiles[f / K4_TILE] + p.ioffs[f] : total;
        if (p.statuses) {
            const uint64_t n = p.in_lens[u];
            if (!valid) set_status(&p.statuses[u], SB_E_INVALID, sum, p.total_in, 0);
            else if (!fits) set_status(&p.statuses[u], SB_BUFFER_TOO_SMALL, p.cap, total, 0);
            else if (k7_refused(n)) set_status(&p.statuses[u], SB_TOO_BIG, n, kMaxInput, 0);
            else set_status(&p.statuses[u], SB_OK, 0, 0, 0);
        }
    }
    if (tid == 0) {
        p.out_offs[p.count] = total;
        sb_frame_result r;
        r.status.code = SB_OK; r.status._pad = 0; r.status.a = r.status.b = r.status.c = 0;
        if (!valid) { r.status.code = SB_E_INVALID; r.status.a = sum; r.status.b = p.total_in; }
        else if (!fits) { r.status.code = SB_BUFFER_TOO_SMALL; r.status.a = p.cap; r.status.b = total; }
        else if (bad < p.count) { r.status.code = SB_TOO_BIG; r.status.a = p.in_lens[bad]; r.status.b = kMaxInput; }
        r.bytes = fits ? total : 0;
        r.nchunks = (uint32_t)k7_item_count(p); r._pad = 0;
        *p.result = r;
    }
    if (!fits) return;
    // per item (warp): the unit's varint in front of its first block, then the block body
    const unsigned wpb = block_dim() >> 5, lane = lane_id();
    const uint64_t nwarps = (uint64_t)grid_dim() * wpb;
    for (uint64_t w = (uint64_t)block_idx() * wpb + warp_id(); w < p.max_items; w += nwarps) {
        const uint32_t i = (uint32_t)w, c = p.clens[i];
        const uint32_t h = k7_head_len(p, i);
        if (c == 0 && h == 0) continue;
        uint8_t* dst = p.out + p.itiles[i / K4_TILE] + p.ioffs[i];
        if (lane < h) {                                                  // src/bytes.rs:61-70
            const uint64_t n = p.in_lens[p.item_unit[i]];
            dst[lane] = (uint8_t)((n >> (7 * lane)) & 0x7F) | (lane + 1 < h ? 0x80 : 0);
        }
        warp_copy_t<true>(dst + h, p.slots + (uint64_t)i * kSlotStride, c);
    }
}

// ---- decompress
// output size of a stream: its header value when usable (get_varint semantics), else 0 (K2 reports the error)
SB_DEVICE uint64_t k7_dsize(const StreamsDecPlan& p, uint32_t u) {
    const uint64_t n = p.in_lens[u];
    if (n == 0 || n > kMaxInput) return 0;
    uint64_t v = 0;
    const uint32_t hl = k2_read_header(p.in_ptrs[u], (uint32_t)n, &v);
    return (hl == 0 || v > kMaxInput) ? 0 : v;
}
// exclusive 64-bit scan inside 1024-unit tiles (a tile of 4GB outputs overflows the 32-bit scan_local_body)
SB_DEVICE void k7_dplan_body(const StreamsDecPlan& p) {
    uint64_t* sh = (uint64_t*)smem();      // 32 warp totals
    const unsigned t = thread_idx(), lane = lane_id(), wid = warp_id();
    const uint64_t i = (uint64_t)block_idx() * K4_TILE + t;
    const uint64_t v = i < p.count ? k7_dsize(p, (uint32_t)i) : 0;
    uint64_t incl = v;
#pragma unroll
    for (unsigned k = 1; k < 32; k <<= 1) { const uint64_t x = shfl(incl, lane >= k ? lane - k : lane); if (lane >= k) incl += x; }
    if (lane == 31) sh[wid] = incl;
    syncthreads();
    if (wid == 0) {
        const uint64_t w = sh[lane];
        uint64_t wi = w;
#pragma unroll
        for (unsigned k = 1; k < 32; k <<= 1) { const uint64_t x = shfl(wi, lane >= k ? lane - k : lane); if (lane >= k) wi += x; }
        sh[lane] = wi - w;
        if (lane == 31) p.tiles[block_idx()] = wi;
    }
    syncthreads();
    if (i < p.count) p.out_offs[i] = sh[wid] + (incl - v);
}
SB_DEVICE void k7_dtiles_body(const StreamsDecPlan& p) { scan_tiles_body(p.count, 0, p.tiles); }

SB_DEVICE void k7_dfill_body(const StreamsDecPlan& p) {
    const uint64_t total = p.tiles[(p.count + K4_TILE - 1) / K4_TILE];
    const bool fits = total <= p.cap;
    const uint64_t tid = (uint64_t)block_idx() * block_dim() + thread_idx(), nthreads = (uint64_t)grid_dim() * block_dim();
    if (tid == 0) p.out_offs[p.count] = total;
    for (uint64_t u = tid; u < p.count; u += nthreads) {
        const uint64_t off = p.tiles[u / K4_TILE] + p.out_offs[u], n = p.in_lens[u];
        p.out_offs[u] = off;
        p.k2_out_ptrs[u] = p.out + off;
        // a unit K2 must not touch gets a zero-length input: K2 returns at once (Empty), k7_dfinish sets its status
        p.k2_out_caps[u] = fits ? (uint32_t)k7_dsize(p, (uint32_t)u) : 0;
        p.k2_in_lens[u] = (fits && n <= kMaxInput) ? (uint32_t)n : 0;
    }
}
SB_DEVICE void k7_dfinish_body(const StreamsDecPlan& p) {
    const uint64_t total = p.out_offs[p.count];
    const bool fits = total <= p.cap;
    const uint64_t nthreads = (uint64_t)grid_dim() * block_dim();
    for (uint64_t u = (uint64_t)block_idx() * block_dim() + thread_idx(); u < p.count; u += nthreads) {
        const uint64_t n = p.in_lens[u];
        if (!fits) set_status(&p.statuses[u], SB_BUFFER_TOO_SMALL, p.cap, total, 0);
        else if (n > kMaxInput) set_status(&p.statuses[u], SB_E_INVALID, n, kMaxInput, 0);   // as sb_decompress
        if (p.statuses[u].code != SB_OK) atomic_min(&p.ctl->first_bad, (uint32_t)u);
    }
}
SB_DEVICE void k7_dresult_body(const StreamsDecPlan& p) {
    if (thread_idx() != 0) return;
    const uint64_t total = p.out_offs[p.count];
    const uint32_t bad = p.ctl->first_bad;
    sb_frame_result r;
    r.status.code = SB_OK; r.status._pad = 0; r.status.a = r.status.b = r.status.c = 0;
    if (bad < p.count) r.status = p.statuses[bad];
    r.bytes = total <= p.cap ? total : 0;
    r.nchunks = p.count; r._pad = 0;
    *p.result = r;
}

}  // namespace sbk
