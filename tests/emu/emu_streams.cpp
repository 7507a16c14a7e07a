// emu_streams.cpp -- TEST TOOLING ONLY. The raw-stream batch kernel sequences of rust-snappy_b200/csrc
// (K7 around K1 / K2, as launched by sb_compress_streams_device_ws / sb_decompress_streams_device_ws), compiled by g++
// against the fiber warp emulator and exposed to pytest (tests/test_emu_streams.py builds and loads this file).
#define SB_EMU 1
#include "simt_emu.h"
#include "../../rust-snappy_b200/csrc/k1_compress.cuh"
#include "../../rust-snappy_b200/csrc/k2_decompress.cuh"
#include "../../rust-snappy_b200/csrc/k7_streams.cuh"

// K1 with 7 shared-memory-table chains + 4 chains with tables in global memory per CTA, block bodies only (flags 0)
struct K1Args { sb_batch b; uint64_t* rings; uint16_t* gtables; uint32_t* work; };
static void k1_entry(void* a) {
    K1Args* x = (K1Args*)a;
    sbk::k1_compress_body_multi<7, 4>(x->b, 0u, x->rings, x->gtables, x->work, nullptr);
}
static void k1_run(const sb_batch& b, unsigned grid) {
    std::vector<uint64_t> rings((size_t)grid * 11 * sbk::K1_RING_GW, 0xCDCDCDCDCDCDCDCDull);
    std::vector<uint16_t> gt((size_t)grid * 5 * (sbk::K1_TABLE_BYTES / 2) + 8, 0xCDCD);
    uint32_t work = 0;
    K1Args a{b, rings.data(), (uint16_t*)(((uintptr_t)gt.data() + 15) & ~(uintptr_t)15), &work};
    sbemu::launch(grid, 11 * 64, sbk::k1_multi_smem(7, 4), k1_entry, &a);
}
static void k2_entry(void* a) { sbk::k2_decompress_body(*(sb_batch*)a); }

static void k7_plan_entry(void* a) { sbk::k7_plan_body(*(sbk::StreamsPlan*)a); }
static void k7_unit_tiles_entry(void* a) { sbk::k7_unit_tiles_body(*(sbk::StreamsPlan*)a); }
static void k7_expand_entry(void* a) { sbk::k7_expand_body(*(sbk::StreamsPlan*)a); }
static void k7_item_scan_entry(void* a) { sbk::k7_item_scan_body(*(sbk::StreamsPlan*)a); }
static void k7_item_tiles_entry(void* a) { sbk::k7_item_tiles_body(*(sbk::StreamsPlan*)a); }
static void k7_gather_entry(void* a) { sbk::k7_gather_body(*(sbk::StreamsPlan*)a); }
static void k7_dplan_entry(void* a) { sbk::k7_dplan_body(*(sbk::StreamsDecPlan*)a); }
static void k7_dtiles_entry(void* a) { sbk::k7_dtiles_body(*(sbk::StreamsDecPlan*)a); }
static void k7_dfill_entry(void* a) { sbk::k7_dfill_body(*(sbk::StreamsDecPlan*)a); }
static void k7_dfinish_entry(void* a) { sbk::k7_dfinish_body(*(sbk::StreamsDecPlan*)a); }
static void k7_dresult_entry(void* a) { sbk::k7_dresult_body(*(sbk::StreamsDecPlan*)a); }

extern "C" {

// plan -> unit tiles -> expand -> K1 (flags 0) -> item scan -> item tiles -> gather
int emu_streams_compress(const uint8_t* const* in_ptrs, const uint64_t* in_lens, uint32_t count, uint64_t total_in,
                         uint8_t* out, uint64_t cap, uint64_t* out_offs, sb_error* statuses, sb_frame_result* result) {
    sbk::StreamsPlan p;
    memset(&p, 0, sizeof p);
    p.in_ptrs = in_ptrs; p.in_lens = in_lens; p.count = count; p.total_in = total_in;
    p.max_items = (uint32_t)(count + total_in / 65536);
    std::vector<uint8_t> slots((size_t)p.max_items * sbk::kSlotStride + 64, 0xEE);
    std::vector<uint8_t> meta(sbk::k7_meta_bytes(count, p.max_items), 0xCD);
    p.slots = slots.data();
    sbk::k7_carve_meta(p, meta.data());
    p.out = out; p.cap = cap; p.out_offs = out_offs; p.statuses = statuses; p.result = result;
    p.ctl->sum_in = 0; p.ctl->first_bad = 0xFFFFFFFFu;
    const unsigned utiles = (count + sbk::K4_TILE - 1) / sbk::K4_TILE, itiles = (p.max_items + sbk::K4_TILE - 1) / sbk::K4_TILE;
    sbemu::launch(utiles ? utiles : 1, sbk::K4_TILE, 128, k7_plan_entry, &p);
    sbemu::launch(1, 1024, 1024 * 8, k7_unit_tiles_entry, &p);
    sbemu::launch(2, 256, 0, k7_expand_entry, &p);
    if (p.max_items) {
        sb_batch b;
        memset(&b, 0, sizeof b);
        b.in_ptrs = p.item_ptr; b.in_lens = p.item_len;
        b.out_base = p.slots; b.out_stride = sbk::kSlotStride; b.out_cap_uniform = sbk::kSlotStride; b.out_lens = p.clens;
        b.count = p.max_items;
        k1_run(b, 2);
    }
    sbemu::launch(itiles ? itiles : 1, sbk::K4_TILE, 128, k7_item_scan_entry, &p);
    sbemu::launch(1, 1024, 1024 * 8, k7_item_tiles_entry, &p);
    sbemu::launch(3, 256, 0, k7_gather_entry, &p);
    return 0;
}

// plan (header + 64-bit scan) -> tiles -> fill -> K2 -> finish -> result
int emu_streams_decompress(const uint8_t* const* in_ptrs, const uint64_t* in_lens, uint32_t count, uint8_t* out, uint64_t cap,
                           uint64_t* out_offs, sb_error* statuses, sb_frame_result* result) {
    sbk::StreamsDecPlan p;
    memset(&p, 0, sizeof p);
    p.in_ptrs = in_ptrs; p.in_lens = in_lens; p.count = count;
    p.out = out; p.cap = cap; p.out_offs = out_offs; p.statuses = statuses; p.result = result;
    std::vector<uint8_t> scratch(sbk::k7_dec_bytes(count), 0xCD);
    sbk::k7_carve_dec(p, scratch.data());
    p.ctl->first_bad = 0xFFFFFFFFu;
    const unsigned tiles = (count + sbk::K4_TILE - 1) / sbk::K4_TILE;
    sbemu::launch(tiles ? tiles : 1, sbk::K4_TILE, 32 * 8, k7_dplan_entry, &p);
    sbemu::launch(1, 1024, 1024 * 8, k7_dtiles_entry, &p);
    sbemu::launch(2, 256, 0, k7_dfill_entry, &p);
    sb_batch b;
    memset(&b, 0, sizeof b);
    b.in_ptrs = p.in_ptrs; b.in_lens = p.k2_in_lens; b.out_ptrs = p.k2_out_ptrs; b.out_caps = p.k2_out_caps;
    b.out_lens = p.k2_out_lens; b.statuses = p.statuses; b.count = count;
    if (count) sbemu::launch(2, 64, 2 * sbk::K2_SMEM_PER_WARP, k2_entry, &b);
    sbemu::launch(2, 256, 0, k7_dfinish_entry, &p);
    sbemu::launch(1, 32, 0, k7_dresult_entry, &p);
    return 0;
}

}
