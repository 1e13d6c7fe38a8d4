// Internal structures of libvlscan.so shared by vl_engine.cu (staging, scan interpreter, C ABI), vl_gen.cu
// (synthetic batch generator) and vl_zstd.cu.  The scan kernels (vl_kernels.cuh) are not included here: they are compiled
// into vl_engine.cu alone.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <algorithm>
#include <string>
#include <vector>
#include "../../include/vlscan.h"
#include "vl_types.h"
#include "vl_zstd.h"
#include "vl_zstd_walk.h"   // BadInput
#include "vl_hostpool.h"

namespace vl {

void set_thread_error(const std::string& s);
#define VL_CUDA(call)                                                                                                   \
    do {                                                                                                                \
        cudaError_t e__ = (call);                                                                                       \
        if (e__ != cudaSuccess) throw CudaFail(std::string(#call) + ": " + cudaGetErrorString(e__), (int)e__);        \
    } while (0)
struct CudaFail { std::string msg; int code; CudaFail(std::string m, int c) : msg(std::move(m)), code(c) {} };

struct DevBuf {
    void* p = nullptr; size_t cap = 0;
    void ensure(size_t n) {
        if (n <= cap) return;
        if (p) VL_CUDA(cudaFree(p));
        p = nullptr; cap = 0;
        size_t want = n + std::min<size_t>(n / 8, (size_t)256 << 20) + 256;   // growth slack, capped: a 150 GB arena must not ask for 170 GB
        VL_CUDA(cudaMalloc(&p, want)); cap = want;
    }
    void release() { if (p) cudaFree(p); p = nullptr; cap = 0; }
    template <class T> T* as() const { return (T*)p; }
};



static const size_t kArenaAlign = 16;
static const size_t kArenaPad = 32;   // readable slack after every payload (vector loads past the end, see k_substr_scan)
inline uint64_t arena_reserve(uint64_t& cursor, uint64_t len) {
    uint64_t off = (cursor + kArenaAlign - 1) / kArenaAlign * kArenaAlign;
    cursor = off + len + kArenaPad;
    return off;
}

}  // namespace vl

// opaque C ABI types
struct vlscan_batch {
    int device = 0;
    uint32_t nfields = 0;
    std::vector<std::string> field_names;
    uint64_t nblocks = 0, nwords = 0, rows = 0;
    uint64_t arena_bytes = 0, harena_bytes = 0;
    vl::DevBuf arena, cols, blk_rows, blk_word_off, word_block, init_bitmap, ts;
    vl::DevBuf harena;                    // bloom-first staging only: header payloads (bloom filters, const values, dict tables) of phase 1
    bool split_hdr = false;               // the columns' bloom_off / meta_off refer to `harena`, not to `arena`
    std::vector<vl::DevColumn> h_cols;    // bloom-first staging: the column table between the two phases
    bool has_ts = false;                  // some block came with its timestamps column
    std::vector<uint32_t> h_rows;
    std::vector<uint64_t> h_word_off;
    std::vector<uint32_t> slot_vt_mask;   // per field slot: bit vt set when some block stores the field with that valueType
    void note_columns(const std::vector<vl::DevColumn>& cols) {
        slot_vt_mask.assign(nfields, 0);
        for (size_t i = 0; i < cols.size(); i++) if (cols[i].kind == vl::COL_VALUES) slot_vt_mask[i % nfields] |= 1u << cols[i].vt;
    }
    vl::BatchView view() const {
        vl::BatchView v;
        v.arena = arena.as<uint8_t>(); v.hdr = split_hdr ? harena.as<uint8_t>() : arena.as<uint8_t>(); v.cols = cols.as<vl::DevColumn>(); v.blk_rows = blk_rows.as<uint32_t>();
        v.blk_word_off = blk_word_off.as<uint64_t>(); v.word_block = word_block.as<uint32_t>();
        v.ts = has_ts ? ts.as<vl::DevTimestamps>() : nullptr;
        v.nblocks = (uint32_t)nblocks; v.nfields = nfields; v.nwords = nwords;
        return v;
    }
    uint64_t device_bytes() const { return arena.cap + harena.cap + cols.cap + blk_rows.cap + blk_word_off.cap + word_block.cap + init_bitmap.cap + ts.cap; }
    ~vlscan_batch() { cudaSetDevice(device); arena.release(); harena.release(); cols.release(); blk_rows.release(); blk_word_off.release(); word_block.release(); init_bitmap.release(); ts.release(); }
};

struct vlscan_ctx {
    int device = 0;
    cudaStream_t stream = nullptr;        // compute stream: kernels, small copies, results
    cudaStream_t copy_stream = nullptr;   // host -> device payload copies of vlscan_batch_upload / vlscan_scan_batch
    std::string err;
    uint64_t launches = 0;
    // scratch (grow-only)
    vl::DevBuf action, payload, leaf_bm, lens_blocks, row_blocks, work_count, stats, totals, counts, slots, hit_offs, hits, tile_block, tile_off;
    std::vector<vl::DevBuf> regs;          // bitmap registers of the tree interpreter
    std::vector<vl::DevBuf> row_off8;      // per batch field slot: byte offset of every 8th row (k_lens_offsets)
    std::vector<vl::DevBuf> ready;         // per batch field slot: row_off8 computed for block b in this scan
    std::vector<char> ready_cleared;
    vl::DevBuf hit_block, glens, goffs, gtiles, gout, gstat;   // hit materialisation (vlscan_gather_*): block of each hit, value lengths / offsets, output staging, error slot
    vl::DevBuf ts_vals;                    // decoded timestamps / running sums, 8 bytes per row of the batch (k_time_match, gather)
    vl::DevBuf need;                       // bloom-first probe pass: one byte per (block, field), set when the column's values must be staged
    const void* bf_prog = nullptr; int bf_skip = 0;   // adaptive bloom-first: after a probe that pruned next to nothing, the next calls with the same program stage everything at once
    vl::DevBuf zsrc, zcols, ztest;         // compressed staging of on-disk values blocks; their column list; test output
    vl::ZstdDev* zdev = nullptr;           // device ZSTD decoder scratch (vl_zstd.cu)
    void* pinned = nullptr; size_t pinned_cap = 0;
    vl::HostPool* pool = nullptr;          // packing threads, started by the first upload from pageable memory
    cudaEvent_t ev_begin = nullptr, ev_end = nullptr;
    std::vector<std::pair<cudaEvent_t, cudaEvent_t>> scan_events; size_t scan_events_used = 0;
    // last scan
    const vlscan_batch* last_batch = nullptr;   // the batch of the last scan: must stay alive until its results have been fetched
    uint64_t last_nblocks = 0, last_nwords = 0, last_rows = 0;   // host-side facts about it, kept here so that counters never touch a freed batch
    vlscan_batch* recycle = nullptr;       // staging batch reused by vlscan_scan_batch
    bool has_result = false;
    uint64_t last_launches = 0;
    int sm_count = 148;
    int scan_occ[2] = {1, 1};              // resident CTAs per SM of k_substr_scan<false> / <true> on this device
    int row_occ = 1;                       // ... and of k_row_match (its persistent grid is exactly the resident set)
    void* ensure_pinned(size_t n);
};

namespace vl {
// fills word_block / init_bitmap / blk_* device arrays of a batch from host row counts (shared by upload + generate)
void finish_batch_layout(vlscan_ctx* ctx, vlscan_batch* b, const std::vector<uint32_t>& rows);
}
