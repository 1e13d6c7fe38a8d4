// libvlscan.so: staging of column blocks into HBM, the filter-tree interpreter that drives the CUDA kernels, and the
// C ABI declared in include/vlscan.h.  There is no CPU code path for the scan itself: without a CUDA device every
// computing entry point fails with an error.
#include <dlfcn.h>
#include <algorithm>
#include <atomic>
#include <chrono>
#include <thread>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <memory>
#include <mutex>
#include "vl_engine.h"
#include "vl_kernels.cuh"
#include "vl_program.h"
#include "vl_part.h"
#include "vl_mathnum.cuh"

using namespace vl;

namespace vl {
static thread_local std::string g_thread_err;
void set_thread_error(const std::string& s) { g_thread_err = s; }
}  // namespace vl

struct vlscan_program {
    Program p;
    struct Image { DevBuf leaves, prepass, regexes, blob, u64s, u32s; DevProgram view; };
    std::map<int, std::unique_ptr<Image>> images;
    std::mutex mu;
    const DevProgram& image(int device, cudaStream_t st) {
        std::lock_guard<std::mutex> g(mu);
        auto it = images.find(device);
        if (it != images.end()) return it->second->view;
        auto im = std::make_unique<Image>();
        auto up = [&](DevBuf& b, const void* src, size_t n) { b.ensure(std::max<size_t>(n, 16)); if (n) VL_CUDA(cudaMemcpyAsync(b.p, src, n, cudaMemcpyHostToDevice, st)); };
        up(im->leaves, p.leaves.data(), p.leaves.size() * sizeof(DevLeaf));
        up(im->prepass, p.prepass.data(), p.prepass.size() * sizeof(DevPrepass));
        up(im->regexes, p.regexes.data(), p.regexes.size() * sizeof(DevRegex));
        up(im->blob, p.blob.data(), p.blob.size());
        up(im->u64s, p.u64s.data(), p.u64s.size() * 8);
        up(im->u32s, p.u32s.data(), p.u32s.size() * 4);
        VL_CUDA(cudaStreamSynchronize(st));
        im->view = DevProgram{im->leaves.as<DevLeaf>(), im->prepass.as<DevPrepass>(), im->regexes.as<DevRegex>(), im->blob.as<uint8_t>(), im->u64s.as<uint64_t>(), im->u32s.as<uint32_t>()};
        auto& ref = *im;
        images[device] = std::move(im);
        return ref.view;
    }
    ~vlscan_program() { for (auto& kv : images) { cudaSetDevice(kv.first); kv.second->leaves.release(); kv.second->prepass.release(); kv.second->regexes.release(); kv.second->blob.release(); kv.second->u64s.release(); kv.second->u32s.release(); } }
};

struct vlscan_host_blocks {
    void* pinned = nullptr; size_t bytes = 0;
    std::vector<vlscan_block> blocks;
    std::vector<vlscan_column> cols;
    std::vector<std::string> fields;
    std::vector<std::vector<uint32_t>> dict_offsets;
    std::vector<std::unique_ptr<std::vector<uint8_t>>> owned;   // dict tables rebuilt from a part's column headers
    std::vector<uint64_t> source;                               // vlscan_part_blocks: index of each block inside the part
};
struct vlscan_part { vl::part::PartReader r; };

void* vlscan_ctx::ensure_pinned(size_t n) {
    if (n <= pinned_cap) return pinned;
    if (pinned) cudaFreeHost(pinned);
    pinned = nullptr; pinned_cap = 0;
    VL_CUDA(cudaMallocHost(&pinned, n));
    pinned_cap = n;
    return pinned;
}

namespace {

// ---- error plumbing --------------------------------------------------------------------------------------------------
template <class F> int guarded(vlscan_ctx* ctx, F&& f) {
    try { f(); return 0; }
    catch (const CudaFail& e) { set_thread_error(e.msg); if (ctx) ctx->err = e.msg; return e.code > 0 ? e.code : 1; }
    catch (const BadInput& e) { set_thread_error(e.msg); if (ctx) ctx->err = e.msg; return -1; }
    catch (const ProgError& e) { set_thread_error(e.what()); if (ctx) ctx->err = e.what(); return -2; }
    catch (const std::exception& e) { set_thread_error(e.what()); if (ctx) ctx->err = e.what(); return -3; }
}

// ---- libzstd, COMPRESSION only: vlscan_host_blocks_compress plays the reference's writer (marshalBytesBlock, encoding.go:343-360) so that
// benches and tests can feed on-disk-stage blocks.  Nothing on the scan path calls into it: frames are decoded on the device (vl_zstd.cuh).
struct ZstdWriter {
    size_t (*compress)(void*, size_t, const void*, size_t, int) = nullptr;
    size_t (*bound)(size_t) = nullptr;
    unsigned (*is_error)(size_t) = nullptr;
    bool ok = false;
    ZstdWriter() {
        void* h = dlopen("libzstd.so.1", RTLD_NOW | RTLD_GLOBAL);
        if (!h) return;
        compress = (decltype(compress))dlsym(h, "ZSTD_compress");
        bound = (decltype(bound))dlsym(h, "ZSTD_compressBound");
        is_error = (decltype(is_error))dlsym(h, "ZSTD_isError");
        ok = compress && bound && is_error;
    }
};
ZstdWriter& zstd_writer() { static ZstdWriter z; return z; }

void launch_check(vlscan_ctx* ctx) { ctx->launches++; VL_CUDA(cudaGetLastError()); }
inline unsigned cdiv(uint64_t a, uint64_t b) { return (unsigned)((a + b - 1) / b); }

}  // namespace

// ---- batch layout shared with the generator ------------------------------------------------------------------------------
namespace vl {
void finish_batch_layout(vlscan_ctx* ctx, vlscan_batch* b, const std::vector<uint32_t>& rows) {
    b->nblocks = rows.size();
    b->h_rows = rows;
    b->h_word_off.assign(rows.size() + 1, 0);
    b->rows = 0;
    for (size_t i = 0; i < rows.size(); i++) { b->h_word_off[i + 1] = b->h_word_off[i] + (rows[i] + 63) / 64; b->rows += rows[i]; }
    b->nwords = b->h_word_off.back();
    std::vector<uint32_t> wb(b->nwords);
    std::vector<uint64_t> init(b->nwords);
    for (size_t i = 0; i < rows.size(); i++) {
        for (uint64_t w = b->h_word_off[i]; w < b->h_word_off[i + 1]; w++) { wb[w] = (uint32_t)i; init[w] = ~0ull; }
        uint32_t tail = rows[i] & 63;   // bitmap.setBits: tail bits beyond bitsLen stay zero (bitmap.go:62-72)
        if (tail) init[b->h_word_off[i + 1] - 1] = (~0ull) >> (64 - tail);
    }
    b->blk_rows.ensure(std::max<size_t>(rows.size() * 4, 16));
    b->blk_word_off.ensure((rows.size() + 1) * 8);
    b->word_block.ensure(std::max<size_t>(b->nwords * 4, 16));
    b->init_bitmap.ensure(std::max<size_t>(b->nwords * 8, 16));
    if (!rows.empty()) VL_CUDA(cudaMemcpyAsync(b->blk_rows.p, rows.data(), rows.size() * 4, cudaMemcpyHostToDevice, ctx->stream));
    VL_CUDA(cudaMemcpyAsync(b->blk_word_off.p, b->h_word_off.data(), (rows.size() + 1) * 8, cudaMemcpyHostToDevice, ctx->stream));
    if (b->nwords) {
        VL_CUDA(cudaMemcpyAsync(b->word_block.p, wb.data(), b->nwords * 4, cudaMemcpyHostToDevice, ctx->stream));
        VL_CUDA(cudaMemcpyAsync(b->init_bitmap.p, init.data(), b->nwords * 8, cudaMemcpyHostToDevice, ctx->stream));
    }
    VL_CUDA(cudaStreamSynchronize(ctx->stream));   // wb / init are stack-owned
}
}  // namespace vl

// ---- upload --------------------------------------------------------------------------------------------------------------
// The on-disk values blocks of a batch in (block, column) order; each one's place in the compressed staging buffer is a running sum that
// starts behind 512 bytes of headroom (the device bit readers load whole aligned words around a stream).  Returns the end of the last one.
// need (may be NULL = all): need[block * nfields + field] != 0 for the columns whose values are staged (phase 2 of a bloom-first upload).
static uint64_t collect_values_blocks(const vlscan_block* blocks, uint64_t nblocks, std::vector<ZValuesBlock>& zv, const uint8_t* need = nullptr, uint32_t nfields = 0) {
    uint64_t zc = 512;
    for (uint64_t b = 0; b < nblocks; b++)
        for (uint32_t k = 0; k < blocks[b].ncols; k++) {
            const vlscan_column& c = blocks[b].cols[k];
            if (c.kind != VLSCAN_COL_VALUES || c.stage != VLSCAN_STAGE_ONDISK) continue;
            if (need && (c.field >= nfields || !need[b * nfields + c.field])) continue;
            zv.push_back({c.values, (size_t)c.values_len, zc});
            zc += c.values_len;
        }
    return zc;
}
// Host threads for the header walk and the descriptor tables of an upload: VLSCAN_HOST_THREADS, else up to 16 (one process per GPU shares the
// box with its peers).  0 selects the single-threaded block-by-block walk.
static int host_threads() {
    if (const char* e = getenv("VLSCAN_HOST_THREADS")) return std::max(0, std::min(256, atoi(e)));
    return (int)std::max(1u, std::min(16u, std::thread::hardware_concurrency()));
}

namespace {
// one host -> device copy: `len` bytes at host address `src` to offset `dst` of a device buffer
struct Piece { const uint8_t* src; uint64_t len; uint64_t dst; };

// The copied part of an arena: payloads reserved one behind the other (arena_reserve), each with the host bytes that go there.
struct ArenaLayout {
    uint64_t cursor = 16;   // the first 16 bytes stay unused so that every payload has a readable byte in front of it
    std::vector<Piece> pieces;
    std::vector<std::unique_ptr<std::vector<uint8_t>>> owned;   // dict tables built here
    uint64_t put(const uint8_t* src, uint64_t len) { const uint64_t off = arena_reserve(cursor, len); if (len) pieces.push_back({src, len, off}); return off; }
    // The header payloads of one column in their arena order: a const column's value (-> meta_off); a values column's bloom filter
    // (-> bloom_off, `bloom_len` bytes: 0 for a filter left on the host), then for a dict column its u32 offsets[dict_len + 1] ++ values
    // (-> meta_off).  vlscan_host_blocks_compress lays out its copied part with this same function, so that its buffer goes out as one DMA.
    void put_headers(const vlscan_column& c, uint64_t bloom_len, DevColumn& d) {
        if (c.kind == VLSCAN_COL_CONST) { d.meta_off = put(c.const_value, c.const_len); return; }
        d.bloom_off = put(c.bloom, bloom_len);
        if (c.value_type != VT_DICT) return;
        const uint32_t total = c.dict_len ? c.dict_offsets[c.dict_len] : 0;
        if (c.dict_len && c.dict_blob == (const uint8_t*)c.dict_offsets + 4 * (c.dict_len + 1)) {
            d.meta_off = put((const uint8_t*)c.dict_offsets, 4 * (c.dict_len + 1) + total);   // caller memory already has the device layout
            return;
        }
        auto meta = std::make_unique<std::vector<uint8_t>>(4 * (c.dict_len + 1) + total);   // zeros: an empty dict has offsets[0] = 0
        if (c.dict_len) memcpy(meta->data(), c.dict_offsets, 4 * (c.dict_len + 1));
        if (total) memcpy(meta->data() + 4 * (c.dict_len + 1), c.dict_blob, total);
        d.meta_off = put(meta->data(), meta->size());
        owned.push_back(std::move(meta));
    }
};

// What one upload puts where, decided on the host alone (no CUDA call): the column and timestamps tables, validated on the way (the
// vlscan_block descriptors are untrusted input), the host pieces of the arena and of the compressed staging buffer, and the arena regions
// the device decoder regenerates on-disk payloads into.
//
// `headers` places what the header dispatch and the bloom probes look at: column kinds, const values, bloom filters, dict tables.  `values`
// places the timestamps and the values payloads.  Both make a full upload.  Headers alone leave every values payload on the host
// (VALUES_DEFERRED); values alone continue the table of such a header phase with the values of the columns `need` marks and flag the
// others VALUES_ABSENT.  On-disk values blocks are not copied into the arena: their bytes go to the compressed staging buffer as they are
// and the device regenerates them (vl_zstd.cuh) into arena regions placed behind everything that is copied, so that host memory laid out
// like the copied part still goes out as one DMA.
class UploadPlan {
public:
    std::vector<DevColumn>& cols;     // [nblocks * nfields]
    std::vector<DevTimestamps> tsv;   // [nblocks], or empty when no block came with its timestamps column
    std::vector<uint32_t> rows;
    ArenaLayout layout;               // the copied part of the arena
    std::vector<Piece> zpieces;       // host -> compressed staging buffer: the on-disk values blocks, then the ZSTD timestamps blocks
    uint64_t zbytes = 0;              // end of the last one
    ZstdJob zjob;                     // the frames inside zpieces, with their arena destinations
    std::vector<OndiskCol> ocols;     // lens header checks + lens_type / lens_const / data_const: k_finish_ondisk_cols
    bool decode = false;              // the device decoder regenerates something
    uint64_t arena_bytes = 0;

    // need_bloom (may be NULL = all): per batch field, whether the program that will scan this batch ever probes that field's bloom filters.
    // A filter nobody probes stays on the host (the reference reads a column's bloom filter lazily, only when a filter asks for it:
    // getBloomFilterForColumn, block_search.go:411-439); the column is staged with an empty filter, which no kernel touches.
    UploadPlan(const vlscan_block* blocks, uint64_t nblocks, uint32_t nfields, bool headers, bool values, const std::vector<char>* need_bloom,
               const uint8_t* need, std::vector<DevColumn>& cols)
        : cols(cols), blocks(blocks), nblocks(nblocks), nfields(nfields), headers(headers), values(values), need_bloom(need_bloom), need(need) {
        if (nblocks > 0xFFFFFFF0ull) throw BadInput("too many blocks in one batch");
        const size_t ncells = (size_t)nblocks * std::max<uint32_t>(nfields, 1);
        if (headers) { cols.assign(ncells, DevColumn{}); memset(cols.data(), 0, cols.size() * sizeof(DevColumn)); }
        else if (cols.size() != ncells || !need) throw BadInput("internal: values phase of a bloom-first upload without its header phase");
        rows.resize(nblocks);
    }

    // The compressed pieces and their places in the staging buffer (values only).  They are known before anything else, so that the
    // caller can have the DMA engine busy while the host walks frame and block headers.
    void collect_compressed() {
        uint64_t zc = collect_values_blocks(blocks, nblocks, zv, headers ? nullptr : need, nfields);
        for (const ZValuesBlock& v : zv) if (v.n) zpieces.push_back({v.p, v.n, v.zoff});
        // ZSTD-compressed timestamps blocks (marshal types 1 and 4) travel the same way, behind the values blocks
        for (uint64_t b = 0; b < nblocks; b++) {
            const vlscan_block& blk = blocks[b];
            if (blk.ts_marshal_type != MT_ZSTD_NEAREST_DELTA2 && blk.ts_marshal_type != MT_ZSTD_NEAREST_DELTA) continue;
            if (blk.timestamps_len > vl::part::kMaxTimestampsBlockSize) throw BadInput("timestamps block size cannot exceed 8 MiB");   // getTimestamps block_search.go:490-493
            zts_off.push_back(zc);
            if (blk.timestamps_len) zpieces.push_back({blk.timestamps, blk.timestamps_len, zc});
            zc += blk.timestamps_len;
        }
        zbytes = zc;
    }
    // frame, block and section headers of the on-disk values blocks, on several host threads; a malformed block is reported when describe()
    // gets to it
    void walk_headers() {
        zinfo.resize(zv.size());
        if (!zv.empty()) zjob.add_values_blocks(zv.data(), zv.size(), host_threads(), zinfo.data(), &zbad, &zmsg);
    }
    size_t values_blocks() const { return zv.size(); }
    // The descriptor pass: every block, its timestamps, its columns in the caller's order (the order of the arena pieces), then the
    // regenerated regions behind the copied part.
    void describe() {
        for (uint64_t b = 0; b < nblocks; b++) {
            const vlscan_block& blk = blocks[b];
            if (blk.rows > (8u << 20)) throw BadInput("block rows exceed maxRowsPerBlock (8Mi)");   // consts.go:24
            rows[b] = (uint32_t)blk.rows;
            if (blk.ts_marshal_type && values) place_timestamps(b, blk);
            for (uint32_t k = 0; k < blk.ncols; k++) {
                const vlscan_column& c = blk.cols[k];
                if (c.field >= nfields) throw BadInput("column refers to a field outside the batch field table");
                place_column(b, blk, c, cols[(size_t)b * nfields + c.field]);
            }
        }
        const uint64_t regen_base = (layout.cursor + kArenaAlign - 1) / kArenaAlign * kArenaAlign;
        for (const Ondisk& o : ondisk) {
            DevColumn& d = cols[o.col];
            d.lens_off += regen_base; d.data_off += regen_base;
            zjob.set_dst(o.lens_frame, regen_base + o.lens_rel); zjob.set_dst(o.data_frame, regen_base + o.data_rel);
        }
        for (const TsFrame& tf : ts_frames) { tsv[tf.block].off = regen_base + tf.rel; zjob.set_dst(tf.frame, regen_base + tf.rel); }
        decode = !ondisk.empty() || !ts_frames.empty();
        arena_bytes = (decode ? regen_base + regen_cursor : layout.cursor) + kArenaPad;
    }

private:
    const vlscan_block* blocks; uint64_t nblocks; uint32_t nfields;
    bool headers, values;
    const std::vector<char>* need_bloom;
    const uint8_t* need;
    std::vector<ZValuesBlock> zv; std::vector<ZValuesInfo> zinfo; size_t zbad = SIZE_MAX, zo = 0; std::string zmsg;
    std::vector<uint64_t> zts_off; size_t zt = 0;   // staging offsets of the ZSTD timestamps blocks
    uint64_t regen_cursor = 0;                      // regenerated regions, relative to the end of the copied part until describe() has sized it
    struct Ondisk { uint64_t col; uint32_t lens_frame, data_frame; uint64_t lens_rel, data_rel; };
    std::vector<Ondisk> ondisk;
    struct TsFrame { uint64_t block; uint32_t frame; uint64_t rel; };
    std::vector<TsFrame> ts_frames;

    // the timestamps column: encoded deltas as stored + timestampsHeader (block_header.go:990-997)
    void place_timestamps(uint64_t b, const vlscan_block& blk) {
        if (blk.ts_marshal_type > MT_NEAREST_DELTA) throw BadInput("unknown MarshalType of a timestamps block");
        if (blk.timestamps_len > vl::part::kMaxTimestampsBlockSize) throw BadInput("timestamps block size cannot exceed 8 MiB");
        if (tsv.empty()) { tsv.resize(nblocks); memset(tsv.data(), 0, nblocks * sizeof(DevTimestamps)); }
        DevTimestamps& t = tsv[b];
        t.first = blk.min_timestamp; t.max = blk.max_timestamp;
        if (blk.ts_marshal_type == MT_ZSTD_NEAREST_DELTA2 || blk.ts_marshal_type == MT_ZSTD_NEAREST_DELTA) {
            uint64_t regen = 0; uint32_t id = 0;
            zjob.add_frame(blk.timestamps, blk.timestamps_len, zts_off[zt++], &regen, &id);   // throws on a malformed frame header
            if (regen > 10ull * blk.rows + 16) throw BadInput("cannot unmarshal timestamps: the decompressed block is larger than its varints can be");
            t.mt = blk.ts_marshal_type == MT_ZSTD_NEAREST_DELTA2 ? MT_NEAREST_DELTA2 : MT_NEAREST_DELTA;
            t.len = (uint32_t)regen;
            ts_frames.push_back({b, id, arena_reserve(regen_cursor, regen)});
        } else {
            t.mt = (uint8_t)blk.ts_marshal_type; t.len = (uint32_t)blk.timestamps_len;
            t.off = layout.put(blk.timestamps, blk.timestamps_len);
        }
    }
    // one column of one block, headers and / or values
    void place_column(uint64_t b, const vlscan_block& blk, const vlscan_column& c, DevColumn& d) {
        if (!headers) {   // the headers are on the device since the header phase; now the values of the columns the probe pass marked
            if (c.kind != VLSCAN_COL_VALUES) return;
            if (!need[b * nfields + c.field]) { d.values_state = VALUES_ABSENT; return; }
            d.values_state = VALUES_STAGED;
            place_values(b, blk, c, d);
            return;
        }
        if (d.kind != COL_MISSING) throw BadInput("duplicate column for one field in a block");
        if (c.kind == VLSCAN_COL_CONST) {
            d.kind = COL_CONST; d.meta_len = (uint32_t)c.const_len;
            layout.put_headers(c, 0, d);
            return;
        }
        if (c.kind != VLSCAN_COL_VALUES) throw BadInput("unknown column kind");
        if (c.value_type < VT_STRING || c.value_type >= VT_MAX) throw BadInput("unknown valueType");
        d.kind = COL_VALUES; d.vt = c.value_type; d.min_value = c.min_value; d.max_value = c.max_value;
        if (values) place_values(b, blk, c, d);
        else {
            if (c.stage != VLSCAN_STAGE_ONDISK && c.stage != VLSCAN_STAGE_DECODED) throw BadInput("unknown values stage");
            d.values_state = VALUES_DEFERRED;
        }
        if (c.bloom_len % 8) throw BadInput("cannot unmarshal bloomFilter from src with size not multiple by 8");   // bloomfilter.go:59-61
        const bool keep_bloom = !need_bloom || (*need_bloom)[c.field];
        d.bloom_words = keep_bloom ? (uint32_t)(c.bloom_len / 8) : 0;
        if (c.value_type == VT_DICT) {
            if (c.dict_len > 8) throw BadInput("valuesDict may contain max 8 items");
            d.dict_len = c.dict_len;
            d.meta_len = c.dict_len ? c.dict_offsets[c.dict_len] : 0;
        }
        layout.put_headers(c, keep_bloom ? c.bloom_len : 0, d);
    }
    // the values payload of one column: on-disk stage -> regenerated by the device decoder, decoded stage -> copied
    void place_values(uint64_t b, const vlscan_block& blk, const vlscan_column& c, DevColumn& d) {
        if (c.stage == VLSCAN_STAGE_ONDISK) {
            // stringsBlockUnmarshaler.unmarshal: bytesBlock(lens) ++ bytesBlock(data) (encoding.go:83-108).  The host reads the
            // containers, the frame header and the block headers; the payload is regenerated on the device.
            if (zo == zbad) throw BadInput(zmsg);
            const uint64_t lens_len = zinfo[zo].lens_len, data_len = zinfo[zo].data_len;
            const uint32_t f1 = (uint32_t)(2 * zo), f2 = f1 + 1;
            zo++;
            if (data_len > 0xFFFFFFFFull) throw BadInput("values block too large");
            // the uint block type byte lands on offset 15 of its region, so the lens items behind it are 16-byte aligned
            const uint64_t lr = arena_reserve(regen_cursor, lens_len + 15), dr = arena_reserve(regen_cursor, data_len);
            d.lens_off = lr + 16; d.data_off = dr; d.data_len = data_len;
            const uint64_t ci = (uint64_t)b * nfields + c.field;
            ondisk.push_back({ci, f1, f2, lr + 15, dr});
            ocols.push_back({ci, lens_len, blk.rows});
        } else if (c.stage == VLSCAN_STAGE_DECODED) {
            const uint8_t* lens_items = c.lens_items; const uint64_t lens_len = c.lens_items_len, data_len = c.data_len;
            // unmarshalUint64Items header checks (encoding.go:246-336)
            if (lens_len < 1) throw BadInput("cannot unmarshal uint64 block type from empty src");
            uint8_t lt = lens_items[0];
            if (lt > 7) throw BadInput("unexpected uint64 block type");
            uint64_t want = lt < 4 ? (blk.rows << lt) : (1ull << (lt - 4));
            if (lens_len - 1 != want) throw BadInput("unexpected block length for uint items");
            d.lens_type = lt;
            if (lt >= 4) { uint64_t v = 0; for (uint64_t i = 0; i < want; i++) v = (v << 8) | lens_items[1 + i]; if (v > 0xFFFFFFFFull) throw BadInput("row length does not fit 32 bits"); d.lens_const = (uint32_t)v; }
            if (data_len > 0xFFFFFFFFull) throw BadInput("values block too large");
            d.lens_off = layout.put(lens_items + 1, lens_len - 1);
            d.data_off = layout.put(c.data, data_len); d.data_len = data_len;
            // decode rule of encoding.go:113-120: rows >= 2, all lens equal, len(data) == lens[0] => every row = data
            d.data_const = (blk.rows >= 2 && lt >= 4 && data_len == d.lens_const) ? 1 : 0;
        } else throw BadInput("unknown values stage");
    }
};

// cuPointerGetAttribute of the driver library the runtime has loaded (the runtime API only classifies single addresses)
typedef int (*PointerAttrFn)(void*, int, unsigned long long);
PointerAttrFn pointer_attr_fn() {
    static const PointerAttrFn fn = [] { void* h = dlopen("libcuda.so.1", RTLD_NOW | RTLD_GLOBAL); return h ? (PointerAttrFn)dlsym(h, "cuPointerGetAttribute") : (PointerAttrFn) nullptr; }();
    if (!fn) throw CudaFail("cuPointerGetAttribute not found in libcuda.so.1: page-locked host ranges cannot be told apart", (int)cudaErrorSharedObjectSymbolNotFound);
    return fn;
}

// The host -> device payload copies of one upload, all on the ctx's copy stream; the compute stream picks them up through events.  A run of
// pieces that are contiguous on both sides (src stride == dst stride) and lie inside one page-locked allocation goes out as one
// cudaMemcpyAsync; everything else is packed into a pinned two-chunk staging ring.  Marked copies record (end offset, event) pairs, so
// that the decoder of a launch group can start as soon as the bytes of that group have landed, while later bytes are still in flight.
// Every event lives until the copier is destroyed, by return or by exception (a worker that keeps hitting malformed parts must not leak one
// event per batch).
class H2DCopier {
public:
    uint64_t h2d = 0;       // bytes this upload sent
    bool staged = false;    // some run went through the staging ring

    explicit H2DCopier(vlscan_ctx* ctx) : ctx(ctx), cs(ctx->copy_stream), pointer_attr(pointer_attr_fn()) {}
    ~H2DCopier() { for (cudaEvent_t e : events) cudaEventDestroy(e); }
    H2DCopier(const H2DCopier&) = delete;
    H2DCopier& operator=(const H2DCopier&) = delete;

    // Is [p, p + len) inside ONE page-locked allocation?  The driver knows the range of the allocation an address belongs to
    // (RANGE_START_ADDR / RANGE_SIZE).  Pointer queries cost microseconds each and a part's descriptors come as tens of thousands of small
    // pieces (timestamps, const values) out of the same mmap()ed files: the last answers are remembered.  A 2 MiB-aligned region around a
    // pageable address is taken as pageable as a whole (if a page-locked allocation begins inside it, its pieces merely take the staging
    // ring), a page-locked allocation by its exact range.
    bool pinned(const uint8_t* p, uint64_t len) {
        const uintptr_t a = (uintptr_t)p;
        if (a >= pageable_lo && a < pageable_hi) return false;
        if (a >= locked_lo && a + len <= locked_hi) return true;
        cudaPointerAttributes at;
        if (cudaPointerGetAttributes(&at, p) != cudaSuccess) { cudaGetLastError(); at.type = cudaMemoryTypeUnregistered; }
        if (at.type != cudaMemoryTypeHost) { pageable_lo = a & ~(uintptr_t)((2u << 20) - 1); pageable_hi = pageable_lo + (2u << 20); return false; }
        unsigned long long base = 0; size_t size = 0;
        if (pointer_attr(&base, 11 /* CU_POINTER_ATTRIBUTE_RANGE_START_ADDR */, (unsigned long long)a) != 0 ||
            pointer_attr(&size, 12 /* CU_POINTER_ATTRIBUTE_RANGE_SIZE */, (unsigned long long)a) != 0) return false;
        if (size) { locked_lo = (uintptr_t)base; locked_hi = (uintptr_t)(base + size); }
        return (unsigned long long)a >= base && (unsigned long long)a + len <= base + size;
    }
    // pieces [i0, i1) to the device buffer `base`; with `marks`, every DMA records its end offset for wait_for.  The staging ring is
    // flushed at the end.
    void copy(const std::vector<Piece>& pieces, size_t i0, size_t i1, uint8_t* base, bool marks) {
        dev_base = base; marking = marks;
        size_t i = i0;
        const size_t end = std::min(i1, pieces.size());
        while (i < end) {
            // maximal run of pieces laid out identically on both sides (same stride between source and destination)
            size_t j = i;
            while (j + 1 < end && pieces[j + 1].src > pieces[j].src && pieces[j + 1].src - pieces[i].src == (ptrdiff_t)(pieces[j + 1].dst - pieces[i].dst)) j++;
            // one DMA for the whole run (gaps included) only when the run lies inside a single page-locked allocation: two pinned buffers
            // that merely line up could have pageable memory between them
            if (pinned(pieces[i].src, (pieces[j].dst - pieces[i].dst) + pieces[j].len)) {
                flush();
                // (split at piece boundaries every ~128 MB so that consumers can be released chunk by chunk)
                size_t a = i;
                while (a <= j) {
                    size_t b2 = a;
                    while (b2 < j && (pieces[b2].dst + pieces[b2].len) - pieces[a].dst < (128ull << 20)) b2++;
                    const uint64_t len = (pieces[b2].dst - pieces[a].dst) + pieces[b2].len;
                    VL_CUDA(cudaMemcpyAsync(dev_base + pieces[a].dst, pieces[a].src, len, cudaMemcpyHostToDevice, cs));
                    if (marking) mark(pieces[b2].dst + pieces[b2].len);
                    h2d += len; a = b2 + 1;
                }
                i = j + 1;
                continue;
            }
            staged = true;
            need_stage();
            for (; i <= j; i++) {
                const Piece& pc = pieces[i];
                uint64_t done = 0;
                while (done < pc.len) {
                    if (chunk_open && (chunk_dst + fill != pc.dst + done || fill == CH)) flush();
                    if (!chunk_open) { chunk_open = true; chunk_dst = pc.dst + done; fill = 0; }
                    size_t take = (size_t)std::min<uint64_t>(pc.len - done, CH - fill);
                    segs.push_back({pc.src + done, fill, take});
                    fill += take; done += take;
                }
                // pack the space up to the next piece as zeros when it follows closely, so chunks stay large: between two pieces of the copied
                // part there is nothing but alignment slack and empty reservations (a bloom filter left on the host is 48 bytes of them), zero
                // in the arena already.  With a 64-byte limit every timestamps block of a part was a chunk, a DMA and an event of its own: 16 k
                // per batch.
                if (i + 1 < end) {
                    uint64_t gap = pieces[i + 1].dst - (pc.dst + pc.len);
                    if (gap <= 1024 && fill + gap < CH) { if (gap) segs.push_back({nullptr, fill, (size_t)gap}); fill += gap; } else flush();
                }
            }
        }
        flush();
    }
    // The compressed staging buffer is filled in order: enqueue every piece of `z` not sent yet that starts below `limit`, marked
    void copy_compressed(const std::vector<Piece>& z, uint8_t* zsrc, uint64_t limit) {
        size_t hi = zsent;
        while (hi < z.size() && z[hi].dst < limit) hi++;
        if (hi == zsent) return;
        copy(z, zsent, hi, zsrc, true);
        zsent = hi;
    }
    // `st` waits until the marked copies have landed up to source offset `src_end`
    void wait_for(cudaStream_t st, uint64_t src_end) {
        for (auto& m : zmarks) if (m.first >= src_end) { VL_CUDA(cudaStreamWaitEvent(st, m.second, 0)); return; }
        if (!zmarks.empty()) VL_CUDA(cudaStreamWaitEvent(st, zmarks.back().second, 0));
    }
    // a table built on the host, counted like the pieces
    void copy_table(void* dst, const void* src, size_t n) { if (n) VL_CUDA(cudaMemcpyAsync(dst, src, n, cudaMemcpyHostToDevice, cs)); h2d += n; }
    // the copies enqueued from now on start after what `st` has enqueued so far
    void after(cudaStream_t st) { cudaEvent_t e = make(); VL_CUDA(cudaEventRecord(e, st)); VL_CUDA(cudaStreamWaitEvent(cs, e, 0)); }
    // an event that completes with every copy enqueued so far
    cudaEvent_t done() { cudaEvent_t e = make(); VL_CUDA(cudaEventRecord(e, cs)); return e; }

private:
    static constexpr size_t CH = 64u << 20;   // staging ring chunk
    vlscan_ctx* ctx; cudaStream_t cs;
    PointerAttrFn pointer_attr;
    std::vector<cudaEvent_t> events;
    std::vector<std::pair<uint64_t, cudaEvent_t>> zmarks;
    size_t zsent = 0;
    uintptr_t pageable_lo = 1, pageable_hi = 0, locked_lo = 1, locked_hi = 0;
    // the ring, and the copy being made
    uint8_t* stage = nullptr; cudaEvent_t evs[2] = {nullptr, nullptr}; int cur = 0; size_t fill = 0; uint64_t chunk_dst = 0; bool chunk_open = false;
    uint8_t* dev_base = nullptr; bool marking = false;
    // Packing pageable memory (a part's mmap()ed files) into the ring is a memcpy, ~10 GB/s on one core and page faults on cold files: the
    // segments of a chunk are only recorded while the pieces are walked, and copied by all host threads when the chunk is flushed (each
    // thread takes an equal byte range of the chunk).
    struct Seg { const uint8_t* src; size_t at, len; };   // src == nullptr: zeros
    std::vector<Seg> segs;

    cudaEvent_t make() { cudaEvent_t e; VL_CUDA(cudaEventCreateWithFlags(&e, cudaEventDisableTiming)); events.push_back(e); return e; }
    void mark(uint64_t end_off) { cudaEvent_t e = make(); VL_CUDA(cudaEventRecord(e, cs)); zmarks.push_back({end_off, e}); }
    void need_stage() {
        if (stage) return;
        stage = (uint8_t*)ctx->ensure_pinned(2 * CH);
        for (int k = 0; k < 2; k++) { evs[k] = make(); VL_CUDA(cudaEventRecord(evs[k], cs)); }
    }
    void pack_chunk(uint8_t* buf, size_t bytes) {
        const int nt = (int)std::min<size_t>(std::max(1, host_threads()), bytes / (1u << 20) + 1);
        auto work = [&](int t) {
            const size_t lo = bytes * (size_t)t / nt, hi = bytes * (size_t)(t + 1) / nt;
            size_t i = std::upper_bound(segs.begin(), segs.end(), lo, [](size_t v, const Seg& g) { return v < g.at; }) - segs.begin();
            if (i) i--;
            for (; i < segs.size() && segs[i].at < hi; i++) {
                const Seg& g = segs[i];
                const size_t a = std::max(g.at, lo), b = std::min(g.at + g.len, hi);
                if (a >= b) continue;
                if (g.src) memcpy(buf + a, g.src + (a - g.at), b - a); else memset(buf + a, 0, b - a);
            }
        };
        if (nt <= 1) { work(0); return; }
        if (!ctx->pool) ctx->pool = new HostPool;
        ctx->pool->run(nt, work);
    }
    void flush() {
        if (!chunk_open || !fill) { chunk_open = false; fill = 0; segs.clear(); return; }
        pack_chunk(stage + (size_t)cur * CH, fill);
        segs.clear();
        VL_CUDA(cudaMemcpyAsync(dev_base + chunk_dst, stage + (size_t)cur * CH, fill, cudaMemcpyHostToDevice, cs));
        VL_CUDA(cudaEventRecord(evs[cur], cs));
        if (marking) mark(chunk_dst + fill);
        h2d += fill; cur ^= 1; fill = 0; chunk_open = false;
        VL_CUDA(cudaEventSynchronize(evs[cur]));
    }
};
}  // namespace

// mode: UP_FULL stages everything in one go.  A bloom-first upload (vlscan_scan_batch, the reference's lazy order: a column's values are read only
// after its bloom filter let the block through, block_search.go:411-439 then :444-474) runs the function twice around the probe pass:
// UP_HEADERS stages the headers (-> batch->harena), UP_VALUES then the timestamps and the values of the columns the probe marked in `need`
// (-> batch->arena).
enum UploadMode { UP_FULL = 0, UP_HEADERS = 1, UP_VALUES = 2 };
static void do_upload(vlscan_ctx* ctx, const char* const* field_names, const size_t* field_name_lens, uint32_t nfields, const vlscan_block* blocks,
                      uint64_t nblocks, vlscan_batch* out, vlscan_stats* stats, const std::vector<char>* need_bloom = nullptr, UploadMode mode = UP_FULL,
                      const uint8_t* need = nullptr) {
    VL_CUDA(cudaSetDevice(ctx->device));
    const bool dbg = getenv("VLSCAN_DEBUG_TIMING") != nullptr;
    auto now = [] { return std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count(); };
    double t_start = now(), t_desc = 0, t_alloc = 0, t_copy = 0;
    const bool headers = mode != UP_VALUES, values = mode != UP_HEADERS;
    UploadPlan plan(blocks, nblocks, nfields, headers, values, need_bloom, need, out->h_cols);
    out->device = ctx->device; out->nfields = nfields;
    if (headers) for (uint32_t f = 0; f < nfields; f++) out->field_names.emplace_back(field_names[f], field_name_lens[f]);
    out->split_hdr = !(headers && values);
    DevBuf& arena = values ? out->arena : out->harena;
    H2DCopier copier(ctx);
    bool zlazy = false;
    if (values) {
        plan.collect_compressed();
        // Page-locked sources: everything is enqueued right away (asynchronous DMA), so that the DMA engine is busy while the host walks the
        // headers.  Pageable sources (a part's mmap()ed files) have to be packed through the staging ring by this thread: that is done lazily,
        // launch group by launch group, from the decoder's group hook below, so that the device decodes group g while the host packs group
        // g + 1 (packing it all here would finish before the first kernel starts).
        if (!plan.zpieces.empty()) {
            ctx->zsrc.ensure(plan.zbytes + 512);
            zlazy = !copier.pinned(plan.zpieces[0].src, plan.zpieces[0].len);
            if (!zlazy) copier.copy_compressed(plan.zpieces, ctx->zsrc.as<uint8_t>(), UINT64_MAX);
        }
        const double t_w = now();
        plan.walk_headers();
        if (dbg) fprintf(stderr, "[vlscan upload] header walk of %zu values blocks on %d host threads: %.1f ms (after %.1f ms of collecting and enqueueing the copies)\n",
                         plan.values_blocks(), host_threads(), 1e3 * (now() - t_w), 1e3 * (t_w - t_start));
    }
    plan.describe();
    (values ? out->arena_bytes : out->harena_bytes) = plan.arena_bytes;
    if (headers && values) out->harena_bytes = 0;
    t_desc = now();
    arena.ensure(plan.arena_bytes);
    t_alloc = now();
    // the arena is cleared on the compute stream; the copy stream takes over from there
    VL_CUDA(cudaMemsetAsync(arena.p, 0, plan.arena_bytes, ctx->stream));
    copier.after(ctx->stream);
    // The decoder is enqueued BEFORE anything below that can block this thread (packing pageable pieces through the staging ring, copies
    // from pageable vectors): each launch group then runs as soon as its compressed bytes have landed, beside the DMA of the later ones.
    double t_h2d = 0, t_zrun = 0;
    if (dbg) t_h2d = now();
    if (plan.decode) {
        plan.zjob.set_group_hook([&](uint64_t src_end) {
            if (zlazy) copier.copy_compressed(plan.zpieces, ctx->zsrc.as<uint8_t>(), src_end);
            copier.wait_for(ctx->stream, src_end);
        });
        plan.zjob.run(ctx, ctx->zsrc.as<uint8_t>(), arena.as<uint8_t>());
        if (zlazy) copier.copy_compressed(plan.zpieces, ctx->zsrc.as<uint8_t>(), UINT64_MAX);
        if (dbg) t_zrun = now();
    }
    copier.copy(plan.layout.pieces, 0, plan.layout.pieces.size(), arena.as<uint8_t>(), false);
    const std::vector<DevColumn>& cols = plan.cols;
    out->cols.ensure(std::max<size_t>(cols.size() * sizeof(DevColumn), 16));
    copier.copy_table(out->cols.p, cols.data(), cols.size() * sizeof(DevColumn));
    out->has_ts = !plan.tsv.empty();
    if (out->has_ts) {
        out->ts.ensure(nblocks * sizeof(DevTimestamps));
        copier.copy_table(out->ts.p, plan.tsv.data(), nblocks * sizeof(DevTimestamps));
    }
    const cudaEvent_t ev_copied = copier.done();
    const double t_enq = dbg ? now() : 0;
    if (plan.decode) {
        // the on-disk payloads are being regenerated in HBM; derive lens_type / lens_const / data_const from the regenerated lens blocks
        const std::vector<OndiskCol>& ocols = plan.ocols;
        VL_CUDA(cudaStreamWaitEvent(ctx->stream, ev_copied, 0));
        ctx->zcols.ensure(16 + ocols.size() * sizeof(OndiskCol));
        VL_CUDA(cudaMemsetAsync(ctx->zcols.p, 0, 16, ctx->stream));
        VL_CUDA(cudaMemcpyAsync(ctx->zcols.as<uint8_t>() + 16, ocols.data(), ocols.size() * sizeof(OndiskCol), cudaMemcpyHostToDevice, ctx->stream));
        if (!ocols.empty()) {
            k_finish_ondisk_cols<<<cdiv(ocols.size(), 128), 128, 0, ctx->stream>>>(arena.as<uint8_t>(), out->cols.as<DevColumn>(), (const OndiskCol*)(ctx->zcols.as<uint8_t>() + 16),
                                                                                     (uint32_t)ocols.size(), ctx->zcols.as<unsigned long long>());
            launch_check(ctx);
        }
        copier.h2d += ocols.size() * sizeof(OndiskCol);
        plan.zjob.check(ctx);   // synchronises the stream
        unsigned long long cst[2] = {0, 0};
        VL_CUDA(cudaMemcpy(cst, ctx->zcols.p, 16, cudaMemcpyDeviceToHost));
        static const char* what[] = {"", "cannot unmarshal uint64 block type from empty src", "unexpected uint64 block type", "unexpected block length for uint items", "row length does not fit 32 bits"};
        if (cst[0]) throw BadInput(what[std::min<unsigned long long>(cst[0], 4)]);
    }
    VL_CUDA(cudaStreamWaitEvent(ctx->stream, ev_copied, 0));
    if (dbg) { VL_CUDA(cudaStreamSynchronize(ctx->stream)); t_copy = now(); }
    if (nfields) out->note_columns(cols);
    if (headers) finish_batch_layout(ctx, out, plan.rows);   // synchronises the stream => the plan's tables and the staging ring are free again
    else VL_CUDA(cudaStreamSynchronize(ctx->stream));        // the layout tables are there since the header phase
    uint64_t h2d = copier.h2d;
    if (dbg) fprintf(stderr, "[vlscan upload] blocks=%llu arena=%.1f MB h2d=%.1f MB pieces=%zu+%zu pinned=%d: describe %.1f ms, alloc %.1f ms, copy %.1f ms (%.1f GB/s), "
                             "zstd %llu frames / %llu blocks / %llu sequences: enqueue %.1f ms, decode %.1f ms; layout %.1f ms\n", (unsigned long long)nblocks,
                     plan.arena_bytes / 1e6, h2d / 1e6, plan.layout.pieces.size(), plan.zpieces.size(), (int)!copier.staged, 1e3 * (t_desc - t_start), 1e3 * (t_alloc - t_desc), 1e3 * (t_enq - (t_zrun > 0 ? t_zrun : t_h2d)), h2d / 1e9 / std::max(t_copy - t_start, 1e-9),
                     (unsigned long long)plan.zjob.frames(), (unsigned long long)plan.zjob.compressed_blocks(), (unsigned long long)plan.zjob.sequences(), 1e3 * (t_zrun > 0 ? t_zrun - t_h2d : 0), 1e3 * (t_copy - t_enq), 1e3 * (now() - t_copy));
    if (headers) h2d += out->nwords * 12 + nblocks * 12;
    if (headers && values) std::vector<DevColumn>().swap(out->h_cols);   // only a bloom-first upload needs the table again
    if (stats) stats->h2d_bytes += h2d;
}

// ---- the filter-tree interpreter --------------------------------------------------------------------------------------------
namespace {
struct ScanRun {
    vlscan_ctx* ctx; const vlscan_program* prog; const vlscan_batch* batch;
    DevProgram P; BatchView B; std::vector<int> field_slot;   // program field -> batch field slot or -1
    unsigned long long* stats = nullptr;
    size_t regs_used = 0;
    size_t slots_cursor = 0, slots_total = 0;

    ScanRun(vlscan_ctx* ctx, const vlscan_program* prog, const vlscan_batch* batch) : ctx(ctx), prog(prog), batch(batch) {
        P = const_cast<vlscan_program*>(prog)->image(ctx->device, ctx->stream);
        B = batch->view();
        const Program& pr = prog->p;
        field_slot.assign(pr.fields.size(), -1);
        for (size_t f = 0; f < pr.fields.size(); f++) for (uint32_t s = 0; s < batch->nfields; s++) if (batch->field_names[s] == pr.fields[f]) field_slot[f] = (int)s;
        for (auto& nd : pr.nodes) slots_total += nd.prepass_count;
    }

    uint64_t* new_reg() {
        if (regs_used == ctx->regs.size()) ctx->regs.emplace_back();
        DevBuf& r = ctx->regs[regs_used++];
        r.ensure(std::max<size_t>(B.nwords * 8, 16));
        return r.as<uint64_t>();
    }
    void free_reg() { regs_used--; }
    void copy_reg(uint64_t* dst, const uint64_t* src) { if (B.nwords) VL_CUDA(cudaMemcpyAsync(dst, src, B.nwords * 8, cudaMemcpyDeviceToDevice, ctx->stream)); }
    void andnot(uint64_t* a, const uint64_t* b) { if (!B.nwords) return; k_andnot<<<cdiv(B.nwords, 256), 256, 0, ctx->stream>>>(a, b, B.nwords); launch_check(ctx); }
    void prepass(const PNode& nd, uint64_t* reg) {
        if (nd.prepass_count == 0) return;
        std::vector<int> slots(nd.prepass_count);
        for (int e = 0; e < nd.prepass_count; e++) slots[e] = field_slot[prog->p.prepass[nd.prepass_begin + e].field];
        // slots live in a small device array; successive pre-passes use disjoint regions of it
        size_t off = slots_cursor; slots_cursor += slots.size();
        ctx->slots.ensure(std::max<size_t>(slots_total * 4, 16));
        VL_CUDA(cudaMemcpyAsync(ctx->slots.as<int>() + off, slots.data(), slots.size() * 4, cudaMemcpyHostToDevice, ctx->stream));
        k_prepass<<<cdiv((uint64_t)B.nblocks * 32, 128), 128, 0, ctx->stream>>>(P, B, (uint32_t)nd.prepass_begin, (uint32_t)nd.prepass_count, ctx->slots.as<int>() + off,
                                                                             nd.kind == F_OR, reg, stats);
        launch_check(ctx);
    }

    void leaf(int leaf_idx, uint64_t* reg) {
        const DevLeaf& L = prog->p.leaves[leaf_idx];
        if (L.kind == F_NOOP) return;
        int slot = L.field >= 0 ? field_slot[L.field] : -1;
        uint8_t* action = ctx->action.as<uint8_t>(); uint64_t* payload = ctx->payload.as<uint64_t>(); uint64_t* leaf_bm = ctx->leaf_bm.as<uint64_t>();
        uint32_t* lens_blocks = ctx->lens_blocks.as<uint32_t>(); uint32_t* row_blocks = ctx->row_blocks.as<uint32_t>(); uint32_t* wc = ctx->work_count.as<uint32_t>();
        uint32_t* tb = ctx->tile_block.as<uint32_t>(); uint32_t* to = ctx->tile_off.as<uint32_t>();
        VL_CUDA(cudaMemsetAsync(wc, 0, WC_COUNT * 4, ctx->stream));
        if (L.kind == F_EQ_FIELD || L.kind == F_LE_FIELD) {   // two columns, row by row (filter_eq_field.go, filter_le_field.go)
            const int slot_b = field_slot[L.field2];
            uint32_t* lens_b = tb;   // the tile table is idle for this leaf: it holds the second lens work list
            k_plan_pair<<<cdiv((uint64_t)B.nblocks * 32, 256), 256, 0, ctx->stream>>>(P, B, (uint32_t)leaf_idx, slot, slot_b, reg, action, payload, lens_blocks, lens_b, row_blocks, wc, stats);
            launch_check(ctx);
            if (B.nwords) {
                const int persistent = ctx->sm_count * 8;
                const uint32_t *ro_a = nullptr, *ro_b = nullptr;
                for (int side = 0; side < 2; side++) {
                    const int sl = side ? slot_b : slot;
                    if (sl < 0) continue;
                    uint8_t* ready = ctx->ready[sl].as<uint8_t>();
                    if (!ctx->ready_cleared[sl]) { VL_CUDA(cudaMemsetAsync(ready, 0, B.nblocks, ctx->stream)); ctx->ready_cleared[sl] = 1; }
                    k_lens_offsets<<<persistent, 256, 0, ctx->stream>>>(B, sl, side ? lens_b : lens_blocks, wc, ctx->row_off8[sl].as<uint32_t>(), ready, stats, side ? WC_LENS2 : WC_LENS); launch_check(ctx);
                    (side ? ro_b : ro_a) = ctx->row_off8[sl].as<uint32_t>();
                }
                k_row_pair<<<persistent, 256, 0, ctx->stream>>>(P, B, (uint32_t)leaf_idx, slot, slot_b, row_blocks, wc, payload, reg, ro_a, ro_b, leaf_bm, stats); launch_check(ctx);
                k_apply_leaf<<<cdiv(B.nwords, 256), 256, 0, ctx->stream>>>(B, action, leaf_bm, reg); launch_check(ctx);
            }
            return;
        }
        // bm.isZero() per block, header dispatch + leaf bloom probe -> per-block action, and the work lists of the kernels below
        k_plan_leaf<<<cdiv(B.nblocks, VL_PLAN_WARPS), VL_PLAN_WARPS * 32, 0, ctx->stream>>>(P, B, (uint32_t)leaf_idx, slot, reg, action, payload, lens_blocks, row_blocks, tb, to, wc, stats);
        launch_check(ctx);
        if (slot >= 0 && B.nwords) {
            uint32_t* ro = ctx->row_off8[slot].as<uint32_t>(); uint8_t* ready = ctx->ready[slot].as<uint8_t>();
            if (!ctx->ready_cleared[slot]) { VL_CUDA(cudaMemsetAsync(ready, 0, B.nblocks, ctx->stream)); ctx->ready_cleared[slot] = 1; }
            const int persistent = ctx->sm_count * 8;
            // which kernels can have work is known from the value types this field takes in the batch (header dispatch is per block,
            // on the device, but a field that is never a plain string column cannot produce ACT_SCAN, etc.)
            const uint32_t vts = batch->slot_vt_mask.empty() ? ~0u : batch->slot_vt_mask[slot];
            const bool has_string = vts >> VT_STRING & 1, has_dict = vts >> VT_DICT & 1;
            const bool has_numeric = (vts & ~((1u << VT_STRING) | (1u << VT_DICT))) != 0;
            const bool may_scan = L.str_strategy == STR_SCAN && has_string;
            const bool may_row = (has_string && L.str_strategy != STR_ALL) || has_numeric;   // also the fallback of scan leaves for blocks with short rows (k_plan_leaf)
            if (may_scan || may_row) { k_lens_offsets<<<persistent, 256, 0, ctx->stream>>>(B, slot, lens_blocks, wc, ro, ready, stats); launch_check(ctx); }
            // row-agnostic substring scan
            if (may_scan) {
                VL_CUDA(cudaMemsetAsync(leaf_bm, 0, B.nwords * 8, ctx->stream));
                ScanParams sp; memset(&sp, 0, sizeof sp);
                sp.mode = L.scan_mode; sp.needle_off = L.scan_needle_off; sp.needle_len = L.scan_needle_len; sp.starts_tok = L.starts_tok; sp.ends_tok = L.ends_tok; sp.regex = L.regex;
                const bool masked = fill_scan_patterns(prog->p.blob.data() + L.scan_needle_off, L.scan_needle_len, sp.pat, sp.msk, sp.delta, sp.nd16);
                if (L.scan_mode == SCAN_CONTAINS || L.scan_mode >= SCAN_RX_DOTPLUS) { sp.starts_tok = sp.ends_tok = 0; }
                auto& evp = next_scan_events();
                VL_CUDA(cudaEventRecord(evp.first, ctx->stream));
                // persistent CTAs: exactly the resident set (SMs x resident CTAs per SM), each striding over the tile table
                if (masked) k_substr_scan<true><<<ctx->sm_count * ctx->scan_occ[1], VL_SCAN_THREADS, 0, ctx->stream>>>(P, B, slot, sp, tb, to, wc, ro, leaf_bm);
                else k_substr_scan<false><<<ctx->sm_count * ctx->scan_occ[0], VL_SCAN_THREADS, 0, ctx->stream>>>(P, B, slot, sp, tb, to, wc, ro, leaf_bm);
                launch_check(ctx);
                VL_CUDA(cudaEventRecord(evp.second, ctx->stream));
            }
            // per-row matcher (string exact / in / general regexp; numeric columns through text); persistent grid over the ACT_ROW work list
            if (may_row) { k_row_match<<<ctx->sm_count * ctx->row_occ, 256, 0, ctx->stream>>>(P, B, (uint32_t)leaf_idx, slot, row_blocks, wc, action, payload, reg, ro, leaf_bm); launch_check(ctx); }
            if (has_dict || has_numeric) { k_word_match<<<cdiv(B.nwords, 128), 128, 0, ctx->stream>>>(P, B, (uint32_t)leaf_idx, slot, action, payload, reg, leaf_bm, stats); launch_check(ctx); }
        }
        if (L.kind == F_TIME && B.nwords) {   // blocks the range only partly covers: decode their timestamps, compare per row
            ctx->ts_vals.ensure(B.nwords * 64 * 8);
            k_time_match<<<ctx->sm_count * 4, 256, 0, ctx->stream>>>(B, (long long)L.aux0, (long long)L.aux1, row_blocks, wc, ctx->ts_vals.as<unsigned long long>(), leaf_bm, stats);
            launch_check(ctx);
        }
        if (B.nwords) { k_apply_leaf<<<cdiv(B.nwords, 256), 256, 0, ctx->stream>>>(B, action, leaf_bm, reg); launch_check(ctx); }
    }
    std::pair<cudaEvent_t, cudaEvent_t>& next_scan_events() {
        if (ctx->scan_events_used == ctx->scan_events.size()) { cudaEvent_t a, b; VL_CUDA(cudaEventCreate(&a)); VL_CUDA(cudaEventCreate(&b)); ctx->scan_events.emplace_back(a, b); }
        return ctx->scan_events[ctx->scan_events_used++];
    }
    // ---- probe pass of a bloom-first upload: which (block, column) values can the program reach? ------------------------------------------
    // `reg` only says which blocks are still alive: the AND / OR bloom pre-passes of a leaf's ancestors zero the blocks they rule out
    // (exactly what they do to the bitmaps of the real scan); leaves do not touch it.  The real scan hands a leaf a subset of these rows, so
    // the blocks whose values it reads are a subset of the blocks marked here.
    void probe_leaf(int leaf_idx, const uint64_t* reg, uint8_t* need) {
        const DevLeaf& L = prog->p.leaves[leaf_idx];
        if (L.kind == F_NOOP || L.kind == F_TIME) return;   // timestamps always travel with the block
        const int slot = L.field >= 0 ? field_slot[L.field] : -1;
        if (L.kind == F_EQ_FIELD || L.kind == F_LE_FIELD) {
            k_plan_pair<<<cdiv((uint64_t)B.nblocks * 32, 256), 256, 0, ctx->stream>>>(P, B, (uint32_t)leaf_idx, slot, field_slot[L.field2], reg, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, stats, need);
        } else {
            if (slot < 0) return;   // a field the batch does not have: nothing to stage
            k_plan_leaf<<<cdiv(B.nblocks, VL_PLAN_WARPS), VL_PLAN_WARPS * 32, 0, ctx->stream>>>(P, B, (uint32_t)leaf_idx, slot, reg, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, stats, need);
        }
        launch_check(ctx);
    }
    void probe_node(int id, uint64_t* reg, uint8_t* need) {
        const PNode& nd = prog->p.nodes[id];
        switch (nd.kind) {
        case F_NOOP: break;
        case F_AND: case F_OR: {
            uint64_t* r = reg;
            if (nd.prepass_count) { r = new_reg(); copy_reg(r, reg); prepass(nd, r); }
            for (int k : nd.kids) probe_node(k, r, need);
            if (nd.prepass_count) free_reg();
            break;
        }
        case F_NOT: probe_node(nd.kids[0], reg, need); break;
        default: probe_leaf(nd.leaf, reg, need);
        }
    }
    // applyToBlockSearch of the combinators: filter_and.go:58-74, filter_or.go:55-78, filter_not.go:38-46
    void node(int id, uint64_t* reg) {
        const PNode& nd = prog->p.nodes[id];
        switch (nd.kind) {
        case F_NOOP: break;
        case F_AND: prepass(nd, reg); for (int k : nd.kids) node(k, reg); break;
        case F_OR: {
            prepass(nd, reg);
            uint64_t* res = new_reg(); uint64_t* tmp = new_reg();
            copy_reg(res, reg);
            for (int k : nd.kids) { copy_reg(tmp, res); node(k, tmp); andnot(res, tmp); }
            andnot(reg, res);
            free_reg(); free_reg();
            break;
        }
        case F_NOT: { uint64_t* tmp = new_reg(); copy_reg(tmp, reg); node(nd.kids[0], tmp); andnot(reg, tmp); free_reg(); break; }
        default: leaf(nd.leaf, reg);
        }
    }
};
}  // namespace

static void read_stats(vlscan_ctx* ctx, vlscan_stats* st, bool check_error) {
    unsigned long long h[ST_COUNT];
    VL_CUDA(cudaMemcpyAsync(h, ctx->stats.p, sizeof h, cudaMemcpyDeviceToHost, ctx->stream));
    VL_CUDA(cudaStreamSynchronize(ctx->stream));
    if (check_error && h[ST_ERROR]) {
        static const char* const msg[] = {"", "cannot unmarshal strings: row lengths do not add up to the data length", "too big index for dict value",
                                          "unexpected length for binary representation of a number", "phrase/prefix/regexp over a float64 column needs float->string formatting, which the GPU engine does not implement",
                                          "unexpected uint64 block type", "the filter needs the timestamps of a block that was handed over without them", "cannot unmarshal timestamps",
                                          "internal: a filter reached the values of a column that the bloom-first probe pass had left on the host"};
        throw BadInput(msg[std::min<unsigned long long>(h[ST_ERROR], 8)]);
    }
    if (!st) return;
    st->values_bytes += h[ST_VALUES_BYTES]; st->bloom_probe_bytes += h[ST_BLOOM_BYTES]; st->columns_read += h[ST_COLUMNS_READ];
    st->bitmap_bytes += h[ST_BITMAP_BYTES]; st->rows_matched += h[ST_ROWS_MATCHED]; st->blocks_matched += h[ST_BLOCKS_MATCHED];
    st->scan_kernel_bytes += h[ST_SCAN_BYTES];
    float ms = 0;
    VL_CUDA(cudaEventElapsedTime(&ms, ctx->ev_begin, ctx->ev_end)); st->gpu_ms += ms;
    for (size_t i = 0; i < ctx->scan_events_used; i++) { VL_CUDA(cudaEventElapsedTime(&ms, ctx->scan_events[i].first, ctx->scan_events[i].second)); st->scan_kernel_ms += ms; }
}

static void do_scan(vlscan_ctx* ctx, const vlscan_program* prog, const vlscan_batch* batch, vlscan_stats* stats) {
    VL_CUDA(cudaSetDevice(ctx->device));
    if (batch->device != ctx->device) throw BadInput("batch lives on another device than the ctx");
    ScanRun run(ctx, prog, batch);
    const Program& pr = prog->p;
    uint64_t nb = std::max<uint64_t>(batch->nblocks, 1), nw = std::max<uint64_t>(batch->nwords, 1);
    ctx->action.ensure(nb); ctx->payload.ensure(nb * 8); ctx->leaf_bm.ensure(nw * 8);
    ctx->lens_blocks.ensure(nb * 4); ctx->row_blocks.ensure(nb * 4); ctx->work_count.ensure(WC_COUNT * 4);
    {   // upper bound of 64 KiB tiles of any single column: every payload byte belongs to one column, plus one partial tile per block
        uint64_t max_tiles = batch->arena_bytes / VL_TILE_BYTES + nb + 16;
        ctx->tile_block.ensure(max_tiles * 4); ctx->tile_off.ensure(max_tiles * 4);
    }
    ctx->stats.ensure(ST_COUNT * 8); ctx->totals.ensure(32); ctx->counts.ensure(nb * 4);
    if (ctx->row_off8.size() < batch->nfields) { ctx->row_off8.resize(batch->nfields); ctx->ready.resize(batch->nfields); }
    ctx->ready_cleared.assign(batch->nfields, 0);
    for (uint32_t s = 0; s < batch->nfields; s++) { ctx->row_off8[s].ensure(nw * 32); ctx->ready[s].ensure(nb); }
    uint64_t launches0 = ctx->launches;
    ctx->scan_events_used = 0;
    run.stats = ctx->stats.as<unsigned long long>();
    VL_CUDA(cudaEventRecord(ctx->ev_begin, ctx->stream));
    VL_CUDA(cudaMemsetAsync(ctx->stats.p, 0, ST_COUNT * 8, ctx->stream));
    VL_CUDA(cudaMemsetAsync(ctx->totals.p, 0, 32, ctx->stream));
    // bm.init(rows); bm.setBits()   (block_search.go:213-214)
    uint64_t* reg = run.new_reg();
    run.copy_reg(reg, batch->init_bitmap.as<uint64_t>());
    if (batch->nblocks) {
        run.node(pr.root, reg);
        k_finalize<<<cdiv(batch->nblocks, 8), 256, 0, ctx->stream>>>(run.B, reg, ctx->counts.as<uint32_t>(), run.stats, ctx->totals.as<unsigned long long>());
        launch_check(ctx);
    }
    VL_CUDA(cudaEventRecord(ctx->ev_end, ctx->stream));
    ctx->last_batch = batch; ctx->has_result = true; ctx->last_launches = ctx->launches - launches0;
    ctx->last_nblocks = batch->nblocks; ctx->last_nwords = batch->nwords; ctx->last_rows = batch->rows;
    if (stats) {
        read_stats(ctx, stats, true);
        stats->blocks += batch->nblocks; stats->rows += batch->rows; stats->gpu_launches += ctx->launches - launches0;
    }
}

// The probe pass between the two phases of a bloom-first upload: runs the program's bloom pre-passes, header dispatch and leaf bloom probes on a
// batch whose values are still on the host and returns need[block * nfields + field] = 1 for every values column some filter can reach.
static void do_probe(vlscan_ctx* ctx, const vlscan_program* prog, const vlscan_batch* batch, std::vector<uint8_t>& need) {
    VL_CUDA(cudaSetDevice(ctx->device));
    ScanRun run(ctx, prog, batch);
    const size_t cells = (size_t)batch->nblocks * batch->nfields;
    need.assign(cells, 0);
    if (!cells || !batch->nwords) return;
    ctx->need.ensure(std::max<size_t>(cells, 16)); ctx->stats.ensure(ST_COUNT * 8);
    VL_CUDA(cudaMemsetAsync(ctx->need.p, 0, cells, ctx->stream));
    VL_CUDA(cudaMemsetAsync(ctx->stats.p, 0, ST_COUNT * 8, ctx->stream));
    run.stats = ctx->stats.as<unsigned long long>();
    uint64_t* reg = run.new_reg();
    run.copy_reg(reg, batch->init_bitmap.as<uint64_t>());
    run.probe_node(prog->p.root, reg, ctx->need.as<uint8_t>());
    VL_CUDA(cudaMemcpyAsync(need.data(), ctx->need.p, cells, cudaMemcpyDeviceToHost, ctx->stream));
    VL_CUDA(cudaStreamSynchronize(ctx->stream));
}

// ---- C ABI -------------------------------------------------------------------------------------------------------------------
extern "C" {

int vlscan_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
    return n;
}

vlscan_ctx* vlscan_ctx_create(int device) {
    vlscan_ctx* ctx = new vlscan_ctx();
    int rc = guarded(nullptr, [&] {
        int n = vlscan_device_count();
        if (n <= 0) throw CudaFail("no CUDA device is available: libvlscan has no CPU fallback", 100);
        ctx->device = ((device % n) + n) % n;
        VL_CUDA(cudaSetDevice(ctx->device));
        VL_CUDA(cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking));
        VL_CUDA(cudaStreamCreateWithFlags(&ctx->copy_stream, cudaStreamNonBlocking));
        VL_CUDA(cudaEventCreate(&ctx->ev_begin)); VL_CUDA(cudaEventCreate(&ctx->ev_end));
        cudaDeviceProp prop; VL_CUDA(cudaGetDeviceProperties(&prop, ctx->device)); ctx->sm_count = prop.multiProcessorCount;
        // resident CTAs per SM of the two scan instantiations on THIS device (the persistent grids are sized by it)
        VL_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&ctx->scan_occ[0], k_substr_scan<false>, VL_SCAN_THREADS, 0));
        VL_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&ctx->scan_occ[1], k_substr_scan<true>, VL_SCAN_THREADS, 0));
        for (int& o : ctx->scan_occ) o = std::max(o, 1);
        VL_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&ctx->row_occ, k_row_match, 256, 0));
        ctx->row_occ = std::max(ctx->row_occ, 1);
    });
    if (rc) { delete ctx; return nullptr; }
    return ctx;
}
void vlscan_ctx_free(vlscan_ctx* ctx) {
    if (!ctx) return;
    cudaSetDevice(ctx->device);
    if (ctx->copy_stream) cudaStreamSynchronize(ctx->copy_stream);
    if (ctx->stream) cudaStreamSynchronize(ctx->stream);
    for (DevBuf* b : {&ctx->action, &ctx->payload, &ctx->leaf_bm, &ctx->lens_blocks, &ctx->row_blocks, &ctx->work_count, &ctx->stats, &ctx->totals, &ctx->counts, &ctx->slots, &ctx->hit_offs, &ctx->hits, &ctx->tile_block, &ctx->tile_off}) b->release();
    for (auto& r : ctx->regs) r.release();
    for (auto& r : ctx->row_off8) r.release();
    for (auto& r : ctx->ready) r.release();
    ctx->zsrc.release(); ctx->zcols.release(); ctx->ztest.release(); ctx->ts_vals.release();
    for (DevBuf* b : {&ctx->hit_block, &ctx->glens, &ctx->goffs, &ctx->gtiles, &ctx->gout, &ctx->gstat}) b->release();
    zstd_dev_free(ctx->zdev);
    delete ctx->pool;
    if (ctx->pinned) cudaFreeHost(ctx->pinned);
    delete ctx->recycle;
    for (auto& e : ctx->scan_events) { cudaEventDestroy(e.first); cudaEventDestroy(e.second); }
    if (ctx->ev_begin) cudaEventDestroy(ctx->ev_begin);
    if (ctx->ev_end) cudaEventDestroy(ctx->ev_end);
    if (ctx->copy_stream) cudaStreamDestroy(ctx->copy_stream);
    if (ctx->stream) cudaStreamDestroy(ctx->stream);
    delete ctx;
}
const char* vlscan_last_error(const vlscan_ctx* ctx) { return ctx ? ctx->err.c_str() : g_thread_err.c_str(); }
void* vlscan_ctx_stream(const vlscan_ctx* ctx) { return (void*)ctx->stream; }
int vlscan_ctx_sync(vlscan_ctx* ctx) { return guarded(ctx, [&] { VL_CUDA(cudaSetDevice(ctx->device)); VL_CUDA(cudaStreamSynchronize(ctx->stream)); }); }

int vlscan_program_create(const void* tree, size_t tree_len, vlscan_program** out) {
    *out = nullptr;
    auto* pg = new vlscan_program();
    int rc = guarded(nullptr, [&] { ProgramBuilder(tree, tree_len, pg->p).build(); });
    if (rc) { delete pg; return rc; }
    *out = pg;
    return 0;
}
void vlscan_program_free(vlscan_program* prog) { delete prog; }
uint32_t vlscan_program_nfields(const vlscan_program* prog) { return (uint32_t)prog->p.fields.size(); }
const char* vlscan_program_field(const vlscan_program* prog, uint32_t i, size_t* len) { if (i >= prog->p.fields.size()) { *len = 0; return nullptr; } *len = prog->p.fields[i].size(); return prog->p.fields[i].data(); }
int64_t vlscan_program_leaf_tokens(const vlscan_program* prog, uint32_t leaf, char* buf, size_t cap) {
    if (leaf >= prog->p.leaf_tokens.size()) return -1;
    std::string s; for (size_t i = 0; i < prog->p.leaf_tokens[leaf].size(); i++) { if (i) s.push_back('\n'); s += prog->p.leaf_tokens[leaf][i]; }
    if (s.size() > cap) return -1;
    memcpy(buf, s.data(), s.size());
    return (int64_t)s.size();
}

int vlscan_eval_predicate(int kind, const void* value, size_t value_len, const void* arg1, size_t arg1_len, const void* arg2, size_t arg2_len, uint64_t aux0, uint64_t aux1) {
    if (value_len > 0xFFFFFFFFull || arg1_len > 0xFFFFFFFFull || arg2_len > 0xFFFFFFFFull) return -1;
    const uint8_t* v = (const uint8_t*)value; const uint32_t vn = (uint32_t)value_len;
    const uint8_t* a = (const uint8_t*)arg1; const uint32_t an = (uint32_t)arg1_len;
    switch (kind) {   // predicates of the kinds that are not wired into the row kernels yet (vl_anycase.cuh)
    case F_REGEXP: {   // arg1 = the expression: compiled like a regexp leaf, matched by the host mirror of the device automaton (const / dict values take this path)
        try { return vl::compile_regex(std::string((const char*)a, an)).match(v, vn) ? 1 : 0; } catch (const vl::RxError& e) { vl::set_thread_error(e.what()); return -2; }
    }
    case 14: return vl::any_case_match(v, vn, a, an, false) ? 1 : 0;
    case 15: return vl::any_case_match(v, vn, a, an, true) ? 1 : 0;
    case 16: return vl::match_sequence(v, vn, vl::PhraseList{a, an}) ? 1 : 0;
    case 17: return vl::match_all_phrases(v, vn, vl::PhraseList{a, an}) ? 1 : 0;
    case 18: return vl::match_any_phrase(v, vn, vl::PhraseList{a, an}) ? 1 : 0;
    }
    if (kind < F_EXACT_PREFIX || kind > F_IPV4_RANGE) return -1;
    return vl::range_predicate(kind, (const uint8_t*)value, (uint32_t)value_len, (const uint8_t*)arg1, (uint32_t)arg1_len, (const uint8_t*)arg2, (uint32_t)arg2_len, aux0, aux1) ? 1 : 0;
}

int64_t vlscan_program_prepass_tokens(const vlscan_program* prog, char* buf, size_t cap) {
    const Program& P = prog->p;
    std::string s;
    for (const PNode& nd : P.nodes) {   // nodes are numbered in pre-order
        if (nd.kind != F_AND && nd.kind != F_OR) continue;
        s += nd.kind == F_AND ? "A" : "O";
        for (int k = 0; k < nd.prepass_count; k++) {
            const DevPrepass& pp = P.prepass[(size_t)nd.prepass_begin + k];
            s += "\t" + P.fields[pp.field];
            const uint32_t* offs = (const uint32_t*)(P.blob.data() + pp.tok_offs_off);
            for (uint32_t t = 0; t < pp.ntokens; t++) { s += "\x1f"; s.append((const char*)P.blob.data() + pp.tok_blob_off + offs[t], offs[t + 1] - offs[t]); }
        }
        s += "\n";
    }
    if (s.size() > cap) return -1;
    memcpy(buf, s.data(), s.size());
    return (int64_t)s.size();
}

int64_t vlscan_program_in_hashes(const vlscan_program* prog, uint32_t leaf, uint64_t* out, size_t cap) {
    const Program& P = prog->p;
    if (leaf >= P.leaves.size() || P.leaves[leaf].kind != F_IN) return -1;
    const DevLeaf& L = P.leaves[leaf];
    std::vector<uint64_t> v;
    v.push_back(L.nhashes); v.insert(v.end(), P.u64s.begin() + L.hashes_off, P.u64s.begin() + L.hashes_off + L.nhashes);
    if (L.in_skip_sets) v.push_back(UINT64_MAX);   // more than maxTokenSetsToInit value sets: none is kept
    else {
        v.push_back(L.in_nsets);
        for (uint32_t k = 0; k < L.in_nsets; k++) {
            const uint32_t off = P.u32s[L.in_sets_off + 2 * k], n = P.u32s[L.in_sets_off + 2 * k + 1];
            v.push_back(n); v.insert(v.end(), P.u64s.begin() + off, P.u64s.begin() + off + n);
        }
    }
    if (v.size() > cap) return -1;
    memcpy(out, v.data(), v.size() * 8);
    return (int64_t)v.size();
}

int64_t vlscan_program_in_typed(const vlscan_program* prog, uint32_t leaf, int value_type, uint64_t* out, size_t cap) {
    const Program& P = prog->p;
    if (leaf >= P.leaves.size() || P.leaves[leaf].kind != F_IN || value_type < VT_UINT8 || value_type >= VT_MAX) return -1;
    const DevLeaf& L = P.leaves[leaf];
    const uint32_t n = L.in_typed_cnt[value_type];
    if (n > cap) return -1;
    if (n) memcpy(out, P.u64s.data() + L.in_typed_off[value_type], (size_t)n * 8);
    return (int64_t)n;
}

int vlscan_parse_typed(int value_type, const void* s, size_t len, uint64_t* out) {
    const std::string v((const char*)s, len);
    uint64_t u = 0; int64_t i = 0; double f = 0; uint32_t ip = 0;
    switch (value_type) {
    case VT_UINT8: case VT_UINT16: case VT_UINT32: case VT_UINT64: if (!vl::parse_u64(v, &u)) return 0; *out = u; return 1;
    case VT_INT64: if (!vl::parse_i64(v, &i)) return 0; *out = (uint64_t)i; return 1;
    case VT_FLOAT64: if (!vl::parse_f64_exact(v, &f)) return 0; memcpy(out, &f, 8); return 1;
    case VT_IPV4: if (!vl::parse_ipv4(v, &ip)) return 0; *out = ip; return 1;
    case VT_ISO8601: if (!vl::parse_iso8601(v, &i)) return 0; *out = (uint64_t)i; return 1;
    }
    return -1;
}

double vlscan_parse_math_number(const void* s, size_t len) {
    if (len > 0xFFFFFFFFull) return NAN;
    return vl::mn::parse_math_number((const uint8_t*)s, (uint32_t)len);
}

int vlscan_format_float64(uint64_t ieee_bits, char* buf, size_t cap) {
    uint8_t tmp[VL_FMT_F64_MAX];
    int n = vl::fmt_f64(tmp, ieee_bits);
    if ((size_t)n > cap) return -1;
    memcpy(buf, tmp, (size_t)n);
    return n;
}

int vlscan_batch_upload(vlscan_ctx* ctx, const char* const* field_names, const size_t* field_name_lens, uint32_t nfields, const vlscan_block* blocks,
                        uint64_t nblocks, vlscan_batch** out, vlscan_stats* stats) {
    *out = nullptr;
    auto* b = new vlscan_batch();
    int rc = guarded(ctx, [&] { do_upload(ctx, field_names, field_name_lens, nfields, blocks, nblocks, b, stats); });
    if (rc) { cudaStreamSynchronize(ctx->copy_stream); cudaStreamSynchronize(ctx->stream); }   // nothing may still read the caller's buffers
    if (rc) { delete b; return rc; }
    *out = b;
    return 0;
}
void vlscan_batch_free(vlscan_batch* batch) { delete batch; }
uint64_t vlscan_batch_nblocks(const vlscan_batch* b) { return b->nblocks; }
uint64_t vlscan_batch_rows(const vlscan_batch* b) { return b->rows; }
uint64_t vlscan_batch_words(const vlscan_batch* b) { return b->nwords; }
uint64_t vlscan_batch_device_bytes(const vlscan_batch* b) { return b->device_bytes(); }

int vlscan_batch_download(vlscan_ctx* ctx, const vlscan_batch* batch, vlscan_host_blocks** out) {
    *out = nullptr;
    auto* hb = new vlscan_host_blocks();
    int rc = guarded(ctx, [&] {
        VL_CUDA(cudaSetDevice(ctx->device));
        if (batch->split_hdr) throw BadInput("a batch staged bloom-first cannot be downloaded");
        hb->bytes = batch->arena_bytes;
        VL_CUDA(cudaMallocHost(&hb->pinned, std::max<size_t>(hb->bytes, 16)));
        std::vector<DevColumn> cols((size_t)batch->nblocks * batch->nfields);
        VL_CUDA(cudaMemcpyAsync(hb->pinned, batch->arena.p, hb->bytes, cudaMemcpyDeviceToHost, ctx->stream));
        if (!cols.empty()) VL_CUDA(cudaMemcpyAsync(cols.data(), batch->cols.p, cols.size() * sizeof(DevColumn), cudaMemcpyDeviceToHost, ctx->stream));
        VL_CUDA(cudaStreamSynchronize(ctx->stream));
        hb->fields = batch->field_names;
        const uint8_t* base = (const uint8_t*)hb->pinned;
        hb->blocks.resize(batch->nblocks);
        hb->cols.reserve(cols.size());
        // the lens type byte is not stored in the arena: rebuild "type + items" views in a side buffer kept alive by dict_offsets storage
        std::vector<size_t> first(batch->nblocks + 1, 0);
        for (uint64_t b = 0; b < batch->nblocks; b++) {
            first[b] = hb->cols.size();
            for (uint32_t f = 0; f < batch->nfields; f++) {
                const DevColumn& d = cols[(size_t)b * batch->nfields + f];
                if (d.kind == COL_MISSING) continue;
                vlscan_column c; memset(&c, 0, sizeof c);
                c.field = f;
                if (d.kind == COL_CONST) { c.kind = VLSCAN_COL_CONST; c.const_value = base + d.meta_off; c.const_len = d.meta_len; hb->cols.push_back(c); continue; }
                c.kind = VLSCAN_COL_VALUES; c.value_type = d.vt; c.stage = VLSCAN_STAGE_DECODED; c.dict_len = d.dict_len; c.min_value = d.min_value; c.max_value = d.max_value;
                uint64_t items = d.lens_type < 4 ? ((uint64_t)batch->h_rows[b] << d.lens_type) : (1ull << (d.lens_type - 4));
                // lens items are preceded in the arena by alignment slack; the type byte is materialised in the byte right before them
                uint8_t* tb = (uint8_t*)hb->pinned + d.lens_off - 1;
                *tb = d.lens_type;
                c.lens_items = tb; c.lens_items_len = items + 1;
                c.data = base + d.data_off; c.data_len = d.data_len;
                c.bloom = base + d.bloom_off; c.bloom_len = (uint64_t)d.bloom_words * 8;
                if (d.vt == VT_DICT) { c.dict_offsets = (const uint32_t*)(base + d.meta_off); c.dict_blob = base + d.meta_off + 4 * (d.dict_len + 1); }
                hb->cols.push_back(c);
            }
        }
        first[batch->nblocks] = hb->cols.size();
        for (uint64_t b = 0; b < batch->nblocks; b++) { hb->blocks[b].rows = batch->h_rows[b]; hb->blocks[b].ncols = (uint32_t)(first[b + 1] - first[b]); hb->blocks[b].cols = hb->cols.data() + first[b]; }
    });
    if (rc) { if (hb->pinned) cudaFreeHost(hb->pinned); delete hb; return rc; }
    *out = hb;
    return 0;
}
// The reference's writer for one values block: marshalBytesBlock(lens items) ++ marshalBytesBlock(data) (encoding.go:16-50, 343-370)
static void marshal_bytes_block(std::vector<uint8_t>& dst, const uint8_t* src, size_t n) {
    if (n < 128) { dst.push_back(0); dst.push_back((uint8_t)n); dst.insert(dst.end(), src, src + n); return; }
    ZstdWriter& z = zstd_writer();
    if (!z.ok) throw BadInput("libzstd.so.1 is not available for compressing values blocks");
    int level = n <= 512 ? 1 : n <= 4096 ? 2 : 3;   // getCompressLevel, encoding.go:362-370
    size_t cap = z.bound(n), old = dst.size();
    dst.push_back(1);
    dst.resize(old + 1 + 10 + cap);
    size_t got = z.compress(dst.data() + old + 11, cap, src, n, level);
    if (z.is_error(got)) throw BadInput("ZSTD_compress failed");
    uint8_t vu[10]; int k = 0; uint64_t v = got; while (v >= 0x80) { vu[k++] = (uint8_t)(v | 0x80); v >>= 7; } vu[k++] = (uint8_t)v;   // MarshalVarUint64
    memcpy(dst.data() + old + 1, vu, k);
    memmove(dst.data() + old + 1 + k, dst.data() + old + 11, got);
    dst.resize(old + 1 + k + got);
}

int vlscan_host_blocks_compress(const vlscan_host_blocks* in, int threads, vlscan_host_blocks** out) {
    *out = nullptr;
    auto* hb = new vlscan_host_blocks();
    int rc = guarded(nullptr, [&] {
        const size_t ncols = in->cols.size();
        std::vector<std::vector<uint8_t>> packed(ncols);
        std::atomic<size_t> next{0}; std::atomic<bool> failed{false}; std::string fail_msg; std::mutex mu;
        auto work = [&] {
            for (;;) {
                size_t i0 = next.fetch_add(64); if (i0 >= ncols || failed) return;
                for (size_t i = i0; i < std::min(ncols, i0 + 64); i++) {
                    const vlscan_column& c = in->cols[i];
                    if (c.kind != VLSCAN_COL_VALUES) continue;
                    try {
                        if (c.stage == VLSCAN_STAGE_ONDISK) packed[i].assign(c.values, c.values + c.values_len);
                        else { marshal_bytes_block(packed[i], c.lens_items, c.lens_items_len); marshal_bytes_block(packed[i], c.data, c.data_len); }
                    } catch (const BadInput& e) { std::lock_guard<std::mutex> g(mu); fail_msg = e.msg; failed = true; return; }
                }
            }
        };
        int nt = threads > 0 ? threads : (int)std::max(1u, std::thread::hardware_concurrency());
        std::vector<std::thread> pool; for (int t = 1; t < nt; t++) pool.emplace_back(work);
        work(); for (auto& t : pool) t.join();
        if (failed) throw BadInput(fail_msg);
        // layout: [copied part: consts, blooms, dict tables, placed as a full upload places them][values blocks, back to back]
        ArenaLayout layout;
        std::vector<DevColumn> at(ncols);
        uint64_t vbytes = 0;
        std::vector<uint64_t> off_v(ncols, 0);
        for (size_t i = 0; i < ncols; i++) {
            const vlscan_column& c = in->cols[i];
            layout.put_headers(c, c.bloom_len, at[i]);
            if (c.kind != VLSCAN_COL_CONST) { off_v[i] = vbytes; vbytes += packed[i].size(); }
        }
        const uint64_t vbase = (layout.cursor + kArenaPad + 63) / 64 * 64;
        hb->bytes = vbase + vbytes + 64;
        VL_CUDA(cudaMallocHost(&hb->pinned, hb->bytes));
        uint8_t* base = (uint8_t*)hb->pinned;
        memset(base, 0, vbase);
        for (const Piece& p : layout.pieces) memcpy(base + p.dst, p.src, p.len);
        hb->fields = in->fields; hb->cols = in->cols; hb->blocks = in->blocks;
        for (size_t i = 0; i < ncols; i++) {
            vlscan_column& c = hb->cols[i];
            if (c.kind == VLSCAN_COL_CONST) { c.const_value = base + at[i].meta_off; continue; }
            c.bloom = base + at[i].bloom_off;
            if (c.value_type == VT_DICT) { c.dict_offsets = (const uint32_t*)(base + at[i].meta_off); c.dict_blob = base + at[i].meta_off + 4 * (c.dict_len + 1); }
            memcpy(base + vbase + off_v[i], packed[i].data(), packed[i].size());
            c.stage = VLSCAN_STAGE_ONDISK; c.values = base + vbase + off_v[i]; c.values_len = packed[i].size();
            c.lens_items = nullptr; c.lens_items_len = 0; c.data = nullptr; c.data_len = 0;
            std::vector<uint8_t>().swap(packed[i]);
        }
        size_t k = 0;
        for (size_t b = 0; b < hb->blocks.size(); b++) { hb->blocks[b].cols = hb->cols.data() + k; k += hb->blocks[b].ncols; }
    });
    if (rc) { if (hb->pinned) cudaFreeHost(hb->pinned); delete hb; return rc; }
    *out = hb;
    return 0;
}

int vlscan_zstd_inspect(const void* bytes_block, size_t len, uint64_t out[5]) {
    return guarded(nullptr, [&] {
        ZstdJob job;
        uint64_t regen = 0; uint32_t id = 0;
        size_t used = job.add_bytes_block((const uint8_t*)bytes_block, len, 512, &regen, &id);
        out[0] = used; out[1] = regen; out[2] = job.blocks(); out[3] = job.compressed_blocks(); out[4] = job.sequences();
    });
}

int vlscan_zstd_walk_digest(const vlscan_block* blocks, uint64_t nblocks, int threads, uint64_t out[12]) {
    return guarded(nullptr, [&] {
        auto now = [] { return std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count(); };
        std::vector<ZValuesBlock> zv;
        collect_values_blocks(blocks, nblocks, zv);
        std::vector<ZValuesInfo> info(zv.size());
        ZstdJob job; size_t bad = SIZE_MAX; std::string msg;
        const double t0 = now();
        if (!zv.empty()) job.add_values_blocks(zv.data(), zv.size(), threads, info.data(), &bad, &msg);
        const double t1 = now();
        if (bad != SIZE_MAX) throw BadInput("values block " + std::to_string(bad) + ": " + msg);
        job.prepare();
        const double t2 = now();
        job.digest(out);
        uint64_t h = 5; for (const ZValuesInfo& x : info) { h = (h ^ x.lens_len) * 0x9E3779B97F4A7C15ull; h = (h ^ x.data_len) * 0x9E3779B97F4A7C15ull; h ^= h >> 29; }
        out[0] ^= h;
        out[4] = job.frames(); out[5] = job.blocks(); out[6] = job.groups(); out[7] = job.compressed_blocks(); out[8] = job.sequences();
        out[9] = (uint64_t)((t1 - t0) * 1e9); out[10] = (uint64_t)((t2 - t1) * 1e9); out[11] = 0;
    });
}

// the device decoder on independent frames given as host pointers (metadata of a part, parity tests)
static void zstd_decompress_frames(vlscan_ctx* ctx, uint32_t nframes, const void* const* frames, const size_t* frame_lens, void* dst, const uint64_t* dst_offsets) {
    {
        VL_CUDA(cudaSetDevice(ctx->device));
        ZstdJob job;
        std::vector<uint8_t> packed(512, 0);
        for (uint32_t i = 0; i < nframes; i++) {
            uint64_t regen = 0; uint32_t id = 0;
            job.add_frame((const uint8_t*)frames[i], frame_lens[i], packed.size(), &regen, &id);
            if (regen != dst_offsets[i + 1] - dst_offsets[i]) throw BadInput("cannot decompress block: frame content size differs from the destination size");
            job.set_dst(id, 16 + dst_offsets[i]);
            packed.insert(packed.end(), (const uint8_t*)frames[i], (const uint8_t*)frames[i] + frame_lens[i]);
        }
        const uint64_t total = nframes ? dst_offsets[nframes] : 0;
        ctx->zsrc.ensure(packed.size() + 512); ctx->ztest.ensure(16 + total + 64);
        VL_CUDA(cudaMemcpyAsync(ctx->zsrc.p, packed.data(), packed.size(), cudaMemcpyHostToDevice, ctx->stream));
        VL_CUDA(cudaMemsetAsync(ctx->ztest.p, 0xA5, 16 + total + 64, ctx->stream));
        job.run(ctx, ctx->zsrc.as<uint8_t>(), ctx->ztest.as<uint8_t>());
        job.check(ctx);
        if (total) VL_CUDA(cudaMemcpy(dst, ctx->ztest.as<uint8_t>() + 16, total, cudaMemcpyDeviceToHost));
    }
}

int vlscan_zstd_decompress(vlscan_ctx* ctx, uint32_t nframes, const void* const* frames, const size_t* frame_lens, void* dst, const uint64_t* dst_offsets) {
    return guarded(ctx, [&] { zstd_decompress_frames(ctx, nframes, frames, frame_lens, dst, dst_offsets); });
}

// ---- part directory reader (vl_part.h) ------------------------------------------------------------------------------------
int vlscan_part_open(vlscan_ctx* ctx, const char* path, vlscan_inflate_fn inflate, void* user, vlscan_part** out) {
    *out = nullptr;
    auto* p = new vlscan_part();
    int rc = guarded(ctx, [&] {
        if (!inflate && !ctx) throw BadInput("vlscan_part_open needs a ctx (device ZSTD decoder) or an inflate callback");
        vl::part::Inflate inf;
        if (inflate) inf = [&](const uint8_t* f, size_t n, uint8_t* dst, size_t dn) { if (inflate(user, f, n, dst, dn) != 0) throw BadInput("the inflate callback failed on a metadata frame of the part"); };
        else inf = [&](const uint8_t* f, size_t n, uint8_t* dst, size_t dn) { const void* fr[1] = {f}; const size_t ln[1] = {n}; const uint64_t offs[2] = {0, dn}; zstd_decompress_frames(ctx, 1, fr, ln, dst, offs); };
        p->r.open(path, inf);
    });
    if (rc) { delete p; return rc; }
    *out = p;
    return 0;
}
void vlscan_part_free(vlscan_part* part) { delete part; }
void vlscan_part_header(const vlscan_part* part, uint64_t out[8]) {
    const vl::part::PartHeader& h = part->r.ph;
    out[0] = h.FormatVersion; out[1] = h.CompressedSizeBytes; out[2] = h.UncompressedSizeBytes; out[3] = h.RowsCount; out[4] = h.BlocksCount;
    out[5] = (uint64_t)h.MinTimestamp; out[6] = (uint64_t)h.MaxTimestamp; out[7] = h.BloomValuesShardsCount;
}
uint64_t vlscan_part_nblocks(const vlscan_part* part) { return part->r.blockHeaders.size(); }
int vlscan_part_block_header(const vlscan_part* part, uint64_t i, uint64_t out[15]) {
    return guarded(nullptr, [&] {
        if (i >= part->r.blockHeaders.size()) throw BadInput("block index outside the part");
        const vl::part::BlockHeader& b = part->r.blockHeaders[i];
        out[0] = b.sid.accountID; out[1] = b.sid.projectID; out[2] = b.sid.hi; out[3] = b.sid.lo; out[4] = b.uncompressedSizeBytes; out[5] = b.rowsCount;
        out[6] = b.tsOffset; out[7] = b.tsSize; out[8] = (uint64_t)b.minTimestamp; out[9] = (uint64_t)b.maxTimestamp; out[10] = b.tsMarshalType;
        out[11] = b.chIndexOffset; out[12] = b.chIndexSize; out[13] = b.chOffset; out[14] = b.chSize;
    });
}
int vlscan_part_timestamps(const vlscan_part* part, uint64_t i, const uint8_t** data, uint64_t* len) {
    return guarded(nullptr, [&] {
        if (i >= part->r.blockHeaders.size()) throw BadInput("block index outside the part");
        const vl::part::BlockHeader& b = part->r.blockHeaders[i];
        if (b.tsSize > vl::part::kMaxTimestampsBlockSize) throw BadInput("timestamps block size is too big");   // getTimestamps block_search.go:490-493
        *data = part->r.timestamps_file().at(b.tsOffset, b.tsSize, "a timestamps block"); *len = b.tsSize;
    });
}
uint32_t vlscan_part_ncolumn_names(const vlscan_part* part) { return (uint32_t)part->r.columnNames.size(); }
const char* vlscan_part_column_name(const vlscan_part* part, uint32_t i, size_t* len) { if (i >= part->r.columnNames.size()) { *len = 0; return nullptr; } const std::string& s = part->r.columnNames[i]; *len = s.size(); return s.data(); }
int vlscan_part_blocks(const vlscan_part* part, const char* const* field_names, const size_t* field_name_lens, uint32_t nfields, uint64_t block_lo, uint64_t block_hi,
                       int64_t min_timestamp, int64_t max_timestamp, vlscan_host_blocks** out) {
    *out = nullptr;
    auto* hb = new vlscan_host_blocks();
    int rc = guarded(nullptr, [&] {
        std::vector<std::string> fields;
        for (uint32_t f = 0; f < nfields; f++) { std::string n(field_names[f], field_name_lens[f]); fields.push_back(n.empty() ? "_msg" : n); }
        for (size_t a = 0; a < fields.size(); a++) for (size_t b = a + 1; b < fields.size(); b++) if (fields[a] == fields[b]) throw BadInput("duplicate field name");
        vl::part::Described d;
        part->r.describe(fields, block_lo, block_hi, min_timestamp, max_timestamp, d);
        hb->fields = std::move(d.fields); hb->cols = std::move(d.cols); hb->blocks = std::move(d.blocks); hb->owned = std::move(d.owned); hb->source = std::move(d.source);
        for (const vlscan_column& c : hb->cols) hb->bytes += c.const_len + c.values_len + c.bloom_len;
    });
    if (rc) { delete hb; return rc; }
    *out = hb;
    return 0;
}
const uint64_t* vlscan_host_blocks_source(const vlscan_host_blocks* hb, uint64_t* n) { *n = hb->source.size(); return hb->source.data(); }

const vlscan_block* vlscan_host_blocks_get(const vlscan_host_blocks* hb, uint64_t* nblocks, uint32_t* nfields) { *nblocks = hb->blocks.size(); *nfields = (uint32_t)hb->fields.size(); return hb->blocks.data(); }
const char* vlscan_host_blocks_field(const vlscan_host_blocks* hb, uint32_t i, size_t* len) { if (i >= hb->fields.size()) { *len = 0; return nullptr; } *len = hb->fields[i].size(); return hb->fields[i].data(); }
uint64_t vlscan_host_blocks_bytes(const vlscan_host_blocks* hb) { return hb->bytes; }
void vlscan_host_blocks_free(vlscan_host_blocks* hb) { if (!hb) return; if (hb->pinned) cudaFreeHost(hb->pinned); delete hb; }

int vlscan_scan_resident(vlscan_ctx* ctx, const vlscan_program* prog, const vlscan_batch* batch, vlscan_stats* stats) {
    return guarded(ctx, [&] { do_scan(ctx, prog, batch, stats); });
}

int vlscan_last_scan_stats(vlscan_ctx* ctx, vlscan_stats* stats) {
    return guarded(ctx, [&] {
        if (!ctx->has_result) throw BadInput("no scan on this ctx yet");
        VL_CUDA(cudaSetDevice(ctx->device));
        read_stats(ctx, stats, true);
        stats->blocks += ctx->last_nblocks; stats->rows += ctx->last_rows; stats->gpu_launches += ctx->last_launches;
    });
}

int vlscan_fetch_results(vlscan_ctx* ctx, uint64_t* out_bitmap_words, uint32_t* out_match_counts, vlscan_stats* stats) {
    return guarded(ctx, [&] {
        if (!ctx->has_result) throw BadInput("no scan result to fetch on this ctx");
        VL_CUDA(cudaSetDevice(ctx->device));
        uint64_t d2h = 0;   // bitmaps and counts live in ctx scratch: no access to the batch here
        if (out_bitmap_words && ctx->last_nwords) { VL_CUDA(cudaMemcpyAsync(out_bitmap_words, ctx->regs[0].p, ctx->last_nwords * 8, cudaMemcpyDeviceToHost, ctx->stream)); d2h += ctx->last_nwords * 8; }
        if (out_match_counts && ctx->last_nblocks) { VL_CUDA(cudaMemcpyAsync(out_match_counts, ctx->counts.p, ctx->last_nblocks * 4, cudaMemcpyDeviceToHost, ctx->stream)); d2h += ctx->last_nblocks * 4; }
        read_stats(ctx, nullptr, true);
        if (stats) stats->d2h_bytes += d2h;
    });
}

int vlscan_fetch_hits(vlscan_ctx* ctx, uint32_t* out_hit_rows, uint64_t cap, uint64_t* out_hit_offsets) {
    return guarded(ctx, [&] {
        if (!ctx->has_result) throw BadInput("no scan result to fetch on this ctx");
        VL_CUDA(cudaSetDevice(ctx->device));
        const vlscan_batch* b = ctx->last_batch;
        BatchView B = b->view();
        ctx->hit_offs.ensure((b->nblocks + 1) * 8); ctx->hits.ensure(std::max<uint64_t>(cap, 4) * 4);
        k_scan_counts<<<1, 1024, 0, ctx->stream>>>(ctx->counts.as<uint32_t>(), (uint32_t)b->nblocks, ctx->hit_offs.as<uint64_t>()); launch_check(ctx);
        if (b->nblocks) { k_hits_compact<<<cdiv((uint64_t)b->nblocks * 32, 256), 256, 0, ctx->stream>>>(B, ctx->regs[0].as<uint64_t>(), ctx->hit_offs.as<uint64_t>(), ctx->hits.as<uint32_t>(), cap); launch_check(ctx); }
        VL_CUDA(cudaMemcpyAsync(out_hit_offsets, ctx->hit_offs.p, (b->nblocks + 1) * 8, cudaMemcpyDeviceToHost, ctx->stream));
        VL_CUDA(cudaStreamSynchronize(ctx->stream));
        uint64_t total = out_hit_offsets[b->nblocks];
        if (total > cap) throw BadInput("hit buffer too small");
        if (total) VL_CUDA(cudaMemcpyAsync(out_hit_rows, ctx->hits.p, total * 4, cudaMemcpyDeviceToHost, ctx->stream));
        VL_CUDA(cudaStreamSynchronize(ctx->stream));
    });
}

// ---- hit materialisation ----------------------------------------------------------------------------------------------------------------------
// hits of the last scan on the device: ctx->hits (row inside its block), ctx->hit_block, ctx->hit_offs (first hit of every block); returns their number
static uint64_t build_hit_list(vlscan_ctx* ctx, uint64_t* out_hit_offsets) {
    if (!ctx->has_result) throw BadInput("no scan result on this ctx");
    VL_CUDA(cudaSetDevice(ctx->device));
    const vlscan_batch* b = ctx->last_batch;
    BatchView B = b->view();
    ctx->hit_offs.ensure((b->nblocks + 1) * 8);
    k_scan_counts<<<1, 1024, 0, ctx->stream>>>(ctx->counts.as<uint32_t>(), (uint32_t)b->nblocks, ctx->hit_offs.as<uint64_t>()); launch_check(ctx);
    uint64_t total = 0;
    VL_CUDA(cudaMemcpyAsync(&total, ctx->hit_offs.as<uint64_t>() + b->nblocks, 8, cudaMemcpyDeviceToHost, ctx->stream));
    if (out_hit_offsets) VL_CUDA(cudaMemcpyAsync(out_hit_offsets, ctx->hit_offs.p, (b->nblocks + 1) * 8, cudaMemcpyDeviceToHost, ctx->stream));
    VL_CUDA(cudaStreamSynchronize(ctx->stream));
    ctx->hits.ensure(std::max<uint64_t>(total, 4) * 4); ctx->hit_block.ensure(std::max<uint64_t>(total, 4) * 4);
    if (b->nblocks && total) {
        k_hits_compact2<<<cdiv((uint64_t)b->nblocks * 32, 256), 256, 0, ctx->stream>>>(B, ctx->regs[0].as<uint64_t>(), ctx->hit_offs.as<uint64_t>(), ctx->hits.as<uint32_t>(), ctx->hit_block.as<uint32_t>(), total);
        launch_check(ctx);
    }
    ctx->gstat.ensure(ST_COUNT * 8);
    VL_CUDA(cudaMemsetAsync(ctx->gstat.p, 0, ST_COUNT * 8, ctx->stream));
    return total;
}
static void check_gather_errors(vlscan_ctx* ctx) {
    unsigned long long h[ST_COUNT];
    VL_CUDA(cudaMemcpyAsync(h, ctx->gstat.p, sizeof h, cudaMemcpyDeviceToHost, ctx->stream));
    VL_CUDA(cudaStreamSynchronize(ctx->stream));
    static const char* const msg[] = {"", "cannot unmarshal strings: row lengths do not add up to the data length", "too big index for dict value", "unexpected length for binary representation of a number", "",
                                      "unexpected uint64 block type", "the timestamps of a block with selected rows were not handed over", "cannot unmarshal timestamps"};
    if (h[ST_ERROR]) throw BadInput(msg[std::min<unsigned long long>(h[ST_ERROR], 7)]);
}

int vlscan_gather_timestamps(vlscan_ctx* ctx, int64_t* out_timestamps, uint64_t cap, uint64_t* out_hit_offsets) {
    return guarded(ctx, [&] {
        const uint64_t n = build_hit_list(ctx, out_hit_offsets);
        if (n > cap) throw BadInput("timestamps buffer too small");
        if (!n) return;
        const vlscan_batch* b = ctx->last_batch;
        BatchView B = b->view();
        uint32_t* wc = ctx->work_count.as<uint32_t>(); uint32_t* row_blocks = ctx->row_blocks.as<uint32_t>();
        unsigned long long* gstat = ctx->gstat.as<unsigned long long>();
        VL_CUDA(cudaMemsetAsync(wc, 0, WC_COUNT * 4, ctx->stream));
        k_hit_blocks_list<<<cdiv(b->nblocks, 256), 256, 0, ctx->stream>>>(B, ctx->counts.as<uint32_t>(), -1, 1, row_blocks, wc); launch_check(ctx);
        ctx->ts_vals.ensure(b->nwords * 64 * 8);
        k_ts_decode_list<<<ctx->sm_count * 4, 256, 0, ctx->stream>>>(B, row_blocks, wc, ctx->ts_vals.as<unsigned long long>(), gstat); launch_check(ctx);
        ctx->gout.ensure(n * 8);
        k_gather_ts<<<cdiv(n, 256), 256, 0, ctx->stream>>>(B, ctx->hits.as<uint32_t>(), ctx->hit_block.as<uint32_t>(), n, ctx->ts_vals.as<unsigned long long>(), ctx->gout.as<long long>()); launch_check(ctx);
        check_gather_errors(ctx);
        VL_CUDA(cudaMemcpy(out_timestamps, ctx->gout.p, n * 8, cudaMemcpyDeviceToHost));
    });
}

int vlscan_gather_values(vlscan_ctx* ctx, const char* field, size_t field_len, uint8_t* out_bytes, uint64_t cap_bytes, uint64_t* out_value_offsets, uint64_t cap_values,
                         uint64_t* out_total_bytes, uint64_t* out_hit_offsets) {
    if (out_total_bytes) *out_total_bytes = 0;
    return guarded(ctx, [&] {
        const uint64_t n = build_hit_list(ctx, out_hit_offsets);
        if (n > cap_values) throw BadInput("value offsets buffer too small");
        if (out_value_offsets) out_value_offsets[0] = 0;
        if (!n) return;
        const vlscan_batch* b = ctx->last_batch;
        BatchView B = b->view();
        std::string name(field, field_len); if (name.empty()) name = "_msg";   // getCanonicalColumnName
        int slot = -1;
        for (uint32_t s2 = 0; s2 < b->nfields; s2++) if (b->field_names[s2] == name) slot = (int)s2;
        uint32_t* wc = ctx->work_count.as<uint32_t>(); uint32_t* lens_blocks = ctx->lens_blocks.as<uint32_t>();
        unsigned long long* gstat = ctx->gstat.as<unsigned long long>();
        const uint32_t* ro = nullptr;
        if (slot >= 0) {   // row offsets of the strings blocks with hits (kept from the scan where it already computed them)
            VL_CUDA(cudaMemsetAsync(wc, 0, WC_COUNT * 4, ctx->stream));
            k_hit_blocks_list<<<cdiv(b->nblocks, 256), 256, 0, ctx->stream>>>(B, ctx->counts.as<uint32_t>(), slot, 0, lens_blocks, wc); launch_check(ctx);
            uint8_t* ready = ctx->ready[slot].as<uint8_t>();
            if (!ctx->ready_cleared[slot]) { VL_CUDA(cudaMemsetAsync(ready, 0, B.nblocks, ctx->stream)); ctx->ready_cleared[slot] = 1; }
            k_lens_offsets<<<ctx->sm_count * 8, 256, 0, ctx->stream>>>(B, slot, lens_blocks, wc, ctx->row_off8[slot].as<uint32_t>(), ready, gstat); launch_check(ctx);
            ro = ctx->row_off8[slot].as<uint32_t>();
        }
        const uint64_t ntiles = cdiv(n, VL_SCAN_TILE);
        ctx->glens.ensure(n * 4); ctx->goffs.ensure((n + 1) * 8); ctx->gtiles.ensure((ntiles + 1) * 8);
        k_gather_values<<<cdiv(n, 128), 128, 0, ctx->stream>>>(B, slot, ctx->hits.as<uint32_t>(), ctx->hit_block.as<uint32_t>(), n, ro, 0, ctx->glens.as<uint32_t>(), nullptr, nullptr, gstat); launch_check(ctx);
        k_scan_tiles<<<(unsigned)ntiles, 256, 0, ctx->stream>>>(ctx->glens.as<uint32_t>(), n, ctx->gtiles.as<unsigned long long>(), nullptr, 0); launch_check(ctx);
        k_scan_tile_sums<<<1, 1024, 0, ctx->stream>>>(ctx->gtiles.as<unsigned long long>(), ntiles, ctx->goffs.as<unsigned long long>() + n); launch_check(ctx);
        k_scan_tiles<<<(unsigned)ntiles, 256, 0, ctx->stream>>>(ctx->glens.as<uint32_t>(), n, ctx->gtiles.as<unsigned long long>(), ctx->goffs.as<unsigned long long>(), 1); launch_check(ctx);
        uint64_t total = 0;
        VL_CUDA(cudaMemcpyAsync(&total, ctx->goffs.as<uint64_t>() + n, 8, cudaMemcpyDeviceToHost, ctx->stream));
        check_gather_errors(ctx);
        if (out_total_bytes) *out_total_bytes = total;
        if (total > cap_bytes) throw BadInput("values buffer too small (the needed size is reported)");
        ctx->gout.ensure(std::max<uint64_t>(total, 16));
        k_gather_values<<<cdiv(n, 128), 128, 0, ctx->stream>>>(B, slot, ctx->hits.as<uint32_t>(), ctx->hit_block.as<uint32_t>(), n, ro, 1, nullptr, ctx->goffs.as<uint64_t>(), ctx->gout.as<uint8_t>(), gstat); launch_check(ctx);
        if (out_value_offsets) VL_CUDA(cudaMemcpyAsync(out_value_offsets, ctx->goffs.p, (n + 1) * 8, cudaMemcpyDeviceToHost, ctx->stream));
        if (total) VL_CUDA(cudaMemcpyAsync(out_bytes, ctx->gout.p, total, cudaMemcpyDeviceToHost, ctx->stream));
        VL_CUDA(cudaStreamSynchronize(ctx->stream));
    });
}

int vlscan_result_digest(vlscan_ctx* ctx, uint64_t block_lo, uint64_t block_hi, uint64_t key_base, uint64_t* out_digest) {
    return guarded(ctx, [&] {
        if (!ctx->has_result) throw BadInput("no scan result on this ctx");
        if (block_lo > block_hi || block_hi > ctx->last_nblocks) throw BadInput("block range outside the batch of the last scan");
        VL_CUDA(cudaSetDevice(ctx->device));
        ctx->hit_offs.ensure(16);
        VL_CUDA(cudaMemsetAsync(ctx->hit_offs.p, 0, 8, ctx->stream));
        if (block_hi > block_lo) {
            k_bitmap_digest<<<cdiv(block_hi - block_lo, 128), 128, 0, ctx->stream>>>(ctx->last_batch->view(), ctx->regs[0].as<uint64_t>(), (uint32_t)block_lo, (uint32_t)block_hi, key_base, ctx->hit_offs.as<unsigned long long>());
            launch_check(ctx);
        }
        VL_CUDA(cudaMemcpyAsync(out_digest, ctx->hit_offs.p, 8, cudaMemcpyDeviceToHost, ctx->stream));
        VL_CUDA(cudaStreamSynchronize(ctx->stream));
    });
}

int vlscan_totals_sum(vlscan_ctx* const* ctxs, int nctx, uint64_t out4[4]) {
    out4[0] = out4[1] = out4[2] = out4[3] = 0;
    for (int i = 0; i < nctx; i++) {
        vlscan_ctx* ctx = ctxs[i];
        int rc = guarded(ctx, [&] {
            if (!ctx->has_result) throw BadInput("no scan result on this ctx");
            VL_CUDA(cudaSetDevice(ctx->device));
            unsigned long long t[4];
            VL_CUDA(cudaMemcpyAsync(t, ctx->totals.p, 32, cudaMemcpyDeviceToHost, ctx->stream));
            VL_CUDA(cudaStreamSynchronize(ctx->stream));
            for (int k = 0; k < 4; k++) out4[k] += t[k];
        });
        if (rc) return rc;
    }
    return 0;
}

int vlscan_result_device_ptrs(vlscan_ctx* ctx, void** bitmap_words, void** match_counts, void** totals4) {
    if (!ctx->has_result) { ctx->err = "no scan result on this ctx"; return -1; }
    if (bitmap_words) *bitmap_words = ctx->regs[0].p;
    if (match_counts) *match_counts = ctx->counts.p;
    if (totals4) *totals4 = ctx->totals.p;
    return 0;
}

int vlscan_scan_batch(vlscan_ctx* ctx, const vlscan_program* prog, const char* const* field_names, const size_t* field_name_lens, uint32_t nfields,
                      const vlscan_block* blocks, uint64_t nblocks, uint64_t* out_bitmap_words, uint32_t* out_match_counts, vlscan_stats* stats) {
    // the staging batch (HBM arena + descriptor tables) is recycled across calls of this ctx: a search worker submits batch after
    // batch, so cudaMalloc / cudaFree of a multi-GB arena per call would sit on the critical path
    vlscan_batch* b = ctx->recycle ? ctx->recycle : new vlscan_batch();
    ctx->recycle = nullptr;
    b->field_names.clear(); b->slot_vt_mask.clear();
    uint64_t launches0 = ctx->launches;
    // which fields' bloom filters the program can ever probe: leaves with token hashes (or in() / contains_any() token sets) and the per-field
    // tokens of the AND / OR pre-passes
    std::vector<char> need_bloom(nfields, 0);
    {
        const Program& P = prog->p;
        auto mark = [&](int field) { for (uint32_t s = 0; s < nfields; s++) if (std::string(field_names[s], field_name_lens[s]) == P.fields[field]) need_bloom[s] = 1; };
        for (const DevLeaf& L : P.leaves) if (L.nhashes || L.nhashes2 || L.in_nsets) mark(L.field);
        for (const DevPrepass& pp : P.prepass) if (pp.nhashes) mark(pp.field);
    }
    // Bloom-first staging (the reference reads a column's values only after the block got past the bloom filters, block_search.go:411-474): when
    // the program probes bloom filters at all, the headers and bloom filters go first, a probe pass marks the columns some filter can reach,
    // and only their values cross PCIe and get decoded.  VLSCAN_BLOOM_FIRST = 0 never, 2 always, 1 (default) adaptive: after a probe that
    // pruned less than 1/8 of the values bytes the next 7 calls with the same program stage everything at once (the probe serialises the
    // bloom copy with the decode, which costs more than it saves when nearly every block is read anyway).
    int bf = 1;
    if (const char* e = getenv("VLSCAN_BLOOM_FIRST")) bf = atoi(e);
    bool probes = false;
    for (char c : need_bloom) probes |= c != 0;
    if (ctx->bf_prog != (const void*)prog) { ctx->bf_prog = prog; ctx->bf_skip = 0; }
    const bool two_phase = bf != 0 && probes && nblocks > 0 && (bf == 2 || ctx->bf_skip == 0);
    if (!two_phase && ctx->bf_skip > 0) ctx->bf_skip--;
    int rc;
    if (two_phase) {
        rc = guarded(ctx, [&] {
            do_upload(ctx, field_names, field_name_lens, nfields, blocks, nblocks, b, stats, &need_bloom, UP_HEADERS);
            std::vector<uint8_t> need;
            do_probe(ctx, prog, b, need);
            uint64_t vals_all = 0, vals_need = 0, cols_all = 0, cols_need = 0;
            for (uint64_t i = 0; i < nblocks; i++)
                for (uint32_t k = 0; k < blocks[i].ncols; k++) {
                    const vlscan_column& c = blocks[i].cols[k];
                    if (c.kind != VLSCAN_COL_VALUES || c.field >= nfields) continue;
                    const uint64_t n = c.stage == VLSCAN_STAGE_ONDISK ? c.values_len : c.lens_items_len + c.data_len;
                    vals_all += n; cols_all++;
                    if (need[i * nfields + c.field]) { vals_need += n; cols_need++; }
                }
            if (stats) { stats->staged_columns += cols_need; stats->pruned_columns += cols_all - cols_need; }
            if (vals_need * 8 > vals_all * 7) ctx->bf_skip = 7;
            do_upload(ctx, field_names, field_name_lens, nfields, blocks, nblocks, b, stats, &need_bloom, UP_VALUES, need.data());
        });
    } else rc = guarded(ctx, [&] { do_upload(ctx, field_names, field_name_lens, nfields, blocks, nblocks, b, stats, &need_bloom); });
    if (rc) { cudaStreamSynchronize(ctx->copy_stream); cudaStreamSynchronize(ctx->stream); }   // nothing may still read the caller's buffers
    if (!rc) rc = vlscan_scan_resident(ctx, prog, b, nullptr);
    if (!rc) rc = vlscan_fetch_results(ctx, out_bitmap_words, out_match_counts, stats);
    if (!rc && stats) {
        rc = guarded(ctx, [&] { read_stats(ctx, stats, true); stats->blocks += b->nblocks; stats->rows += b->rows; stats->gpu_launches += ctx->launches - launches0; });
    }
    ctx->has_result = false; ctx->last_batch = nullptr;
    ctx->recycle = b;
    return rc;
}

}  // extern "C"
