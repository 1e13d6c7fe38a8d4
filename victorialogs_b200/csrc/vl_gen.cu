// Synthetic data set generator, on the device (benchmark / test infrastructure of libvlscan.so).
//
// Row shape: app/vlogsgenerator/main.go:240-281 (`_msg` template, toIPv4 :335-345, toUUID :347-349, dictValues :288-297),
// made deterministic (counter-based RNG keyed by seed, block, row, draw) and extended with a hit / decoy vocabulary, a
// block-clustering knob and `level` / `path` / `status` fields so that the BASELINE.json queries have something to find.
// The kernels emit, per block, exactly the bytes the reference WRITER would hand to the scanner after ZSTD decoding:
//   * strings columns: uintBlock lens items (u8 or the const form, lib/logstorage/encoding.go:190-243) + concatenated bytes,
//   * `level`: dict column, ids in first-seen order (values_encoder.go:1224-1241), no bloom (block.go:159-168),
//   * `status`: uint16 column, big-endian values + min/max (values_encoder.go:1168-1222),
//   * bloom filters: 16 bits per unique token hash, 6 probes, big-endian u64 words (bloomfilter.go:83-121).
// tests/test_gpu_gen.py checks the output byte-for-byte against the CPU oracle's restatement of that writer path.
//
// Supported envelope (anything else is refused with an error instead of silently diverging from the writer):
// 64 <= rows per block <= 8192, every generated column keeps its expected encoding (string / dict / uint16).
#include <algorithm>
#include <cstring>
#include <vector>
#include "vl_engine.h"
#include "vl_hd.cuh"   // fmt_u64, fmt_ipv4, ascii_tokens, xxh64

using namespace vl;

namespace {

__host__ __device__ inline uint64_t gen_rnd(uint64_t seed, uint64_t b, uint64_t i, uint64_t k) {
    uint64_t z = seed + (b + 1) * 0x9E3779B97F4A7C15ULL + (i + 1) * 0xD1B54A32D192ED03ULL + (k + 1) * 0x8CB92BA72F3D8DD7ULL;
    z ^= z >> 30; z *= 0xBF58476D1CE4E5B9ULL; z ^= z >> 27; z *= 0x94D049BB133111EBULL; z ^= z >> 31;
    return z;
}

__device__ const char* const D_VOCAB[12] = {"error", "timeout", "GET /api/v1/items", "conn 10.0.0.7 refused", "errors", "timeouts", "GETS /api/v2",
                                            "connection refuse", "conn reset by peer", "terror", "error timeout", "POST /api/v1/items"};
__device__ const char* const D_LEVELS[8] = {"debug", "info", "warn", "error", "fatal", "ERROR", "FATAL", "INFO"};
__device__ const uint32_t D_STATUS[9] = {200, 201, 204, 301, 400, 404, 500, 502, 503};

__device__ __forceinline__ int put_str(uint8_t* d, const char* s) { int n = 0; while (s[n]) { d[n] = (uint8_t)s[n]; n++; } return n; }
__device__ __forceinline__ int put_hex(uint8_t* d, uint64_t v, int width) { for (int i = width - 1; i >= 0; i--) { uint32_t x = v & 15; d[i] = (uint8_t)(x < 10 ? '0' + x : 'a' + x - 10); v >>= 4; } return width; }

__device__ int gen_msg(const vlscan_gen_config& c, bool hot, uint64_t b, uint64_t i, uint8_t* d) {
    uint64_t r0 = gen_rnd(c.seed, b, i, 0);
    int n = 0;
    const uint32_t focus = (c.columns_mask >> 8) & 15;   // 1..12: every vocabulary row draws entry focus - 1 (selectivity sweeps); 0: uniform
    if (hot && (r0 % 1000) < c.hit_row_permille) n += put_str(d + n, D_VOCAB[focus ? focus - 1 : (r0 >> 32) % 12]); else n += put_str(d + n, "message");
    n += put_str(d + n, " for the stream "); n += fmt_u64(d + n, b);
    n += put_str(d + n, " and worker "); n += fmt_u64(d + n, b % 7);
    n += put_str(d + n, "; ip="); n += fmt_ipv4(d + n, (uint32_t)gen_rnd(c.seed, b, i, 1));
    uint64_t ua = gen_rnd(c.seed, b, i, 2), ub = gen_rnd(c.seed, b, i, 3);
    n += put_str(d + n, "; uuid=");
    n += put_hex(d + n, ua & 0xffffffffULL, 8); d[n++] = '-'; n += put_hex(d + n, (ua >> 32) & 0xffff, 4); d[n++] = '-'; n += put_hex(d + n, ua >> 48, 4); d[n++] = '-';
    n += put_hex(d + n, ub & 0xffff, 4); d[n++] = '-'; n += put_hex(d + n, ub >> 16, 12);
    n += put_str(d + n, "; u64="); n += fmt_u64(d + n, gen_rnd(c.seed, b, i, 4));
    return n;
}
__device__ int gen_path(const vlscan_gen_config& c, uint64_t b, uint64_t i, uint8_t* d) {
    uint64_t r = gen_rnd(c.seed, b, i, 6);
    int n = 0;
    switch (r % 4) {
    case 0: case 1: n += put_str(d, "api/v1/items/"); n += fmt_u64(d + n, (r >> 8) % 100000); break;
    case 2: n += put_str(d, "static/js/app."); n += fmt_u64(d + n, (r >> 8) % 1000); n += put_str(d + n, ".js"); break;
    default: n += put_str(d, "health");
    }
    return n;
}

// per-block summary produced by pass A
struct GenInfo {
    uint32_t msg_bytes, msg_minlen, msg_maxlen, msg_tokens;
    uint32_t path_bytes, path_minlen, path_maxlen, path_tokens, path_distinct;
    uint32_t level_first[8];     // first row of each level value (0xFFFFFFFF if absent)
    uint32_t status_mask;        // bit k: GEN_STATUS[k] present
    uint32_t overflow;           // hash table overflow (should never happen)
};

// open-addressing set of 64-bit keys (0 = empty); returns true when the key was newly inserted
__device__ bool set_insert(unsigned long long* tab, uint32_t cap_mask, uint64_t key, uint32_t* overflow) {
    if (key == 0) key = 0x9E3779B97F4A7C15ULL;   // never produced by XXH64 of a short token in practice; keeps 0 as the empty marker
    uint32_t slot = (uint32_t)(key * 0x9E3779B97F4A7C15ULL >> 32) & cap_mask;
    for (uint32_t probes = 0; probes <= cap_mask; probes++) {
        unsigned long long prev = atomicCAS(&tab[slot], 0ull, (unsigned long long)key);
        if (prev == 0ull) return true;
        if (prev == key) return false;
        slot = (slot + 1) & cap_mask;
    }
    atomicExch(overflow, 1u);
    return false;
}
template <class F> __device__ void ascii_tokens(const uint8_t* s, int n, F&& f) {   // tokenizer.go:40-78 (generated text is ASCII)
    int i = 0;
    while (i < n) {
        while (i < n && !is_token_char(s[i])) i++;
        int st = i;
        while (i < n && is_token_char(s[i])) i++;
        if (i > st) f(s + st, (uint32_t)(i - st));
    }
}

// pass A: sizes, unique-token counts, encodings
__global__ void k_gen_measure(vlscan_gen_config c, uint64_t block_lo, uint32_t nblocks, GenInfo* __restrict__ info, unsigned long long* __restrict__ tables, uint32_t cap_mask) {
    __shared__ GenInfo s;
    unsigned long long* tab_msg = tables + (size_t)blockIdx.x * 3 * (cap_mask + 1);
    unsigned long long* tab_path = tab_msg + (cap_mask + 1);
    unsigned long long* tab_vals = tab_path + (cap_mask + 1);
    for (uint32_t j = blockIdx.x; j < nblocks; j += gridDim.x) {
        uint64_t b = block_lo + j;
        uint64_t lo = b * c.rows_per_block, hi = min((unsigned long long)c.total_rows, (unsigned long long)(lo + c.rows_per_block));
        uint32_t rows = (uint32_t)(hi - lo);
        for (uint32_t k = threadIdx.x; k < 3 * (cap_mask + 1); k += blockDim.x) tab_msg[k] = 0;
        if (threadIdx.x == 0) { memset(&s, 0, sizeof s); s.msg_minlen = s.path_minlen = 0xFFFFFFFFu; for (int k = 0; k < 8; k++) s.level_first[k] = 0xFFFFFFFFu; }
        __syncthreads();
        bool hot = gen_rnd(c.seed, b, 0xFFFFFFFFULL, 0) % 1000 < c.hot_block_permille;
        uint8_t buf[192];
        for (uint32_t i = threadIdx.x; i < rows; i += blockDim.x) {
            if (c.columns_mask & 1) {
                int n = gen_msg(c, hot, b, i, buf);
                atomicAdd(&s.msg_bytes, (uint32_t)n); atomicMin(&s.msg_minlen, (uint32_t)n); atomicMax(&s.msg_maxlen, (uint32_t)n);
                ascii_tokens(buf, n, [&](const uint8_t* t, uint32_t tl) { if (set_insert(tab_msg, cap_mask, xxh64(t, tl), &s.overflow)) atomicAdd(&s.msg_tokens, 1u); });
            }
            if (c.columns_mask & 2) atomicMin(&s.level_first[gen_rnd(c.seed, b, i, 5) % 8], i);
            if (c.columns_mask & 4) {
                int n = gen_path(c, b, i, buf);
                atomicAdd(&s.path_bytes, (uint32_t)n); atomicMin(&s.path_minlen, (uint32_t)n); atomicMax(&s.path_maxlen, (uint32_t)n);
                // distinct VALUES (dict / const detection)
                if (set_insert(tab_vals, cap_mask, xxh64(buf, (uint32_t)n), &s.overflow)) atomicAdd(&s.path_distinct, 1u);
                ascii_tokens(buf, n, [&](const uint8_t* t, uint32_t tl) { if (set_insert(tab_path, cap_mask, xxh64(t, tl), &s.overflow)) atomicAdd(&s.path_tokens, 1u); });
            }
            if (c.columns_mask & 8) atomicOr(&s.status_mask, 1u << (gen_rnd(c.seed, b, i, 7) % 9));
        }
        __syncthreads();
        if (threadIdx.x == 0) info[j] = s;
        __syncthreads();
    }
}

struct GenPlan {   // per block, arena offsets decided by the host after pass A
    uint64_t msg_lens, msg_data, msg_bloom; uint32_t msg_bloom_words, msg_lens_const;
    uint64_t lvl_data, lvl_meta; uint32_t lvl_dict_len; uint8_t lvl_ids[8];
    uint64_t path_lens, path_data, path_bloom; uint32_t path_bloom_words, path_lens_const;
    uint64_t st_data, st_bloom; uint32_t st_bloom_words;
};

__device__ void bloom_add(unsigned long long* words, uint32_t nwords, uint64_t token_hash) {   // initBloomFilter bloomfilter.go:109-121
    if (!nwords) return;
    uint64_t maxbits = (uint64_t)nwords * 64;
    for (int k = 0; k < 6; k++) { uint64_t idx = xxh64_u64(token_hash + k) % maxbits; atomicOr(&words[idx >> 6], 1ull << (idx & 63)); }
}
__device__ __forceinline__ unsigned long long bswap64(unsigned long long x) {
    uint32_t lo = (uint32_t)x, hi = (uint32_t)(x >> 32);
    return ((unsigned long long)__byte_perm(lo, 0, 0x0123) << 32) | __byte_perm(hi, 0, 0x0123);
}

// pass B: write payloads
__global__ void __launch_bounds__(256) k_gen_fill(vlscan_gen_config c, uint64_t block_lo, uint32_t nblocks, const GenPlan* __restrict__ plans, uint8_t* __restrict__ arena) {
    __shared__ uint32_t s_off[8192 + 1];
    __shared__ uint32_t s_carry;
    __shared__ uint32_t s_wsum[8];
    for (uint32_t j = blockIdx.x; j < nblocks; j += gridDim.x) {
        const GenPlan& pl = plans[j];
        uint64_t b = block_lo + j;
        uint64_t lo = b * c.rows_per_block, hi = min((unsigned long long)c.total_rows, (unsigned long long)(lo + c.rows_per_block));
        uint32_t rows = (uint32_t)(hi - lo);
        bool hot = gen_rnd(c.seed, b, 0xFFFFFFFFULL, 0) % 1000 < c.hot_block_permille;
        uint8_t buf[192];
        for (int col = 0; col < 2; col++) {   // the two strings columns: _msg (bit0), path (bit2)
            if (!(c.columns_mask & (col == 0 ? 1 : 4))) continue;
            uint64_t o_lens = col == 0 ? pl.msg_lens : pl.path_lens, o_data = col == 0 ? pl.msg_data : pl.path_data, o_bloom = col == 0 ? pl.msg_bloom : pl.path_bloom;
            uint32_t bw = col == 0 ? pl.msg_bloom_words : pl.path_bloom_words, lconst = col == 0 ? pl.msg_lens_const : pl.path_lens_const;
            // lens + exclusive offsets in shared memory
            if (threadIdx.x == 0) s_carry = 0;
            __syncthreads();
            for (uint32_t base = 0; base < rows; base += blockDim.x) {
                uint32_t i = base + threadIdx.x;
                uint32_t n = 0;
                if (i < rows) n = (uint32_t)(col == 0 ? gen_msg(c, hot, b, i, buf) : gen_path(c, b, i, buf));
                uint32_t incl = n;
#pragma unroll
                for (int d = 1; d < 32; d <<= 1) { uint32_t t = __shfl_up_sync(0xffffffffu, incl, d); if ((threadIdx.x & 31) >= d) incl += t; }
                if ((threadIdx.x & 31) == 31) s_wsum[threadIdx.x >> 5] = incl;
                __syncthreads();
                uint32_t pre = 0; for (uint32_t k = 0; k < (threadIdx.x >> 5); k++) pre += s_wsum[k];
                uint32_t excl = s_carry + pre + incl - n;
                if (i < rows) { s_off[i] = excl; if (lconst == 0xFFFFFFFFu) arena[o_lens + i] = (uint8_t)n; }
                __syncthreads();
                if (threadIdx.x == blockDim.x - 1) s_carry = excl + n;
                __syncthreads();
            }
            if (lconst != 0xFFFFFFFFu && threadIdx.x == 0) arena[o_lens] = (uint8_t)lconst;   // uintBlockTypeConst8 item
            // bytes + bloom bits
            unsigned long long* bloom = (unsigned long long*)(arena + o_bloom);
            for (uint32_t i = threadIdx.x; i < rows; i += blockDim.x) {
                int n = col == 0 ? gen_msg(c, hot, b, i, buf) : gen_path(c, b, i, buf);
                uint8_t* dst = arena + o_data + s_off[i];
                for (int k = 0; k < n; k++) dst[k] = buf[k];
                ascii_tokens(buf, n, [&](const uint8_t* t, uint32_t tl) { bloom_add(bloom, bw, xxh64(t, tl)); });
            }
            __syncthreads();
            for (uint32_t k = threadIdx.x; k < bw; k += blockDim.x) bloom[k] = bswap64(bloom[k]);   // marshal: big-endian words (bloomfilter.go:49-55)
            __syncthreads();
        }
        if (c.columns_mask & 2) {
            for (uint32_t i = threadIdx.x; i < rows; i += blockDim.x) arena[pl.lvl_data + i] = pl.lvl_ids[gen_rnd(c.seed, b, i, 5) % 8];
            if (threadIdx.x == 0) {   // dict meta: u32 offsets[d+1] then the values in id order
                uint32_t* offs = (uint32_t*)(arena + pl.lvl_meta); uint8_t* vals = arena + pl.lvl_meta + 4 * (pl.lvl_dict_len + 1);
                uint32_t o = 0;
                for (uint32_t id = 0; id < pl.lvl_dict_len; id++) {
                    for (int v = 0; v < 8; v++) if (pl.lvl_ids[v] == id) { offs[id] = o; o += (uint32_t)put_str(vals + o, D_LEVELS[v]); }
                }
                offs[pl.lvl_dict_len] = o;
            }
        }
        if (c.columns_mask & 8) {
            unsigned long long* bloom = (unsigned long long*)(arena + pl.st_bloom);
            for (uint32_t i = threadIdx.x; i < rows; i += blockDim.x) {
                uint32_t v = D_STATUS[gen_rnd(c.seed, b, i, 7) % 9];
                arena[pl.st_data + 2 * i] = (uint8_t)(v >> 8); arena[pl.st_data + 2 * i + 1] = (uint8_t)v;
                int n = fmt_u64(buf, v);
                bloom_add(bloom, pl.st_bloom_words, xxh64(buf, (uint32_t)n));
            }
            __syncthreads();
            for (uint32_t k = threadIdx.x; k < pl.st_bloom_words; k += blockDim.x) bloom[k] = bswap64(bloom[k]);
        }
        __syncthreads();
    }
}

__global__ void k_gen_poke(uint8_t* arena, const uint64_t* offs, const uint8_t* vals, size_t n) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) arena[offs[i]] = vals[i];
}

}  // namespace

extern "C" int vlscan_batch_generate(vlscan_ctx* ctx, const vlscan_gen_config* cfgp, uint64_t block_lo, uint64_t block_hi, vlscan_batch** out) {
    *out = nullptr;
    vlscan_batch* bt = new vlscan_batch();
    try {
        vlscan_gen_config c = *cfgp;
        VL_CUDA(cudaSetDevice(ctx->device));
        uint64_t total_blocks = (c.total_rows + c.rows_per_block - 1) / c.rows_per_block;
        if (c.rows_per_block < 64 || c.rows_per_block > 8192) throw BadInput("generator: rows_per_block must be within [64, 8192]");
        if (block_hi > total_blocks || block_lo > block_hi) throw BadInput("generator: block range outside the data set");
        uint32_t nb = (uint32_t)(block_hi - block_lo);
        std::vector<uint32_t> rows(nb);
        for (uint32_t j = 0; j < nb; j++) { uint64_t lo = (block_lo + j) * c.rows_per_block, hi = std::min<uint64_t>(c.total_rows, lo + c.rows_per_block); rows[j] = (uint32_t)(hi - lo); if (rows[j] < 64) throw BadInput("generator: the last block must keep at least 64 rows"); }
        bt->device = ctx->device;
        static const char* const names[4] = {"_msg", "level", "path", "status"};
        int slot_of[4]; bt->nfields = 0;
        for (int k = 0; k < 4; k++) { slot_of[k] = -1; if (c.columns_mask >> k & 1) { slot_of[k] = (int)bt->nfields++; bt->field_names.push_back(names[k]); } }
        if (!bt->nfields) throw BadInput("generator: empty columns_mask");
        if (((c.columns_mask >> 8) & 15) > 12 || (c.columns_mask >> 12)) throw BadInput("generator: bits 8..11 of columns_mask select a vocabulary entry 1..12, higher bits must be zero");
        // pass A
        uint32_t cap = 1; while (cap < c.rows_per_block * 40u) cap <<= 1;   // <= ~26 tokens per _msg row
        int grid = std::min<int>(std::max<uint32_t>(nb, 1), ctx->sm_count * 2);
        DevBuf tables, info_d, plans_d;
        tables.ensure((size_t)grid * 3 * cap * 8); info_d.ensure(std::max<size_t>((size_t)nb * sizeof(GenInfo), 16));
        std::vector<GenInfo> info(nb);
        if (nb) {
            k_gen_measure<<<grid, 256, 0, ctx->stream>>>(c, block_lo, nb, info_d.as<GenInfo>(), tables.as<unsigned long long>(), cap - 1);
            ctx->launches++; VL_CUDA(cudaGetLastError());
            VL_CUDA(cudaMemcpyAsync(info.data(), info_d.p, (size_t)nb * sizeof(GenInfo), cudaMemcpyDeviceToHost, ctx->stream));
            VL_CUDA(cudaStreamSynchronize(ctx->stream));
        }
        tables.release();
        // layout: block-major, columns in field order, (lens, data, bloom[, dict meta]) -- the same order vlscan_batch_upload uses
        std::vector<DevColumn> cols((size_t)nb * bt->nfields); memset(cols.data(), 0, cols.size() * sizeof(DevColumn));
        std::vector<GenPlan> plans(nb); memset(plans.data(), 0, plans.size() * sizeof(GenPlan));
        uint64_t cursor = 16;
        for (uint32_t j = 0; j < nb; j++) {
            const GenInfo& gi = info[j]; GenPlan& pl = plans[j]; uint32_t R = rows[j];
            if (gi.overflow) throw BadInput("generator: token set overflow");
            auto strings_col = [&](int slot, uint32_t bytes, uint32_t minl, uint32_t maxl, uint32_t tokens, uint64_t* o_lens, uint64_t* o_data, uint64_t* o_bloom, uint32_t* bw, uint32_t* lconst) {
                if (maxl >= 256) throw BadInput("generator: row longer than 255 bytes");
                DevColumn& d = cols[(size_t)j * bt->nfields + slot];
                d.kind = COL_VALUES; d.vt = VT_STRING;
                bool cl = R >= 2 && minl == maxl;   // marshalUint64Items: const form when >= 2 equal items (encoding.go:201)
                d.lens_type = cl ? 4 : 0; d.lens_const = cl ? maxl : 0; *lconst = cl ? maxl : 0xFFFFFFFFu;
                d.lens_off = *o_lens = arena_reserve(cursor, cl ? 1 : R);
                d.data_off = *o_data = arena_reserve(cursor, bytes); d.data_len = bytes;
                *bw = (tokens * 16 + 63) / 64; d.bloom_words = *bw; d.bloom_off = *o_bloom = arena_reserve(cursor, (uint64_t)*bw * 8);
            };
            if (slot_of[0] >= 0) strings_col(slot_of[0], gi.msg_bytes, gi.msg_minlen, gi.msg_maxlen, gi.msg_tokens, &pl.msg_lens, &pl.msg_data, &pl.msg_bloom, &pl.msg_bloom_words, &pl.msg_lens_const);
            if (slot_of[1] >= 0) {
                // dict ids in first-seen order (valuesDict.getOrAdd values_encoder.go:1269-1288)
                std::vector<std::pair<uint32_t, int>> seen;
                for (int v = 0; v < 8; v++) if (gi.level_first[v] != 0xFFFFFFFFu) seen.emplace_back(gi.level_first[v], v);
                std::sort(seen.begin(), seen.end());
                if (seen.size() < 2) throw BadInput("generator: `level` would become a const column in this block");
                memset(pl.lvl_ids, 0xFF, 8);
                uint32_t total = 0; static const uint32_t lvl_len[8] = {5, 4, 4, 5, 5, 5, 5, 4};
                for (size_t id = 0; id < seen.size(); id++) { pl.lvl_ids[seen[id].second] = (uint8_t)id; total += lvl_len[seen[id].second]; }
                pl.lvl_dict_len = (uint32_t)seen.size();
                DevColumn& d = cols[(size_t)j * bt->nfields + slot_of[1]];
                d.kind = COL_VALUES; d.vt = VT_DICT; d.dict_len = (uint8_t)seen.size();
                d.lens_type = 4; d.lens_const = 1;   // R >= 64 rows of 1-byte ids => const8 lens
                d.lens_off = arena_reserve(cursor, 1);
                d.data_off = pl.lvl_data = arena_reserve(cursor, R); d.data_len = R;
                d.bloom_off = arena_reserve(cursor, 0); d.bloom_words = 0;
                d.meta_len = total; d.meta_off = pl.lvl_meta = arena_reserve(cursor, 4 * (seen.size() + 1) + total);
            }
            if (slot_of[2] >= 0) {
                if (gi.path_distinct <= 8) throw BadInput("generator: `path` would become a dict / const column in this block");
                strings_col(slot_of[2], gi.path_bytes, gi.path_minlen, gi.path_maxlen, gi.path_tokens, &pl.path_lens, &pl.path_data, &pl.path_bloom, &pl.path_bloom_words, &pl.path_lens_const);
            }
            if (slot_of[3] >= 0) {
                int present = __builtin_popcount(gi.status_mask);
                if (present <= 8) throw BadInput("generator: `status` would become a dict / const column in this block");
                static const uint32_t st[9] = {200, 201, 204, 301, 400, 404, 500, 502, 503};
                uint32_t mn = 0xFFFFFFFFu, mx = 0; for (int k = 0; k < 9; k++) if (gi.status_mask >> k & 1) { mn = std::min(mn, st[k]); mx = std::max(mx, st[k]); }
                DevColumn& d = cols[(size_t)j * bt->nfields + slot_of[3]];
                d.kind = COL_VALUES; d.vt = VT_UINT16; d.min_value = mn; d.max_value = mx;
                d.lens_type = 4; d.lens_const = 2;
                d.lens_off = arena_reserve(cursor, 1);
                d.data_off = pl.st_data = arena_reserve(cursor, 2ull * R); d.data_len = 2ull * R;
                pl.st_bloom_words = ((uint32_t)present * 16 + 63) / 64; d.bloom_words = pl.st_bloom_words; d.bloom_off = pl.st_bloom = arena_reserve(cursor, (uint64_t)pl.st_bloom_words * 8);
            }
        }
        bt->arena_bytes = cursor + kArenaPad;
        bt->arena.ensure(bt->arena_bytes);
        VL_CUDA(cudaMemsetAsync(bt->arena.p, 0, bt->arena_bytes, ctx->stream));
        plans_d.ensure(std::max<size_t>((size_t)nb * sizeof(GenPlan), 16));
        bt->cols.ensure(std::max<size_t>(cols.size() * sizeof(DevColumn), 16));
        if (nb) {
            VL_CUDA(cudaMemcpyAsync(plans_d.p, plans.data(), (size_t)nb * sizeof(GenPlan), cudaMemcpyHostToDevice, ctx->stream));
            VL_CUDA(cudaMemcpyAsync(bt->cols.p, cols.data(), cols.size() * sizeof(DevColumn), cudaMemcpyHostToDevice, ctx->stream));
            // const lens items of dict / uint16 columns: one byte each, written from the host-side table through a tiny staging copy
            k_gen_fill<<<std::min<int>(nb, ctx->sm_count * 4), 256, 0, ctx->stream>>>(c, block_lo, nb, plans_d.as<GenPlan>(), bt->arena.as<uint8_t>());
            ctx->launches++; VL_CUDA(cudaGetLastError());
            // lens item bytes for the const-lens columns (level: 1, status: 2)
            std::vector<std::pair<uint64_t, uint8_t>> pokes;
            for (uint32_t j = 0; j < nb; j++) {
                if (slot_of[1] >= 0) pokes.emplace_back(cols[(size_t)j * bt->nfields + slot_of[1]].lens_off, (uint8_t)1);
                if (slot_of[3] >= 0) pokes.emplace_back(cols[(size_t)j * bt->nfields + slot_of[3]].lens_off, (uint8_t)2);
            }
            if (!pokes.empty()) {
                // batch the single-byte writes: build a sparse host image chunk by chunk would be wasteful; use a small kernel-free approach
                std::vector<uint64_t> offs(pokes.size()); std::vector<uint8_t> vals(pokes.size());
                for (size_t k = 0; k < pokes.size(); k++) { offs[k] = pokes[k].first; vals[k] = pokes[k].second; }
                DevBuf d_offs, d_vals; d_offs.ensure(offs.size() * 8); d_vals.ensure(vals.size());
                VL_CUDA(cudaMemcpyAsync(d_offs.p, offs.data(), offs.size() * 8, cudaMemcpyHostToDevice, ctx->stream));
                VL_CUDA(cudaMemcpyAsync(d_vals.p, vals.data(), vals.size(), cudaMemcpyHostToDevice, ctx->stream));
                k_gen_poke<<<(unsigned)((offs.size() + 255) / 256), 256, 0, ctx->stream>>>(bt->arena.as<uint8_t>(), d_offs.as<uint64_t>(), d_vals.as<uint8_t>(), offs.size());
                ctx->launches++; VL_CUDA(cudaGetLastError());
                VL_CUDA(cudaStreamSynchronize(ctx->stream));
                d_offs.release(); d_vals.release();
            }
        }
        bt->note_columns(cols);
        finish_batch_layout(ctx, bt, rows);
        plans_d.release(); info_d.release();
        *out = bt;
        return 0;
    } catch (const CudaFail& e) { set_thread_error(e.msg); ctx->err = e.msg; delete bt; return e.code > 0 ? e.code : 1; }
    catch (const BadInput& e) { set_thread_error(e.msg); ctx->err = e.msg; delete bt; return -1; }
    catch (const std::exception& e) { set_thread_error(e.what()); ctx->err = e.what(); delete bt; return -3; }
}

