// CUDA kernels of the block-scan engine (sm_100a).  HBM-bound byte / bitmap work: coalesced 16-byte vector loads,
// warp ballots / shuffles, no tensor cores.  Each kernel names the reference code it replaces.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include "vl_hd.cuh"
#include "vl_anycase.cuh"
#include "vl_mathnum.cuh"
#include "vl_types.h"

namespace vl {

static __device__ __forceinline__ uint32_t lane_id() { return threadIdx.x & 31; }
#define VL_SHORT_ROW_BYTES 48u   /* average row length below which a string block is matched per row instead of row-agnostically */
static __device__ __forceinline__ uint32_t width_of_vt(uint32_t vt) {
    switch (vt) { case VT_DICT: case VT_UINT8: return 1; case VT_UINT16: return 2; case VT_UINT32: case VT_IPV4: return 4; case VT_UINT64: case VT_FLOAT64: case VT_ISO8601: case VT_INT64: return 8; }
    return 0;
}
static __device__ __forceinline__ uint64_t lens_stored_bytes(const DevColumn& c, uint32_t rows) {
    return 1 + (c.lens_type < 4 ? ((uint64_t)rows << c.lens_type) : (1ull << (c.lens_type - 4)));
}
// length of row r (unmarshalUint64Items lib/logstorage/encoding.go:246-336)
static __device__ __forceinline__ uint32_t row_len(const DevColumn& c, const uint8_t* lens, uint32_t r) {
    switch (c.lens_type) {
    case 0: return lens[r];
    case 1: return ld_be16(lens + 2 * (uint64_t)r);
    case 2: return ld_be32(lens + 4 * (uint64_t)r);
    case 3: return (uint32_t)ld_be64(lens + 8 * (uint64_t)r);
    default: return c.lens_const;
    }
}
static __device__ __forceinline__ uint64_t load_fixed_be(const uint8_t* p, uint32_t w) {
    switch (w) { case 1: return p[0]; case 2: return ld_be16(p); case 4: return ld_be32(p); default: return ld_be64(p); }
}
static __device__ __forceinline__ int64_t unzigzag64(uint64_t u) { return (int64_t)(u >> 1) ^ -(int64_t)(u & 1); }

// ---- regex on device (regexutil.Regex.MatchString, regex.go:86-212) -----------------------------------------------------------
static __device__ __forceinline__ uint32_t rx_class(const DevRegex& R, const uint8_t* blob, int32_t r) {
    if (r < 128) return blob[R.ascii_off + r];
    const int32_t* b = (const int32_t*)(blob + R.bounds_off);
    int lo = 0, hi = (int)R.nclasses - 1;
    while (lo < hi) { int mid = (lo + hi + 1) >> 1; if (b[mid] <= r) lo = mid; else hi = mid - 1; }
    return (uint32_t)lo;
}
static __device__ bool dfa_run(const DevRegex& R, const uint8_t* blob, const uint8_t* s, uint32_t n) {
    const uint16_t* T = (const uint16_t*)(blob + R.trans_off);
    uint32_t st = 0;
    for (uint32_t i = 0; i < n;) {
        int w; int32_t r = s[i];
        if (r < 0x80) w = 1; else r = decode_rune(s + i, n - i, &w);
        i += w;
        uint32_t e = T[st * R.nclasses + rx_class(R, blob, r)];
        if (e & 0x8000) return true;
        st = e & 0x7FFF;
        if (st == 0x7FFF) return false;
    }
    return blob[R.accept_off + st] != 0;
}
static __device__ bool regex_match(const DevRegex& R, const uint8_t* blob, const uint8_t* s, uint32_t n) {
    const uint8_t* pre = blob + R.prefix_off; uint32_t pl = R.prefix_len;
    const uint8_t* sub = blob + R.sub_off; uint32_t sl = R.sub_len;
    if (R.only_prefix) return pl == 0 || find_bytes(s, n, pre, pl, 0) >= 0;
    if (pl == 0) {
        if (R.dot_star) return true;
        if (R.dot_plus) return n > 0;
        if (R.sub_kind == 1) return find_bytes(s, n, sub, sl, 0) >= 0;
        if (R.sub_kind == 2) { int k = find_bytes(s, n, sub, sl, 0); return k > 0 && (uint32_t)k + sl < n; }
        return dfa_run(R, blob, s, n);
    }
    int k = find_bytes(s, n, pre, pl, 0);
    if (k < 0) return false;
    uint32_t rem = (uint32_t)k + pl;
    if (R.dot_star) return true;
    if (R.dot_plus) return n > rem;
    if (R.sub_kind == 1) return find_bytes(s + rem, n - rem, sub, sl, 0) >= 0;
    if (R.sub_kind == 2) { int m = find_bytes(s + rem, n - rem, sub, sl, 0); return m > 0 && (uint32_t)m + sl < n - rem; }
    if (R.tail_len) return find_bytes(s + rem, n - rem, blob + R.tail_off, R.tail_len, 0) >= 0;   // `.*LIT` after the first prefix occurrence
    for (;;) {
        if (dfa_run(R, blob, s + rem, n - rem)) return true;
        k = find_bytes(s, n, pre, pl, (uint32_t)k + 1);
        if (k < 0) return false;
        rem = (uint32_t)k + pl;
    }
}

// in(): is the string one of the values (filter_in.go:187-200 for string columns / const / dict)
static __device__ bool in_contains_string(const DevLeaf& L, const uint8_t* blob, const uint8_t* s, uint32_t n) {
    const uint32_t* offs = (const uint32_t*)(blob + L.in_offs_off);
    const uint8_t* base = blob + L.in_blob_off;
    for (uint32_t i = 0; i < L.in_count; i++) { uint32_t a = offs[i], b = offs[i + 1]; if (b - a == n && bytes_equal(base + a, n, s, n)) return true; }
    return false;
}
static __device__ __forceinline__ bool in_contains_typed(const DevLeaf& L, const uint64_t* u64s, uint32_t vt, uint64_t v) {
    const uint64_t* set = u64s + L.in_typed_off[vt];
    int lo = 0, hi = (int)L.in_typed_cnt[vt] - 1;
    while (lo <= hi) { int mid = (lo + hi) >> 1; uint64_t x = set[mid]; if (x == v) return true; if (x < v) lo = mid + 1; else hi = mid - 1; }
    return false;
}

// generic string predicate of a leaf: the closure passed to visitValues / applied to const + dict values
static __device__ bool leaf_match_string(const DevProgram& P, const DevLeaf& L, const uint8_t* s, uint32_t n) {
    const uint8_t* nd = P.blob + L.needle_off;
    switch (L.kind) {
    case F_PHRASE: return match_phrase(s, n, nd, L.needle_len);
    case F_PREFIX: return match_prefix(s, n, nd, L.needle_len);
    case F_EXACT: return bytes_equal(s, n, nd, L.needle_len);
    case F_IN: return in_contains_string(L, P.blob, s, n);
    case F_REGEXP: return regex_match(P.regexes[L.regex], P.blob, s, n);
    case F_EXACT_PREFIX: case F_LEN_RANGE: case F_STRING_RANGE: case F_IPV4_RANGE:   // matchExactPrefix / matchLenRange / matchStringRange / matchIPv4Range
        return range_predicate(L.kind, s, n, nd, L.needle_len, P.blob + L.needle2_off, L.needle2_len, L.aux0, L.aux1);
    case F_VALUE_TYPE: return false;   // decided from the column header alone (k_plan_leaf)
    case F_ANY_CASE_PHRASE: return any_case_match(s, n, nd, L.needle_len, false);   // matchAnyCasePhrase: needle = the lower-cased phrase
    case F_ANY_CASE_PREFIX: return any_case_match(s, n, nd, L.needle_len, true);
    case F_SEQUENCE: return match_sequence(s, n, PhraseList{P.blob + L.list_off, L.list_len});
    case F_CONTAINS_ALL: return match_all_phrases(s, n, PhraseList{P.blob + L.list_off, L.list_len});
    case F_CONTAINS_ANY: return match_any_phrase(s, n, PhraseList{P.blob + L.list_off, L.list_len});
    case F_RANGE: {   // matchRange filter_range.go:352-355: the value as parseMathNumber reads it; NaN is outside every range
        const double f = mn::parse_math_number(s, n);
        return f >= __longlong_as_double((long long)L.rng_fmin) && f <= __longlong_as_double((long long)L.rng_fmax);
    }
    }
    return true;
}
// The text of a typed value (number, IPv4, timestamp) against the leaf.  i(...) leaves run the plain phrase / prefix matcher here, with the
// lower-cased needle and, on iso8601 columns, the upper-cased one ("T", "Z"): filter_any_case_phrase.go:103-126, filter_any_case_prefix.go:106-129.
static __device__ bool leaf_match_typed_text(const DevProgram& P, const DevLeaf& L, uint32_t vt, const uint8_t* s, uint32_t n) {
    if (L.kind == F_ANY_CASE_PHRASE || L.kind == F_ANY_CASE_PREFIX) {
        const uint8_t* nd = P.blob + (vt == VT_ISO8601 ? L.needle2_off : L.needle_off); const uint32_t nl = vt == VT_ISO8601 ? L.needle2_len : L.needle_len;
        return L.kind == F_ANY_CASE_PHRASE ? match_phrase(s, n, nd, nl) : match_prefix(s, n, nd, nl);
    }
    return leaf_match_string(P, L, s, n);
}

// numeric value -> string (toUint8String .. toTimestampISO8601String, filter_prefix.go:365-408, filter_phrase.go:310-346)
static __device__ int encoded_to_string(uint32_t vt, uint64_t raw, uint8_t* buf) {
    switch (vt) {
    case VT_UINT8: case VT_UINT16: case VT_UINT32: case VT_UINT64: return fmt_u64(buf, raw);
    case VT_INT64: return fmt_i64(buf, unzigzag64(raw));
    case VT_IPV4: return fmt_ipv4(buf, (uint32_t)raw);
    case VT_ISO8601: return fmt_iso8601(buf, (int64_t)raw);
    }
    return -1;   // float64 takes leaf_match_f64 (its text can be 300+ bytes long)
}

// float64 value -> shortest decimal text -> string matcher (toFloat64String, filter_phrase.go:304-308; matchFloat64ByPrefix,
// filter_prefix.go:224-252; matchFloat64ByRegex filter_regexp.go).  Kept out of line: the 352-byte text buffer must not
// grow the frame of the common integer path.
static __device__ __noinline__ bool leaf_match_f64(const DevProgram& P, const DevLeaf& L, uint64_t raw) {
    uint8_t buf[VL_FMT_F64_MAX];
    int n = fmt_f64(buf, raw);
    return leaf_match_typed_text(P, L, VT_FLOAT64, buf, (uint32_t)n);
}

// ---- bloom probe, warp wide (bloomFilter.containsAll, lib/logstorage/bloomfilter.go:173-191) -----------------------------------
// All 32 lanes call with identical arguments; lanes split the probe hashes; result is uniform.
static __device__ bool bloom_contains_all_warp(const uint8_t* bloom_be, uint32_t nwords, const uint64_t* hashes, uint32_t nh) {
    if (nwords == 0) return true;
    uint64_t maxbits = (uint64_t)nwords * 64;
    bool ok = true;
    for (uint32_t i = lane_id(); i < nh; i += 32) {
        uint64_t idx = hashes[i] % maxbits;
        uint64_t w = ld_be64(bloom_be + (idx >> 6) * 8);   // words are stored big-endian (bloomfilter.go:49-55)
        if (!((w >> (idx & 63)) & 1)) ok = false;
    }
    return __all_sync(0xffffffffu, ok);
}

// ---- bitmap helpers --------------------------------------------------------------------------------------------------
// is the bitmap of block b non-zero (bitmap.isZero, bitmap.go:74-81)?  All 32 lanes call with the same b; the result is uniform.
static __device__ __forceinline__ bool block_alive_warp(const uint64_t* __restrict__ reg, const BatchView& B, uint32_t b) {
    const uint64_t lo = B.blk_word_off[b], hi = B.blk_word_off[b + 1];
    bool any = false;
    for (uint64_t w = lo + lane_id(); w < hi; w += 32) any |= reg[w] != 0;
    return __any_sync(0xffffffffu, any);
}
// number of rows still selected in block b (bitmap.onesCount); uniform result
static __device__ __forceinline__ uint32_t block_ones_warp(const uint64_t* __restrict__ reg, const BatchView& B, uint32_t b) {
    const uint64_t lo = B.blk_word_off[b], hi = B.blk_word_off[b + 1];
    uint32_t n = 0;
    for (uint64_t w = lo + lane_id(); w < hi; w += 32) n += __popcll(reg[w]);
#pragma unroll
    for (int d = 16; d; d >>= 1) n += __shfl_xor_sync(0xffffffffu, n, d);
    return n;
}
static __global__ void k_andnot(uint64_t* __restrict__ a, const uint64_t* __restrict__ b, uint64_t n) {   // bitmap.andNot bitmap.go:99-111
    uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) a[i] &= ~b[i];
}

// ---- AND / OR bloom pre-pass (filterAnd.matchBloomFilters filter_and.go:76-111, filterOr.matchBloomFilters filter_or.go:80-115) ----
// one warp per block; a failing block gets its bitmap words zeroed (bm.resetBits()).
static __global__ void k_prepass(DevProgram P, BatchView B, uint32_t pp_begin, uint32_t pp_count, const int* __restrict__ slots /* per prepass entry */,
                          int is_or, uint64_t* __restrict__ reg, unsigned long long* __restrict__ stats) {
    uint32_t b = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (b >= B.nblocks || !block_alive_warp(reg, B, b)) return;
    bool pass = is_or ? false : true;
    unsigned long long bloom_bytes = 0;
    for (uint32_t e = 0; e < pp_count; e++) {
        const DevPrepass& pp = P.prepass[pp_begin + e];
        int slot = slots[e];
        const DevColumn* c = slot >= 0 ? &B.cols[(uint64_t)b * B.nfields + slot] : nullptr;
        bool ok;
        bool skip = false;   // OR: "continue" without a verdict
        if (c && c->kind == COL_CONST) {
            // matchStringByAllTokens(v, tokens)
            const uint32_t* to = (const uint32_t*)(P.blob + pp.tok_offs_off);
            const uint8_t* v = B.hdr + c->meta_off;
            ok = true;
            for (uint32_t t = 0; t < pp.ntokens && ok; t++) ok = match_phrase(v, c->meta_len, P.blob + pp.tok_blob_off + to[t], to[t + 1] - to[t]);
        } else if (!c || c->kind == COL_MISSING) {
            ok = false; skip = true;
        } else if (c->vt == VT_DICT) {
            // matchDictValuesByAllTokens: dict values joined with ',' (filter_and.go:198-208); a token never contains ','
            // so a phrase occurrence lies inside one value; value edges behave like the ',' separator (non-token char).
            const uint32_t* dof = (const uint32_t*)(B.hdr + c->meta_off);
            const uint8_t* dv = B.hdr + c->meta_off + 4 * (c->dict_len + 1);
            const uint32_t* to = (const uint32_t*)(P.blob + pp.tok_offs_off);
            ok = true;
            for (uint32_t t = 0; t < pp.ntokens && ok; t++) {
                bool found = false;
                for (uint32_t d = 0; d < c->dict_len && !found; d++) found = match_phrase(dv + dof[d], dof[d + 1] - dof[d], P.blob + pp.tok_blob_off + to[t], to[t + 1] - to[t]);
                ok = found;
            }
        } else {
            bloom_bytes += 8ull * pp.nhashes;
            ok = bloom_contains_all_warp(B.hdr + c->bloom_off, c->bloom_words, P.u64s + pp.hashes_off, pp.nhashes);
        }
        if (is_or) { if (!skip && ok) { pass = true; break; } }
        else if (!ok) { pass = false; break; }
    }
    if (is_or && pp_count == 0) pass = true;
    if (lane_id() == 0 && bloom_bytes) atomicAdd(&stats[ST_BLOOM_BYTES], bloom_bytes);
    if (!pass) for (uint64_t w = B.blk_word_off[b] + lane_id(); w < B.blk_word_off[b + 1]; w += 32) reg[w] = 0;
}

// ---- per (block, leaf) header dispatch: const / missing / dict / typed columns + leaf-level bloom probe ----------------------------
// filterPhrase.applyToBlockSearch filter_phrase.go:61-111, filterPrefix :59-106, filterExact :186-235, filterIn :120-185,
// filterRegexp :78-127 and the match*By* helpers they call.  One warp per block, all lanes run the same scalar logic.
// The same kernel decides bm.isZero() for the block and appends the block to the work lists of the kernels that follow: blocks whose lens
// items must be decoded, the 64 KiB tiles of the row-agnostic scan, blocks of the per-row matcher.  The lists are unordered (appended with
// one atomic per CTA and list): every consumer only needs the set.
#define VL_PLAN_WARPS 8
enum { WC_LENS = 0, WC_TILES = 1, WC_ROW = 2, WC_LENS2 = 3, WC_COUNT = 4 };   // WC_LENS2: the second column of a two-column leaf
#define VL_TILE_BYTES 65536u                  /* row bytes per work item of the substring scan */
static __global__ void __launch_bounds__(VL_PLAN_WARPS * 32) k_plan_leaf(DevProgram P, BatchView B, uint32_t leaf_idx, int slot, const uint64_t* __restrict__ reg,
                            uint8_t* __restrict__ action, uint64_t* __restrict__ payload, uint32_t* __restrict__ lens_blocks, uint32_t* __restrict__ row_blocks,
                            uint32_t* __restrict__ tile_block, uint32_t* __restrict__ tile_off, uint32_t* __restrict__ work_count,
                            unsigned long long* __restrict__ stats, uint8_t* __restrict__ need = nullptr) {
    // need != NULL: PROBE pass of a bloom-first upload (phase 1: headers, bloom filters and dict tables are on the device, no values yet).
    // `reg` then only carries which blocks are still alive behind the AND / OR bloom pre-passes of the leaf's ancestors; the kernel runs the
    // same header dispatch and bloom probes and sets need[block * nfields + slot] when the leaf would go on to read the column's values.
    // Nothing else is written.  Every block the real scan reads values of is marked: the real scan reaches a leaf with a subset of the rows
    // (hence blocks) the probe reaches it with, and the gates below do not depend on the rows.
    __shared__ uint32_t s_cnt[VL_PLAN_WARPS][3], s_off[VL_PLAN_WARPS][3];
    __shared__ unsigned long long s_stat[VL_PLAN_WARPS][4];
    const uint32_t warp = threadIdx.x >> 5;
    const uint32_t b = blockIdx.x * VL_PLAN_WARPS + warp;
    const DevLeaf& L = P.leaves[leaf_idx];
    uint8_t act = ACT_NONE; uint64_t pay = 0;
    unsigned long long bloom_bytes = 0, values_bytes = 0, scan_bytes = 0; int err = 0;
    uint32_t need_lens = 0, need_row = 0, ntiles = 0;
    const bool valid = b < B.nblocks;
    const uint32_t ones = valid ? block_ones_warp(reg, B, b) : 0;
    const bool alive = ones != 0;
    if (alive && L.kind == F_NOOP) act = ACT_ALL;
    else if (alive) {
    act = ACT_ALL;
    uint32_t rows = B.blk_rows[b];
    const DevColumn* c = slot >= 0 ? &B.cols[(uint64_t)b * B.nfields + slot] : nullptr;
    const uint8_t* nd = P.blob + L.needle_off; uint32_t nl = L.needle_len;
    if ((L.kind == F_IN && L.in_count == 0) || L.always_none) act = ACT_NONE;   // fi.values.isEmpty(); minLen > maxLen, minValue > maxValue
    else if (L.kind == F_TIME) {   // filterTime.applyToBlockSearch filter_time.go:114-137: header-level decisions first
        const int64_t mn = (int64_t)L.aux0, mx = (int64_t)L.aux1;
        if (!B.ts || B.ts[b].mt == 0) { act = ACT_NONE; err = ERR_NO_TIMESTAMPS; }
        else if (mn > B.ts[b].max || mx < B.ts[b].first) act = ACT_NONE;
        else if (mn <= B.ts[b].first && mx >= B.ts[b].max) act = ACT_ALL;
        else { act = ACT_TIME; need_row = 1; }
    }
    else if (c && c->kind == COL_CONST) {
        if (L.kind == F_VALUE_TYPE) act = L.aux0 == VTYPE_CONST ? ACT_ALL : ACT_NONE;   // filter_value_type.go:46-52
        else act = leaf_match_string(P, L, B.hdr + c->meta_off, c->meta_len) ? ACT_ALL : ACT_NONE;
    } else if (!c || c->kind == COL_MISSING) {
        switch (L.kind) {
        case F_PHRASE: case F_EXACT: case F_EXACT_PREFIX: act = nl == 0 ? ACT_ALL : ACT_NONE; break;
        case F_PREFIX: act = ACT_NONE; break;
        case F_IN: act = L.in_has_empty ? ACT_ALL : ACT_NONE; break;
        case F_REGEXP: act = regex_match(P.regexes[L.regex], P.blob, nullptr, 0) ? ACT_ALL : ACT_NONE; break;
        case F_LEN_RANGE: act = L.aux0 == 0 ? ACT_ALL : ACT_NONE; break;                                // matchLenRange("", min, max)
        case F_STRING_RANGE: act = (nl == 0 && L.needle2_len > 0) ? ACT_ALL : ACT_NONE; break;           // "" >= min && "" < max
        case F_IPV4_RANGE: case F_VALUE_TYPE: case F_RANGE: act = ACT_NONE; break;
        case F_ANY_CASE_PHRASE: act = nl == 0 ? ACT_ALL : ACT_NONE; break;                               // filter_any_case_phrase.go:88-95
        case F_ANY_CASE_PREFIX: act = ACT_NONE; break;                                                   // filter_any_case_prefix.go:92-97
        case F_SEQUENCE: case F_CONTAINS_ALL: case F_CONTAINS_ANY: act = leaf_match_string(P, L, nullptr, 0) ? ACT_ALL : ACT_NONE; break;   // the predicate on ""
        }
    } else if (L.kind == F_VALUE_TYPE) {
        act = L.aux0 == c->vt ? ACT_ALL : ACT_NONE;   // valueType.String() == wanted name (filter_value_type.go:59-66); no payload is read
    } else if (c->vt == VT_DICT) {
        const uint32_t* dof = (const uint32_t*)(B.hdr + c->meta_off);
        const uint8_t* dv = B.hdr + c->meta_off + 4 * (c->dict_len + 1);
        uint32_t mask = 0;
        for (uint32_t d = 0; d < c->dict_len; d++) if (leaf_match_string(P, L, dv + dof[d], dof[d + 1] - dof[d])) mask |= 1u << d;
        if (mask == 0) act = ACT_NONE; else { act = ACT_DICT; pay = mask; }
    } else {
        uint32_t vt = c->vt;
        const uint8_t* bloom = B.hdr + c->bloom_off;
        auto probe = [&](const uint64_t* h, uint32_t nh) -> bool {
            if (nh == 0) return true;
            bloom_bytes += 8ull * nh;
            return bloom_contains_all_warp(bloom, c->bloom_words, h, nh);
        };
        const uint64_t* H = P.u64s + L.hashes_off; uint32_t nH = L.nhashes;
        if (vt == VT_STRING) {
            bool ok = true;
            if (L.kind == F_IN) {
                // matchBloomFilterAnyTokenSet filter_in.go:202-218
                ok = probe(H, L.nhashes);
                if (ok && !(L.in_skip_sets || (uint64_t)L.in_nsets > 10ull * rows)) {
                    bool any = false;
                    const uint32_t* sets = P.u32s + L.in_sets_off;
                    for (uint32_t s = 0; s < L.in_nsets && !any; s++) { bloom_bytes += 8ull * sets[2 * s + 1]; any = bloom_contains_all_warp(bloom, c->bloom_words, P.u64s + sets[2 * s], sets[2 * s + 1]); }
                    ok = any;
                }
            } else if (L.kind == F_CONTAINS_ANY) {
                // matchValuesAnyPhrase filter_contains_any.go:170-189: the common tokens, then EVERY phrase's own tokens (the reference keeps the
                // phrases that pass; a phrase that does not pass cannot match a row, so trying all of them on the rows gives the same bits)
                ok = probe(H, L.nhashes);
                if (ok) {
                    bool any = false;
                    const uint32_t* sets = P.u32s + L.in_sets_off;
                    for (uint32_t s = 0; s < L.in_nsets; s++) { bloom_bytes += 8ull * sets[2 * s + 1]; any |= bloom_contains_all_warp(bloom, c->bloom_words, P.u64s + sets[2 * s], sets[2 * s + 1]); }
                    ok = any;
                }
            } else if (L.kind == F_ANY_CASE_PHRASE || L.kind == F_ANY_CASE_PREFIX || L.kind == F_RANGE) ok = true;   // i(...): tokens are case sensitive, range(): no tokens - no probe
            else ok = probe(H, L.nhashes);
            if (!ok) act = ACT_NONE;
            else if (need) { act = ACT_ROW; values_bytes = 1; }   // probe: the values would be read
            else if (c->data_const) act = leaf_match_string(P, L, B.arena + c->data_off, (uint32_t)c->data_len) ? ACT_ALL : ACT_NONE, values_bytes = 1;
            else {
                act = L.str_strategy == STR_SCAN ? ACT_SCAN : L.str_strategy == STR_ALL ? ACT_ALL : ACT_ROW; values_bytes = 1;
                // short rows (ids, paths, codes ...): candidates of the row-agnostic scan become dense relative to the bytes streamed and
                // each costs a warp-wide verification, so such blocks take the per-row matcher instead (same predicate, same result)
                if (act == ACT_SCAN && c->data_len < (uint64_t)VL_SHORT_ROW_BYTES * rows) act = ACT_ROW;
                // few rows of the block are still selected (an earlier filter of an AND chain was selective): visit just those, like
                // bm.forEachSetBit does, instead of streaming the whole block
                if (act == ACT_SCAN && (uint64_t)ones * 16 < rows) act = ACT_ROW;
            }
        } else {
            // numeric / ipv4 / iso8601 columns
            uint32_t w = width_of_vt(vt);
            bool fixed_ok = c->lens_type >= 4 && c->lens_const == w && c->data_len == (uint64_t)rows * w && !c->data_const;
            const TypedNeedle& tn = L.typed[vt];
            // i(phrase) / i(prefix*) on typed columns: the phrase / prefix filter's path with the lower-cased needle and this filter's tokens; on
            // iso8601 columns the upper-cased needle and tokens (filter_any_case_phrase.go:103-126)
            uint32_t kind = L.kind;
            if (kind == F_ANY_CASE_PHRASE || kind == F_ANY_CASE_PREFIX) {
                kind = kind == F_ANY_CASE_PHRASE ? F_PHRASE : F_PREFIX;
                if (vt == VT_ISO8601) { H = P.u64s + L.hashes2_off; nH = L.nhashes2; nd = P.blob + L.needle2_off; nl = L.needle2_len; }
            }
            auto in_range = [&]() -> bool {
                switch (vt) {
                case VT_UINT8: case VT_UINT16: case VT_UINT32: case VT_UINT64: case VT_IPV4: return tn.val >= c->min_value && tn.val <= c->max_value;
                case VT_INT64: case VT_ISO8601: return tn.sval >= (int64_t)c->min_value && tn.sval <= (int64_t)c->max_value;
                case VT_FLOAT64: { double f = __longlong_as_double((long long)tn.val), mn = __longlong_as_double((long long)c->min_value), mx = __longlong_as_double((long long)c->max_value); return !(f < mn) && !(f > mx); }
                }
                return false;
            };
            auto exact_path = [&]() {   // match*ByExactValue -> matchBinaryValue (filter_exact.go:237-364)
                if (!tn.ok || !in_range()) { act = ACT_NONE; return; }
                if (!probe(H, nH)) { act = ACT_NONE; return; }
                act = fixed_ok ? ACT_FIXED_EQ : ACT_ROW_EQ; pay = tn.val;
            };
            auto tostring_path = [&](bool use_bloom) {
                if (use_bloom && !probe(H, nH)) { act = ACT_NONE; return; }
                act = ACT_ROW;
            };
            const bool is_uintN = vt == VT_UINT8 || vt == VT_UINT16 || vt == VT_UINT32 || vt == VT_UINT64;
            switch (kind) {
            case F_EXACT: exact_path(); break;
            case F_PHRASE:
                if (vt == VT_FLOAT64) { if (!L.f64_phrase_gate) act = ACT_NONE; else if (L.f64_exact_form) exact_path(); else tostring_path(true); }
                else if (vt == VT_IPV4 || vt == VT_ISO8601) { if (tn.ok) exact_path(); else tostring_path(true); }
                else exact_path();
                break;
            case F_PREFIX:
                if (nl == 0) act = ACT_ALL;
                else if (vt == VT_UINT8 || vt == VT_UINT16 || vt == VT_UINT32 || vt == VT_UINT64) { if (!tn.ok || tn.val > c->max_value) act = ACT_NONE; else tostring_path(false); }
                else if (vt == VT_INT64) { bool dash = nl == 1 && nd[0] == '-'; if (!dash && (!tn.ok || !in_range())) act = ACT_NONE; else tostring_path(false); }
                else if (vt == VT_FLOAT64) { if (!L.f64_prefix_gate) act = ACT_NONE; else tostring_path(true); }
                else tostring_path(true);
                break;
            case F_REGEXP: tostring_path(true); break;
            case F_IN:
                if (L.in_typed_cnt[vt] == 0) act = ACT_NONE;
                else {
                    bool ok = probe(H, L.nhashes);
                    if (ok && !(L.in_skip_sets || (uint64_t)L.in_nsets > 10ull * rows)) {
                        bool any = false;
                        const uint32_t* sets = P.u32s + L.in_sets_off;
                        for (uint32_t s = 0; s < L.in_nsets && !any; s++) { bloom_bytes += 8ull * sets[2 * s + 1]; any = bloom_contains_all_warp(bloom, c->bloom_words, P.u64s + sets[2 * s], sets[2 * s + 1]); }
                        ok = any;
                    }
                    act = !ok ? ACT_NONE : fixed_ok ? ACT_FIXED_IN : ACT_ROW_IN;
                }
                break;
            case F_SEQUENCE:         // filter_sequence.go:139-258
                if (is_uintN || vt == VT_INT64) { if (L.in_count > 1) act = ACT_NONE; else exact_path(); }          // one phrase: the exact value
                else if (vt == VT_FLOAT64) tostring_path(true);
                else if (L.in_count == 1 && tn.ok) exact_path();                                                  // ipv4 / iso8601, one phrase that is a whole value
                else tostring_path(true);
                break;
            case F_CONTAINS_ALL:     // filter_contains_all.go:168-189 (matchAllValues), :191-300
                if (is_uintN) {
                    const uint32_t n_values = (uint32_t)L.aux0;   // distinct non-empty values
                    if (n_values == 0) act = ACT_ALL;
                    else if (n_values != 1 || L.in_typed_cnt[vt] != 1) act = ACT_NONE;
                    else if (!probe(H, nH)) act = ACT_NONE;
                    else { act = fixed_ok ? ACT_FIXED_EQ : ACT_ROW_EQ; pay = P.u64s[L.in_typed_off[vt]]; }
                } else tostring_path(true);
                break;
            case F_CONTAINS_ANY:     // filter_contains_any.go:120-168: uintN like in(), the rest like the strings path over the value's text
                if (is_uintN) {
                    if (L.in_typed_cnt[vt] == 0) act = ACT_NONE;
                    else {
                        bool ok = probe(H, nH);
                        if (ok && !(L.in_skip_sets || (uint64_t)L.in_nsets > 10ull * rows)) {
                            bool any = false;
                            const uint32_t* sets = P.u32s + L.in_sets_off;
                            for (uint32_t s = 0; s < L.in_nsets && !any; s++) { bloom_bytes += 8ull * sets[2 * s + 1]; any = bloom_contains_all_warp(bloom, c->bloom_words, P.u64s + sets[2 * s], sets[2 * s + 1]); }
                            ok = any;
                        }
                        act = !ok ? ACT_NONE : fixed_ok ? ACT_FIXED_IN : ACT_ROW_IN;
                    }
                } else {
                    bool ok = probe(H, nH);
                    if (ok) {
                        bool any = false;
                        const uint32_t* sets = P.u32s + L.in_sets_off;
                        for (uint32_t s = 0; s < L.in_nsets; s++) { bloom_bytes += 8ull * sets[2 * s + 1]; any |= bloom_contains_all_warp(bloom, c->bloom_words, P.u64s + sets[2 * s], sets[2 * s + 1]); }
                        ok = any;
                    }
                    act = ok ? ACT_ROW : ACT_NONE;
                }
                break;
            case F_RANGE: {          // match*ByRange filter_range.go:216-347: header min / max first, then the encoded values themselves
                const double fmn = __longlong_as_double((long long)L.rng_fmin), fmx = __longlong_as_double((long long)L.rng_fmax);
                if (is_uintN) act = (fmx < 0 || L.rng_ulo > c->max_value || L.rng_uhi < c->min_value) ? ACT_NONE : ACT_ROW;
                else if (vt == VT_INT64) act = (L.rng_ilo > (int64_t)c->max_value || L.rng_ihi < (int64_t)c->min_value) ? ACT_NONE : ACT_ROW;
                else if (vt == VT_FLOAT64) act = (fmn > __longlong_as_double((long long)c->max_value) || fmx < __longlong_as_double((long long)c->min_value)) ? ACT_NONE : ACT_ROW;
                else if (vt == VT_IPV4) act = (c->min_value > (uint64_t)L.rng_iphi || c->max_value < (uint64_t)L.rng_iplo) ? ACT_NONE : ACT_ROW;
                else act = (fmx < 0 || L.rng_ilo > (int64_t)c->max_value || L.rng_ihi < (int64_t)c->min_value) ? ACT_NONE : ACT_ROW;   // iso8601: nanoseconds
                break;
            }
            case F_EXACT_PREFIX: {   // match*ByExactPrefix filter_exact_prefix.go:105-273
                const bool is_uint = vt == VT_UINT8 || vt == VT_UINT16 || vt == VT_UINT32 || vt == VT_UINT64;
                if (nl == 0) act = ACT_ALL;
                else if (is_uint) act = (L.nhashes > 0 || !tn.ok || tn.val > c->max_value) ? ACT_NONE : ACT_ROW;   // matchMinMaxExactPrefix
                else if (vt == VT_INT64) {
                    bool dash = nl == 1 && nd[0] == '-';
                    if (L.nhashes > 0) act = ACT_NONE;
                    else if (!dash && (!tn.ok || tn.sval > (int64_t)c->max_value || tn.sval < (int64_t)c->min_value)) act = ACT_NONE;
                    else act = ACT_ROW;
                }
                else if (vt == VT_FLOAT64) act = (L.nhashes > 2 * 6 || !probe(H, L.nhashes)) ? ACT_NONE : ACT_ROW;
                else if (vt == VT_IPV4) act = (!(L.gates & GATE_DIGIT_PREFIX) || L.nhashes > 3 * 6 || !probe(H, L.nhashes)) ? ACT_NONE : ACT_ROW;
                else act = (!(L.gates & GATE_DIGIT_PREFIX) || !probe(H, L.nhashes)) ? ACT_NONE : ACT_ROW;   // iso8601
                break;
            }
            case F_LEN_RANGE: {      // match*ByLenRange filter_len_range.go:209-348
                const uint64_t mn = L.aux0, mx = L.aux1;
                uint8_t tmp[24];
                if (vt == VT_UINT8 || vt == VT_UINT16 || vt == VT_UINT32 || vt == VT_UINT64) {
                    const uint64_t maxd = vt == VT_UINT8 ? 3 : vt == VT_UINT16 ? 5 : vt == VT_UINT32 ? 10 : 20;
                    if (mn > maxd || mx == 0) act = ACT_NONE;
                    else if (mx < (uint64_t)fmt_u64(tmp, c->min_value) || mn > (uint64_t)fmt_u64(tmp, c->max_value)) act = ACT_NONE;   // matchMinMaxValueLen
                    else act = ACT_ROW;
                } else if (vt == VT_INT64) {
                    if (mn > 21 || mx == 0) act = ACT_NONE;
                    else { int a = fmt_i64(tmp, (int64_t)c->min_value), b2 = fmt_i64(tmp, (int64_t)c->max_value); act = (uint64_t)(a > b2 ? a : b2) < mn ? ACT_NONE : ACT_ROW; }
                } else if (vt == VT_FLOAT64) act = (mn > 24 || mx == 0) ? ACT_NONE : ACT_ROW;
                else if (vt == VT_IPV4) act = (mn > 15 || mx < 7) ? ACT_NONE : ACT_ROW;
                else act = (mn > 24 || mx < 24) ? ACT_NONE : ACT_ALL;   // iso8601: every value is 24 characters long, nothing is read
                break;
            }
            case F_STRING_RANGE:     // match*ByStringRange filter_string_range.go:88-224
                if (vt == VT_INT64) act = (L.gates & GATE_SR_INT) ? ACT_ROW : ACT_NONE;
                else if (vt == VT_FLOAT64) act = (L.gates & GATE_SR_FLOAT) ? ACT_ROW : ACT_NONE;
                else act = (L.gates & GATE_SR_UINT) ? ACT_ROW : ACT_NONE;
                break;
            case F_IPV4_RANGE:       // filter_ipv4_range.go:113-131, matchIPv4ByRange :176-191
                if (vt != VT_IPV4) act = ACT_NONE;
                else act = (c->min_value > L.aux1 || c->max_value < L.aux0) ? ACT_NONE : ACT_ROW;
                break;
            }
        }
        if (act >= ACT_DICT || values_bytes) values_bytes = lens_stored_bytes(*c, rows) + c->data_len;   // getValuesForColumn was reached
    }
    if (c && c->kind == COL_VALUES && c->vt == VT_DICT && act == ACT_DICT) values_bytes = lens_stored_bytes(*c, rows) + c->data_len;
    if (need) {
        if (c && c->kind == COL_VALUES && (values_bytes || act >= ACT_DICT) && lane_id() == 0) need[(uint64_t)b * B.nfields + slot] = 1;
        act = ACT_NONE; values_bytes = 0; bloom_bytes = 0; err = 0;
    } else if (c && c->kind == COL_VALUES && c->values_state != VALUES_STAGED && (values_bytes || act >= ACT_DICT)) {
        // cannot happen unless the probe pass and this dispatch disagree: fail loudly rather than read values that were never uploaded
        act = ACT_NONE; values_bytes = 0; err = ERR_VALUES_ABSENT;
    }
    if (c && c->kind == COL_VALUES && (act == ACT_SCAN || act >= ACT_ROW)) {
        need_lens = 1;
        if (act == ACT_SCAN) { ntiles = (uint32_t)((c->data_len + VL_TILE_BYTES - 1) / VL_TILE_BYTES); scan_bytes = c->data_len; }
        else need_row = 1;
    }
    }
    if (need) return;   // probe pass: uniform for the whole grid
    if (lane_id() == 0) {
        if (valid) { action[b] = act; payload[b] = pay; }
        if (err) atomicMax(&stats[ST_ERROR], (unsigned long long)err);
        s_cnt[warp][0] = need_lens; s_cnt[warp][1] = ntiles; s_cnt[warp][2] = need_row;
        s_stat[warp][0] = bloom_bytes; s_stat[warp][1] = values_bytes; s_stat[warp][2] = values_bytes ? 1 : 0; s_stat[warp][3] = scan_bytes;
    }
    __syncthreads();
    if (threadIdx.x < 3) {            // one atomic per CTA and list
        uint32_t tot = 0;
        for (int w = 0; w < VL_PLAN_WARPS; w++) { s_off[w][threadIdx.x] = tot; tot += s_cnt[w][threadIdx.x]; }
        const uint32_t base = tot ? atomicAdd(&work_count[threadIdx.x], tot) : 0;
        for (int w = 0; w < VL_PLAN_WARPS; w++) s_off[w][threadIdx.x] += base;
    } else if (threadIdx.x >= 32 && threadIdx.x < 36) {
        const int k = threadIdx.x - 32;
        unsigned long long tot = 0;
        for (int w = 0; w < VL_PLAN_WARPS; w++) tot += s_stat[w][k];
        if (tot) atomicAdd(&stats[k == 0 ? ST_BLOOM_BYTES : k == 1 ? ST_VALUES_BYTES : k == 2 ? ST_COLUMNS_READ : ST_SCAN_BYTES], tot);
    }
    __syncthreads();
    if (need_lens && lane_id() == 0) lens_blocks[s_off[warp][0]] = b;
    if (need_row && lane_id() == 0) row_blocks[s_off[warp][2]] = b;
    for (uint32_t k = lane_id(); k < ntiles; k += 32) { tile_block[s_off[warp][1] + k] = b; tile_off[s_off[warp][1] + k] = k * VL_TILE_BYTES; }
}

// ---- on-disk columns: header checks of the lens block (unmarshalUint64Items, encoding.go:246-336) once the device has regenerated it ----
// The uint block type byte sits right in front of the lens items (lens_off - 1).  status[0] = max error code.
static __global__ void k_finish_ondisk_cols(const uint8_t* __restrict__ arena, DevColumn* __restrict__ cols, const OndiskCol* __restrict__ oc, uint32_t n,
                                            unsigned long long* __restrict__ status) {
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    DevColumn& c = cols[oc[i].col];
    const uint64_t total = oc[i].lens_total, rows = oc[i].rows;
    unsigned err = 0;
    if (total < 1) err = 1;
    else {
        const uint8_t* p = arena + c.lens_off - 1;
        uint32_t lt = p[0];
        if (lt > 7) err = 2;
        else {
            uint64_t want = lt < 4 ? (rows << lt) : (1ull << (lt - 4));
            if (total - 1 != want) err = 3;
            else {
                c.lens_type = (uint8_t)lt;
                if (lt >= 4) {
                    uint64_t v = 0; for (uint64_t k = 0; k < want; k++) v = (v << 8) | p[1 + k];
                    if (v > 0xFFFFFFFFull) err = 4;
                    else { c.lens_const = (uint32_t)v; c.data_const = (rows >= 2 && c.data_len == v) ? 1 : 0; }   // encoding.go:113-120
                }
            }
        }
    }
    if (err) atomicMax(&status[0], (unsigned long long)err);
}

// ---- lens decode -> byte offset of every 8th row (unmarshalUint64Items + the offsets implied by encoding.go:122-130) --------------------
// row_off8[8 * w + g] = byte offset (within the block's data) of row 64 * (w - first word of the block) + 8 * g, for every bitmap word w of the
// block.  One warp per block of the lens work list, one lane per bitmap word.  Sums are taken in 64 bits: a lens block whose items do not add
// up to the data length (encoding.go:124-126) is reported, never wrapped into agreement.
static __global__ void k_lens_offsets(BatchView B, int slot, const uint32_t* __restrict__ lens_blocks, const uint32_t* __restrict__ work_count,
                               uint32_t* __restrict__ row_off8, uint8_t* __restrict__ ready, unsigned long long* __restrict__ stats, int wc_idx = WC_LENS) {
    // one WARP per block of the lens work list (a block of 2000..6400 rows has 32..100 bitmap words: a whole CTA per block left most of its
    // threads idle between barriers); lane = bitmap word, 32 words per step, the running sum travels in a register
    const uint32_t nwork = work_count[wc_idx];
    const uint32_t warps = (gridDim.x * blockDim.x) >> 5, lane = lane_id();
    for (uint32_t j = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; j < nwork; j += warps) {
        const uint32_t b = lens_blocks[j];
        if (ready[b]) continue;   // uniform per warp
        const DevColumn& c = B.cols[(uint64_t)b * B.nfields + slot];
        const uint32_t rows = B.blk_rows[b];
        const uint64_t w0 = B.blk_word_off[b]; const uint32_t nw = (uint32_t)(B.blk_word_off[b + 1] - w0);
        const uint8_t* lens = B.arena + c.lens_off;
        if (c.lens_type >= 4) {   // one const item: nothing to decode, the consumers divide
            if (lane == 0) {
                if ((unsigned long long)rows * c.lens_const != c.data_len) atomicMax(&stats[ST_ERROR], (unsigned long long)ERR_LENS_MISMATCH);
                ready[b] = 1;
            }
            continue;
        }
        unsigned long long carry = 0;
        for (uint32_t base = 0; base < nw; base += 32) {
            const uint32_t w = base + lane;
            uint32_t g[8] = {0, 0, 0, 0, 0, 0, 0, 0};
            unsigned long long sum = 0;
            if (w < nw) {
                const uint32_t r0 = w * 64, r1 = min(rows, r0 + 64);
                if (c.lens_type == 0) {
                    if (r1 - r0 == 64) {   // 64 u8 lens = four 16-byte vectors (r0 is a multiple of 64; lens_off is 16-byte aligned)
                        const uint4* v = (const uint4*)(lens + r0);
#pragma unroll
                        for (int q = 0; q < 4; q++) { uint4 x = v[q]; g[2 * q] = __vsadu4(x.x, 0) + __vsadu4(x.y, 0); g[2 * q + 1] = __vsadu4(x.z, 0) + __vsadu4(x.w, 0); }
                    } else for (uint32_t r = r0; r < r1; r++) g[(r - r0) >> 3] += lens[r];
#pragma unroll
                    for (int q = 0; q < 8; q++) sum += g[q];
                } else {
                    unsigned long long g64[8] = {0, 0, 0, 0, 0, 0, 0, 0};
                    for (uint32_t r = r0; r < r1; r++) g64[(r - r0) >> 3] += c.lens_type == 3 ? ld_be64(lens + 8 * (uint64_t)r) : (unsigned long long)row_len(c, lens, r);
#pragma unroll
                    for (int q = 0; q < 8; q++) { sum += g64[q]; g[q] = (uint32_t)min(g64[q], 0xFFFFFFFFull); }
                    if (sum > 0xFFFFFFFFull) sum = 0x100000000ull;   // cannot equal a data length (< 4 GiB); keeps the running sum from wrapping
                }
            }
            unsigned long long incl = sum;
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) { unsigned long long t = __shfl_up_sync(0xffffffffu, incl, d); if (lane >= d) incl += t; }
            const unsigned long long excl = carry + incl - sum;
            if (w < nw) {
                uint32_t o = (uint32_t)min(excl, 0xFFFFFFFFull);
                uint4 a, bq;
                a.x = o; o += g[0]; a.y = o; o += g[1]; a.z = o; o += g[2]; a.w = o; o += g[3];
                bq.x = o; o += g[4]; bq.y = o; o += g[5]; bq.z = o; o += g[6]; bq.w = o;
                uint4* dst = (uint4*)(row_off8 + ((w0 + w) << 3));
                dst[0] = a; dst[1] = bq;
            }
            carry += __shfl_sync(0xffffffffu, incl, 31);
        }
        if (lane == 0) {
            if (carry != c.data_len) atomicMax(&stats[ST_ERROR], (unsigned long long)ERR_LENS_MISMATCH);   // encoding.go:124-126
            ready[b] = 1;
        }
    }
}

// ---- the hot kernel: row-agnostic substring scan over the decoded strings payload -------------------------------------------------------
// Replaces bm.forEachSetBit(func(idx){ matchPhrase(values[idx], phrase) }) (filter_phrase.go:201-270, bitmap.go:128-153),
// matchPrefix (filter_prefix.go:318-352) and the strings.Index(literal) loop of regexutil (regex.go:162-212).
//
// Filter.  Every thread streams 16-byte vectors of the block's concatenated row bytes and looks only at ALIGNED 4-byte words.  An occurrence of
// the needle that starts at byte r (0..3) of some word leaves min(4 - r, L) of its bytes in that word and min(4, L - (4 - r)) in the next one;
// the host picks, per r, the word that carries more needle bytes and hands the kernel its (mask, pattern) pair and the distance `delta[r]` from
// that word back to the start of the occurrence.  A word of the stream that equals one of the four patterns under its mask is a candidate:
// <= 4 LOP3 + 4 ISETP per word, no funnel shifts, no bytes from the neighbour lane.  For needles of >= 7 bytes all four masks are full (every
// occurrence covers a whole aligned word) and the instantiation without masks is used.
//
// Verification.  Candidates are verified by the lane that found them, all lanes of a warp in parallel: full compare, byte offset -> row through
// row_off8 (interpolation guess, bracket check, binary search, then at most 8 lens items), rejection of occurrences that straddle a row, the
// boundary rules of the filter kind, atomicOr of the row's bit.  An occurrence in the reference's retry loop ("pos++; continue") is any
// occurrence, so occurrences are independent and order-free -- that is what makes the row-agnostic formulation exact.
struct ScanParams {
    uint32_t mode;            // SCAN_*
    uint32_t needle_off, needle_len;
    uint32_t pat[4], msk[4];  // per start alignment r: (word & msk[r]) == pat[r]
    int32_t delta[4];         // occurrence start = byte address of the matching word + delta[r]
    uint32_t nd16[4];         // the first 16 needle bytes (little-endian words), compared out of registers
    uint8_t starts_tok, ends_tok;
    int32_t regex;
};

static __device__ __forceinline__ uint32_t ld_u32_unaligned(const uint8_t* p) {   // two aligned loads + a funnel shift; reads up to 7 bytes past p
    const uint32_t* a = (const uint32_t*)((uintptr_t)p & ~(uintptr_t)3);
    return __funnelshift_r(a[0], a[1], 8 * (uint32_t)((uintptr_t)p & 3));
}

// Verification of one candidate occurrence at byte `pos` of block b's data by a single lane.
static __device__ __forceinline__ void scan_verify_lane(const DevProgram& P, const BatchView& B, const DevColumn& c, const ScanParams& sp, uint32_t b,
                                                     const uint32_t* __restrict__ row_off8, uint32_t pos, uint64_t* __restrict__ leaf_bm) {
    // everything the chain below depends on is requested up front: column header fields, the block's row count and first bitmap word
    const uint8_t* data = B.arena + c.data_off;
    const uint32_t L = sp.needle_len, n = (uint32_t)c.data_len;
    const uint32_t lens_type = c.lens_type, lens_const = c.lens_const;
    const uint8_t* lens = B.arena + c.lens_off;
    const uint32_t rows = B.blk_rows[b];
    const uint64_t w0 = B.blk_word_off[b];
    if ((uint64_t)pos + L > n) return;
    // the filter only vouches for some of the L bytes.  Payloads keep >= 32 readable bytes past data_len, so whole words may be compared.
    {
        const uint32_t head = L < 16 ? L : 16;
#pragma unroll
        for (uint32_t k = 0; k < 16; k += 4) {
            if (k >= head) break;
            const uint32_t m = head - k >= 4 ? 0xFFFFFFFFu : (1u << (8 * (head - k))) - 1;
            if ((ld_u32_unaligned(data + pos + k) ^ sp.nd16[k >> 2]) & m) return;
        }
        const uint8_t* nd = P.blob + sp.needle_off;
        for (uint32_t k = 16; k < L; k++) if (data[pos + k] != nd[k]) return;
    }
    // byte offset -> row
    uint32_t r, off, len;
    if (lens_type >= 4) {
        len = lens_const;
        if (len == 0) return;
        r = pos / len; off = r * len;
        if (r >= rows) return;
    } else {
        const uint32_t* ro = row_off8 + (w0 << 3);
        const uint32_t n8 = (rows + 7) >> 3;
        // last group of 8 rows that starts at or before pos.  Row lengths of one block are close to uniform, so pos * n8 / n is almost always
        // within one group of the answer: check that bracket first, fall back to the whole range.
        uint32_t lo, hi;
        {
            const uint32_t g = min((uint32_t)(__uint2float_rz(pos) * __fdividef(__uint2float_rz(n8), __uint2float_rz(n))), n8 - 1);
            lo = g ? g - 1 : 0; hi = min(g + 1, n8 - 1);
            if (!(ro[lo] <= pos && (hi + 1 >= n8 || ro[hi + 1] > pos))) { lo = 0; hi = n8 - 1; }
        }
        while (lo < hi) { const uint32_t mid = (lo + hi + 1) >> 1; if (ro[mid] <= pos) lo = mid; else hi = mid - 1; }
        // the row holding pos is the LAST row whose start is <= pos (zero-length rows share a start with their successor)
        const uint32_t r0 = lo * 8, kmax = min(8u, rows - r0);
        uint32_t o = ro[lo];
        r = r0; off = o; len = 0;
        if (lens_type == 0) {
            const uint2 lw = *(const uint2*)(lens + r0);   // r0 is a multiple of 8 and lens_off is 16-byte aligned
            const uint64_t l8 = ((uint64_t)lw.y << 32) | lw.x;
            for (uint32_t k = 0; k < kmax && o <= pos; k++) { const uint32_t l = (uint32_t)(l8 >> (8 * k)) & 0xFF; r = r0 + k; off = o; len = l; o += l; }
        } else {
            for (uint32_t k = 0; k < kmax && o <= pos; k++) { const uint32_t l = row_len(c, lens, r0 + k); r = r0 + k; off = o; len = l; o += l; }
        }
        if (pos < off || pos - off >= len) return;
    }
    if ((uint64_t)off + len > n) return;   // malformed lens (reported by k_lens_offsets): never read outside the payload
    if (pos + L > off + len) return;       // the occurrence straddles a row boundary
    const uint8_t* s = data + off; const uint32_t p = pos - off;
    bool hit;
    switch (sp.mode) {
    case SCAN_PHRASE: hit = phrase_boundaries_ok(s, len, p, L, sp.starts_tok, sp.ends_tok); break;
    case SCAN_PREFIX: hit = phrase_boundaries_ok(s, len, p, L, sp.starts_tok, false); break;
    case SCAN_CONTAINS: hit = true; break;
    case SCAN_RX_DOTPLUS: hit = p + L < len; break;
    case SCAN_RX_TAIL: {   // the needle is the literal of a `PREFIX.*LITERAL` expression: it matches iff PREFIX occurs entirely before this occurrence
        const DevRegex& R = P.regexes[sp.regex];
        hit = find_bytes(s, p, P.blob + R.prefix_off, R.prefix_len, 0) >= 0;
        break;
    }
    default: {             // SCAN_RX_SUFFIX: the needle is the literal prefix, the remainder of the row goes through the suffix automaton
        const DevRegex& R = P.regexes[sp.regex];
        if (R.tail_len) hit = find_bytes(s + p + L, len - p - L, P.blob + R.tail_off, R.tail_len, 0) >= 0;   // suffix `.*LIT`
        else hit = dfa_run(R, P.blob, s + p + L, len - p - L);
        break;
    }
    }
    if (hit) atomicOr((unsigned long long*)&leaf_bm[w0 + (r >> 6)], 1ull << (r & 63));
}

#define VL_SCAN_THREADS 256
#define VL_SCAN_UNROLL 4                       /* independent 16-byte loads in flight per thread */
#define VL_SCAN_ROUNDS 4                       /* rounds per tile */
#define VL_SCAN_QSTRIDE (VL_TILE_BYTES / VL_SCAN_UNROLL)                          /* distance between a thread's loads of one round */
static_assert(VL_TILE_BYTES == VL_SCAN_THREADS * 16 * VL_SCAN_UNROLL * VL_SCAN_ROUNDS, "tile size");

template <bool MASKED>
static __device__ __forceinline__ uint32_t scan_word_hits(uint32_t w, const ScanParams& sp) {   // bit r: the word matches pattern r
    if (MASKED) return (uint32_t)((w & sp.msk[0]) == sp.pat[0]) | (uint32_t)((w & sp.msk[1]) == sp.pat[1]) << 1 | (uint32_t)((w & sp.msk[2]) == sp.pat[2]) << 2 | (uint32_t)((w & sp.msk[3]) == sp.pat[3]) << 3;
    return (uint32_t)(w == sp.pat[0]) | (uint32_t)(w == sp.pat[1]) << 1 | (uint32_t)(w == sp.pat[2]) << 2 | (uint32_t)(w == sp.pat[3]) << 3;
}

// does any of the four words of v match one of the four (mask, pattern) pairs?  -> 0 / 1
template <bool MASKED>
static __device__ __forceinline__ uint32_t scan_vector_hit(const uint4& v, const ScanParams& sp) {
    uint32_t h;
    if (MASKED) {
        asm("{\n\t.reg .pred p;\n\t.reg .b32 t;\n\t"
            "lop3.b32 t, %1, %5, %9, 0x28;\n\tsetp.eq.u32 p, t, 0;\n\t"
            "lop3.b32 t, %1, %6, %10, 0x28;\n\tsetp.eq.or.u32 p, t, 0, p;\n\t"
            "lop3.b32 t, %1, %7, %11, 0x28;\n\tsetp.eq.or.u32 p, t, 0, p;\n\t"
            "lop3.b32 t, %1, %8, %12, 0x28;\n\tsetp.eq.or.u32 p, t, 0, p;\n\t"
            "lop3.b32 t, %2, %5, %9, 0x28;\n\tsetp.eq.or.u32 p, t, 0, p;\n\t"
            "lop3.b32 t, %2, %6, %10, 0x28;\n\tsetp.eq.or.u32 p, t, 0, p;\n\t"
            "lop3.b32 t, %2, %7, %11, 0x28;\n\tsetp.eq.or.u32 p, t, 0, p;\n\t"
            "lop3.b32 t, %2, %8, %12, 0x28;\n\tsetp.eq.or.u32 p, t, 0, p;\n\t"
            "lop3.b32 t, %3, %5, %9, 0x28;\n\tsetp.eq.or.u32 p, t, 0, p;\n\t"
            "lop3.b32 t, %3, %6, %10, 0x28;\n\tsetp.eq.or.u32 p, t, 0, p;\n\t"
            "lop3.b32 t, %3, %7, %11, 0x28;\n\tsetp.eq.or.u32 p, t, 0, p;\n\t"
            "lop3.b32 t, %3, %8, %12, 0x28;\n\tsetp.eq.or.u32 p, t, 0, p;\n\t"
            "lop3.b32 t, %4, %5, %9, 0x28;\n\tsetp.eq.or.u32 p, t, 0, p;\n\t"
            "lop3.b32 t, %4, %6, %10, 0x28;\n\tsetp.eq.or.u32 p, t, 0, p;\n\t"
            "lop3.b32 t, %4, %7, %11, 0x28;\n\tsetp.eq.or.u32 p, t, 0, p;\n\t"
            "lop3.b32 t, %4, %8, %12, 0x28;\n\tsetp.eq.or.u32 p, t, 0, p;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t}"
            : "=r"(h)
            : "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w), "r"(sp.pat[0]), "r"(sp.pat[1]), "r"(sp.pat[2]), "r"(sp.pat[3]), "r"(sp.msk[0]), "r"(sp.msk[1]), "r"(sp.msk[2]), "r"(sp.msk[3]));
    } else {
        asm("{\n\t.reg .pred p;\n\t"
            "setp.eq.u32 p, %1, %5;\n\tsetp.eq.or.u32 p, %1, %6, p;\n\tsetp.eq.or.u32 p, %1, %7, p;\n\tsetp.eq.or.u32 p, %1, %8, p;\n\t"
            "setp.eq.or.u32 p, %2, %5, p;\n\tsetp.eq.or.u32 p, %2, %6, p;\n\tsetp.eq.or.u32 p, %2, %7, p;\n\tsetp.eq.or.u32 p, %2, %8, p;\n\t"
            "setp.eq.or.u32 p, %3, %5, p;\n\tsetp.eq.or.u32 p, %3, %6, p;\n\tsetp.eq.or.u32 p, %3, %7, p;\n\tsetp.eq.or.u32 p, %3, %8, p;\n\t"
            "setp.eq.or.u32 p, %4, %5, p;\n\tsetp.eq.or.u32 p, %4, %6, p;\n\tsetp.eq.or.u32 p, %4, %7, p;\n\tsetp.eq.or.u32 p, %4, %8, p;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t}"
            : "=r"(h)
            : "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w), "r"(sp.pat[0]), "r"(sp.pat[1]), "r"(sp.pat[2]), "r"(sp.pat[3]));
    }
    return h;
}

// Candidates are not verified where they are found.  A lane whose 16-byte vector holds a candidate word appends (block, byte position of the
// VECTOR) to a queue in shared memory and goes on streaming; out of the queue, the CTA's 256 threads take one vector each, re-read it (it is
// still in L2), enumerate its candidate words / alignments and verify them.  Verifying in place costs a chain of ~6 dependent memory round trips
// (column header, row offsets, lens items, neighbouring bytes) during which the other 31 lanes of the warp wait; in the drain all lanes are
// busy and the chains overlap.  Round 2, second step: the streaming side used to enumerate the candidates itself (4 compares on each of a
// lane's 16 words, by every lane of a warp in which ANY lane had a hit): at selectivity 0.5 that enumeration was 43 % of all instructions of
// the kernel (profiles/kernel_history_r02.md).  Now it only ballots which lanes have a hit in each of their four vectors and reserves queue
// slots with one shared-memory atomic per vector index.  The queue is drained when a tile ends with at least VL_SCAN_QFLUSH entries, and when
// the CTA has run out of tiles.  A vector that finds the queue full is handled by its lane on the spot.
#define VL_SCAN_QCAP 2048
#define VL_SCAN_QFLUSH 192
struct ScanCand { uint32_t block, pos; };   // pos: byte offset of a 16-byte vector inside the block's data

// all candidates of one vector: word i matches pattern r => an occurrence may start at pos + 4 i + delta[r]
template <bool MASKED>
static __device__ __forceinline__ void scan_vector(const DevProgram& P, const BatchView& B, const DevColumn& c, const ScanParams& sp, uint32_t b,
                                                    const uint32_t* __restrict__ row_off8, uint32_t pos, uint64_t* __restrict__ leaf_bm) {
    const uint32_t n = (uint32_t)c.data_len;
    // vectors past the end of the data were streamed as zeros; a zero word can only match a pattern of NUL bytes, rejected by the bounds below
    const uint4 v = pos < n ? __ldg((const uint4*)(B.arena + c.data_off + pos)) : make_uint4(0, 0, 0, 0);
    // All candidates of the vector are collected first (bit 4 i + r: word i matches pattern r) and verified in ONE loop: with the verification
    // nested inside the loop over the words, the lanes of a draining warp - each with its candidate in a different word - took turns through four
    // copies of it, a quarter of the lanes at a time (ncu at 50 % candidate rows: 7.6 active lanes per instruction, 60 % of all instructions).
    uint32_t m = scan_word_hits<MASKED>(v.x, sp) | scan_word_hits<MASKED>(v.y, sp) << 4 | scan_word_hits<MASKED>(v.z, sp) << 8 | scan_word_hits<MASKED>(v.w, sp) << 12;
    while (m) {
        const int j = __ffs((int)m) - 1; m &= m - 1;
        const int64_t q = (int64_t)pos + (j & ~3) + sp.delta[j & 3];
        if (q < 0 || q + (int64_t)sp.needle_len > (int64_t)n) continue;
        scan_verify_lane(P, B, c, sp, b, row_off8, (uint32_t)q, leaf_bm);
    }
}

// One tile of the streaming side.  FULL: the tile lies wholly inside the data, so the four loads of a round go out without bounds predicates at
// immediate offsets from one pointer; otherwise (a block's last tile) every vector is checked against the end of the data and vectors past it
// are streamed as zeros.  INPLACE: candidates are verified where they are found instead of being queued (the re-scan of a tile whose
// candidates did not fit the queue).  Returns true when this lane had a candidate vector that found the queue full.
// The queueing code is inline on purpose: with a call inside the round loop ptxas parks the loop state (pointer, round counter, block) in local
// memory around every round (the call ABI pins most of the 48 registers), 6 local loads / stores per round.
template <bool MASKED, bool FULL, bool INPLACE>
static __device__ __forceinline__ bool scan_tile(const DevProgram& P, const BatchView& B, const DevColumn& c, const ScanParams& sp, uint32_t b,
                                                 const uint32_t* __restrict__ row_off8, uint64_t* __restrict__ leaf_bm, ScanCand* s_q, uint32_t* s_cnt, uint32_t tile0) {
    const uint32_t n = (uint32_t)c.data_len;           // < 4 GiB by construction (upload rejects larger payloads)
    const uint8_t* __restrict__ data = B.arena + c.data_off;
    const uint32_t lane = threadIdx.x & 31;
    bool overflow = false;
#pragma unroll 1
    for (int round = 0; round < VL_SCAN_ROUNDS; round++) {
        const uint32_t round0 = tile0 + (uint32_t)round * (VL_SCAN_THREADS * 16);
        if (!FULL && round0 >= n) break;                  // uniform: the whole round lies past the data
        const uint32_t base = round0 + threadIdx.x * 16;
        uint4 v[VL_SCAN_UNROLL];
        if (FULL) {
            const uint8_t* __restrict__ ptr = data + base;
#pragma unroll
            for (int u = 0; u < VL_SCAN_UNROLL; u++) v[u] = __ldg((const uint4*)(ptr + u * VL_SCAN_QSTRIDE));
        } else {
#pragma unroll
            for (int u = 0; u < VL_SCAN_UNROLL; u++) {
                const uint32_t p = base + u * VL_SCAN_QSTRIDE;
                // payloads keep >= 32 readable bytes past data_len: a vector load that starts before n is always in bounds
                v[u] = p < n ? __ldg((const uint4*)(data + p)) : make_uint4(0, 0, 0, 0);
            }
        }
        // bit u of `hits`: vector u holds a word equal to one of the four patterns (one predicate chain of 16 x setp.eq.or per vector)
        uint32_t hits = 0;
#pragma unroll
        for (int u = 0; u < VL_SCAN_UNROLL; u++) hits |= scan_vector_hit<MASKED>(v[u], sp) << u;
        if (!__any_sync(0xffffffffu, hits != 0)) continue;
        if (INPLACE) {
#pragma unroll 1
            for (int u = 0; u < VL_SCAN_UNROLL; u++) if (hits >> u & 1) scan_vector<MASKED>(P, B, c, sp, b, row_off8, base + u * VL_SCAN_QSTRIDE, leaf_bm);
            continue;
        }
        // some lane has a candidate: the whole warp reserves queue slots with ONE shared-memory atomic per round (lane 0 adds the number of
        // candidate vectors of all four vector indices); a lane's slot = the warp's base + the vectors of lower indices + those of lower lanes
        const uint32_t b0 = __ballot_sync(0xffffffffu, hits & 1), b1 = __ballot_sync(0xffffffffu, hits & 2), b2 = __ballot_sync(0xffffffffu, hits & 4), b3 = __ballot_sync(0xffffffffu, hits & 8);
        const uint32_t n0 = __popc(b0), n1 = n0 + __popc(b1), n2 = n1 + __popc(b2), n3 = n2 + __popc(b3);
        uint32_t at0 = 0;
        if (lane == 0) at0 = atomicAdd(s_cnt, n3);
        at0 = __shfl_sync(0xffffffffu, at0, 0);
        const uint32_t below = (1u << lane) - 1u;
        const uint32_t bal[4] = {b0, b1, b2, b3}, first[4] = {at0, at0 + n0, at0 + n1, at0 + n2};
#pragma unroll
        for (int u = 0; u < VL_SCAN_UNROLL; u++) {
            if (!(hits >> u & 1)) continue;
            const uint32_t at = first[u] + __popc(bal[u] & below);
            if (at < VL_SCAN_QCAP) s_q[at] = ScanCand{b, base + u * VL_SCAN_QSTRIDE}; else overflow = true;
        }
    }
    return overflow;
}
template <bool MASKED>
static __device__ __noinline__ bool scan_tail_tile(const DevProgram& P, const BatchView& B, const DevColumn& c, const ScanParams& sp, uint32_t b,
                                                   const uint32_t* __restrict__ row_off8, uint64_t* __restrict__ leaf_bm, ScanCand* s_q, uint32_t* s_cnt, uint32_t tile0) {
    return scan_tile<MASKED, false, false>(P, B, c, sp, b, row_off8, leaf_bm, s_q, s_cnt, tile0);
}
template <bool MASKED>
static __device__ __noinline__ void scan_tile_inplace(const DevProgram& P, const BatchView& B, const DevColumn& c, const ScanParams& sp, uint32_t b,
                                                      const uint32_t* __restrict__ row_off8, uint64_t* __restrict__ leaf_bm, uint32_t tile0) {
    scan_tile<MASKED, false, true>(P, B, c, sp, b, row_off8, leaf_bm, nullptr, nullptr, tile0);
}
template <bool MASKED>
static __device__ __noinline__ void scan_drain(const DevProgram& P, const BatchView& B, int slot, const ScanParams& sp, const uint32_t* __restrict__ row_off8,
                                               uint64_t* __restrict__ leaf_bm, const ScanCand* s_q, uint32_t count) {
    for (uint32_t i = threadIdx.x; i < count; i += blockDim.x) {
        const ScanCand e = s_q[i];
        scan_vector<MASKED>(P, B, B.cols[(uint64_t)e.block * B.nfields + slot], sp, e.block, row_off8, e.pos, leaf_bm);
    }
}

// Persistent grid: 148 SMs x 5 resident CTAs x 256 threads, each CTA strides over the tile table built by k_plan_leaf.  Per round a thread has
// four independent LDG.128 in flight, 16 KiB apart (a warp's requests spread over more L2 slices / HBM channels than adjacent 4 KiB slices would).
template <bool MASKED>
static __global__ void __launch_bounds__(VL_SCAN_THREADS, 5) k_substr_scan(const __grid_constant__ DevProgram P, const __grid_constant__ BatchView B, int slot, const __grid_constant__ ScanParams sp, const uint32_t* __restrict__ tile_block,
                                                                           const uint32_t* __restrict__ tile_off, const uint32_t* __restrict__ work_count,
                                                                           const uint32_t* __restrict__ row_off8, uint64_t* __restrict__ leaf_bm) {
    __shared__ ScanCand s_q[VL_SCAN_QCAP];
    __shared__ uint32_t s_cnt;
    if (threadIdx.x == 0) s_cnt = 0;
    __syncthreads();
    const uint32_t ntiles = work_count[WC_TILES];
    for (uint32_t t = blockIdx.x; t < ntiles; t += gridDim.x) {
        const uint32_t b = __ldg(tile_block + t), tile0 = __ldg(tile_off + t);
        const DevColumn& c = B.cols[(uint64_t)b * B.nfields + slot];
        bool overflow;
        if (tile0 + VL_TILE_BYTES <= (uint32_t)c.data_len) overflow = scan_tile<MASKED, true, false>(P, B, c, sp, b, row_off8, leaf_bm, s_q, &s_cnt, tile0);
        else overflow = scan_tail_tile<MASKED>(P, B, c, sp, b, row_off8, leaf_bm, s_q, &s_cnt, tile0);
        // end of the tile: drain the queue if it is worth a pass of the whole CTA (thread 0 decides; the barrier makes the decision uniform),
        // or if some candidate vector of this tile did not fit
        if (__syncthreads_or((threadIdx.x == 0 && s_cnt >= VL_SCAN_QFLUSH) || overflow)) {
            // candidates that did not fit were dropped: the tile is gone over again with verification in place (bits are OR-ed, so the
            // candidates that did make it into the queue and are verified again below change nothing)
            if (__syncthreads_or(overflow)) scan_tile_inplace<MASKED>(P, B, c, sp, b, row_off8, leaf_bm, tile0);
            scan_drain<MASKED>(P, B, slot, sp, row_off8, leaf_bm, s_q, min(s_cnt, (uint32_t)VL_SCAN_QCAP));
            __syncthreads();
            if (threadIdx.x == 0) s_cnt = 0;
            __syncthreads();
        }
    }
    __syncthreads();
    scan_drain<MASKED>(P, B, slot, sp, row_off8, leaf_bm, s_q, min(s_cnt, (uint32_t)VL_SCAN_QCAP));
}

// ---- dict LUT / fixed-width equality / typed in(): one thread per bitmap word ---------------------------------------------------------------
// matchEncodedValuesDict filter_phrase.go:272-289, matchBinaryValue filter_exact.go:356-364, matchAnyValue filter_in.go:187-200
static __global__ void k_word_match(DevProgram P, BatchView B, uint32_t leaf_idx, int slot, const uint8_t* __restrict__ action, const uint64_t* __restrict__ payload, const uint64_t* __restrict__ reg,
                             uint64_t* __restrict__ leaf_bm, unsigned long long* __restrict__ stats) {
    uint64_t gw = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (gw >= B.nwords) return;
    uint32_t b = B.word_block[gw];
    uint8_t act = action[b];
    if (act != ACT_DICT && act != ACT_FIXED_EQ && act != ACT_FIXED_IN) return;
    if (!reg[gw]) { leaf_bm[gw] = 0; return; }   // no selected row left in these 64 (bm.forEachSetBit visits none)
    const DevColumn& c = B.cols[(uint64_t)b * B.nfields + slot];
    const DevLeaf& L = P.leaves[leaf_idx];
    uint32_t rows = B.blk_rows[b];
    uint32_t r0 = (uint32_t)(gw - B.blk_word_off[b]) * 64, r1 = min(rows, r0 + 64);
    const uint8_t* data = B.arena + c.data_off;
    uint64_t bits = 0, pay = payload[b];
    if (act == ACT_DICT) {
        // dict ids: 1 byte per row; lens must be const 1 (or a per-row u8 block of ones for single-row blocks)
        bool bad = false;
        if (r1 - r0 == 64 && ((c.data_off + r0) & 15) == 0) {
            const uint4* v = (const uint4*)(data + r0);
#pragma unroll
            for (int q = 0; q < 4; q++) {
                uint4 x = __ldg(v + q); uint32_t ww[4] = {x.x, x.y, x.z, x.w};
#pragma unroll
                for (int i = 0; i < 4; i++)
#pragma unroll
                    for (int j = 0; j < 4; j++) { uint32_t id = (ww[i] >> (8 * j)) & 0xFF; bad |= id >= c.dict_len; bits |= (uint64_t)((pay >> (id & 7)) & 1) << (q * 16 + i * 4 + j); }
            }
        } else for (uint32_t r = r0; r < r1; r++) { uint32_t id = data[r]; bad |= id >= c.dict_len; bits |= (uint64_t)((pay >> (id & 7)) & 1) << (r - r0); }
        if (bad) atomicMax(&stats[ST_ERROR], (unsigned long long)ERR_DICT_INDEX);   // "too big index for dict value" filter_phrase.go:284-286
    } else {
        uint32_t w = width_of_vt(c.vt);
        for (uint32_t r = r0; r < r1; r++) {
            uint64_t v = load_fixed_be(data + (uint64_t)r * w, w);
            bool hit = act == ACT_FIXED_EQ ? v == pay : in_contains_typed(L, P.u64s, c.vt, v);
            bits |= (uint64_t)hit << (r - r0);
        }
    }
    leaf_bm[gw] = bits;
}

// ---- generic per-row matcher: one warp per bitmap word, lanes take rows l and l+32 ------------------------------------------------------------
// exact / in() / regexp-without-literal-prefix on string columns; numeric columns that must be formatted to text first.
// Persistent grid over the ACT_ROW work list of k_plan_leaf: work item j = block work_blocks[j]; its bitmap words are dealt out to the CTA's warps.
// The kernel is a chain of dependent loads per block and per bitmap word (work list -> column header -> register word -> lens -> row bytes), so it
// lives on resident warps: capped at 64 registers (4 CTAs per SM; the rarely taken predicates spill a little) it runs the `path:api*` leaf of C4
// in a quarter of the time it took with the 153 registers (1 CTA per SM) the compiler picks on its own.
static __global__ void __launch_bounds__(256, 4) k_row_match(DevProgram P, BatchView B, uint32_t leaf_idx, int slot, const uint32_t* __restrict__ work_blocks,
                                   const uint32_t* __restrict__ work_count, const uint8_t* __restrict__ action, const uint64_t* __restrict__ payload, const uint64_t* __restrict__ reg,
                                   const uint32_t* __restrict__ row_off8, uint64_t* __restrict__ leaf_bm) {
  if (work_count[WC_ROW] == 0) return;   // k_plan_leaf sent no block of the batch to the row matcher for this leaf
  const DevLeaf& L = P.leaves[leaf_idx];
  // Behind a selective filter of an AND chain most bitmap words are zero (like bm.forEachSetBit, bitmap.go:128-153, only rows that are still
  // selected are looked at).  A warp therefore reads 32 consecutive register words at once - one word per lane, coalesced - and goes through
  // the live ones among them one after the other; dead words cost 8 bytes of a coalesced load instead of a dependent round trip each.
  // (work_blocks, the block list, is not walked any more: the words of blocks with another action are dropped by the action test below.)
  const uint64_t nwarps = (uint64_t)gridDim.x * (blockDim.x >> 5), warp = (uint64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  for (uint64_t base = warp * 32; base < B.nwords; base += nwarps * 32) {
    uint64_t live_l = 0; uint32_t b_l = 0;
    if (base + lane_id() < B.nwords) {
        live_l = reg[base + lane_id()];
        if (live_l) { b_l = B.word_block[base + lane_id()]; const uint8_t a = action[b_l]; if (a < ACT_ROW || a > ACT_ROW_IN) live_l = 0; }
    }
    uint32_t todo = __ballot_sync(0xffffffffu, live_l != 0);
   while (todo) {
    const int src = __ffs((int)todo) - 1; todo &= todo - 1;
    const uint64_t gw = base + (uint32_t)src;
    const uint64_t live = __shfl_sync(0xffffffffu, live_l, src);
    const uint32_t b = __shfl_sync(0xffffffffu, b_l, src);
    const DevColumn& c = B.cols[(uint64_t)b * B.nfields + slot];
    const uint32_t rows = B.blk_rows[b];
    const uint8_t act = action[b]; const uint64_t pay = payload[b];
    const uint64_t w_lo = B.blk_word_off[b];
    uint32_t r0 = (uint32_t)(gw - w_lo) * 64;
    const uint8_t* data = B.arena + c.data_off;
    const uint8_t* lens = B.arena + c.lens_off;
    uint32_t la = 0, lb = 0;
    uint32_t ra = r0 + lane_id(), rb = r0 + 32 + lane_id();
    if (ra < rows) la = row_len(c, lens, ra);
    if (rb < rows) lb = row_len(c, lens, rb);
    // exclusive offsets: rows r0..r0+31 then r0+32..r0+63
    uint32_t ia = la, ib = lb;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) { uint32_t t = __shfl_up_sync(0xffffffffu, ia, d), u = __shfl_up_sync(0xffffffffu, ib, d); if (lane_id() >= d) { ia += t; ib += u; } }
    uint32_t tot_a = __shfl_sync(0xffffffffu, ia, 31);
    uint64_t base = c.lens_type >= 4 ? (uint64_t)r0 * c.lens_const : row_off8[gw << 3];
    uint64_t oa = base + ia - la, ob = base + tot_a + ib - lb;
    if (c.data_const) { oa = ob = 0; la = lb = (uint32_t)c.data_len; }   // every row = data (encoding.go:113-120)
    bool ha = false, hb = false;
    uint32_t vt = c.vt;
    auto eval = [&](uint64_t off, uint32_t len) -> bool {
        if (off + len > c.data_len) return false;   // malformed; k_lens_offsets reports the error
        const uint8_t* s = data + off;
        if (vt == VT_STRING) return leaf_match_string(P, L, s, len);
        uint32_t w = width_of_vt(vt);
        if (len != w) return false;
        uint64_t raw = load_fixed_be(s, w);
        if (act == ACT_ROW_EQ) return raw == pay;                              // matchBinaryValue filter_exact.go:356-364
        if (act == ACT_ROW_IN) return in_contains_typed(L, P.u64s, vt, raw);   // matchAnyValue filter_in.go:187-200
        if (L.kind == F_IPV4_RANGE) return raw >= L.aux0 && raw <= L.aux1;     // only ipv4 columns get here (k_plan_leaf)
        if (L.kind == F_RANGE) {
            switch (vt) {
            case VT_UINT8: case VT_UINT16: case VT_UINT32: case VT_UINT64: return raw >= L.rng_ulo && raw <= L.rng_uhi;
            case VT_INT64: { const int64_t v = unzigzag64(raw); return v >= L.rng_ilo && v <= L.rng_ihi; }
            case VT_FLOAT64: { const double f = __longlong_as_double((long long)raw); return f >= __longlong_as_double((long long)L.rng_fmin) && f <= __longlong_as_double((long long)L.rng_fmax); }
            case VT_IPV4: return raw >= L.rng_iplo && raw <= L.rng_iphi;
            default: return (int64_t)raw >= L.rng_ilo && (int64_t)raw <= L.rng_ihi;   // iso8601
            }
        }
        if (vt == VT_FLOAT64) return leaf_match_f64(P, L, raw);
        uint8_t buf[32];
        int n = encoded_to_string(vt, raw, buf);
        if (n < 0) return false;
        return leaf_match_typed_text(P, L, vt, buf, (uint32_t)n);
    };
    if (ra < rows && (live >> lane_id() & 1)) ha = eval(oa, la);
    if (rb < rows && (live >> (32 + lane_id()) & 1)) hb = eval(ob, lb);
    uint32_t lo = __ballot_sync(0xffffffffu, ha), hi = __ballot_sync(0xffffffffu, hb);
    if (lane_id() == 0) leaf_bm[gw] = ((uint64_t)hi << 32) | lo;
   }
  }
}

// ---- fold a leaf result into the running bitmap -------------------------------------------------------------------------------------------------
static __global__ void k_apply_leaf(BatchView B, const uint8_t* __restrict__ action, const uint64_t* __restrict__ leaf_bm, uint64_t* __restrict__ reg) {
    uint64_t gw = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (gw >= B.nwords) return;
    uint8_t act = action[B.word_block[gw]];
    if (act == ACT_ALL) return;
    reg[gw] = act == ACT_NONE ? 0 : (reg[gw] & leaf_bm[gw]);
}

// ---- finalize: per-block popcount (bitmap.onesCount bitmap.go:185-191 == blockResult.rowsLen) + totals -------------------------------------------
static __global__ void __launch_bounds__(256) k_finalize(BatchView B, const uint64_t* __restrict__ reg, uint32_t* __restrict__ counts, unsigned long long* __restrict__ stats,
                           unsigned long long* __restrict__ totals4) {
    __shared__ unsigned long long s_acc[8][4];   // per warp: rows, rows matched, blocks matched, bitmap bytes
    const uint32_t warp = threadIdx.x >> 5;
    const uint32_t b = blockIdx.x * 8 + warp;
    unsigned long long rows = 0, matched = 0, blocks = 0, bm_bytes = 0;
    if (b < B.nblocks) {
        uint64_t lo = B.blk_word_off[b], hi = B.blk_word_off[b + 1];
        uint32_t n = 0;
        for (uint64_t w = lo + lane_id(); w < hi; w += 32) n += __popcll(reg[w]);
#pragma unroll
        for (int d = 16; d; d >>= 1) n += __shfl_xor_sync(0xffffffffu, n, d);
        if (lane_id() == 0) counts[b] = n;
        rows = B.blk_rows[b];
        if (n) { matched = n; blocks = 1; bm_bytes = 8ull * (hi - lo); }
    }
    if (lane_id() == 0) { s_acc[warp][0] = rows; s_acc[warp][1] = matched; s_acc[warp][2] = blocks; s_acc[warp][3] = bm_bytes; }
    __syncthreads();
    if (threadIdx.x < 4) {   // one atomic per CTA and counter instead of six per block
        unsigned long long t = 0;
        for (int w = 0; w < 8; w++) t += s_acc[w][threadIdx.x];
        if (t) {
            if (threadIdx.x == 0) atomicAdd(&totals4[0], t);
            else if (threadIdx.x == 1) { atomicAdd(&stats[ST_ROWS_MATCHED], t); atomicAdd(&totals4[1], t); }
            else if (threadIdx.x == 2) { atomicAdd(&stats[ST_BLOCKS_MATCHED], t); atomicAdd(&totals4[2], t); }
            else atomicAdd(&stats[ST_BITMAP_BYTES], t);
        }
    }
}

// ---- hit-row offsets (bitmap.forEachSetBitReadonly bitmap.go:156-183) ----------------------------------------------------------------------------------
static __global__ void k_scan_counts(const uint32_t* __restrict__ counts, uint32_t n, uint64_t* __restrict__ offs) {   // single CTA exclusive scan
    __shared__ uint64_t s[1024];
    __shared__ uint64_t carry;
    if (threadIdx.x == 0) carry = 0;
    __syncthreads();
    for (uint32_t base = 0; base < n; base += blockDim.x) {
        uint32_t i = base + threadIdx.x;
        uint64_t v = i < n ? counts[i] : 0;
        s[threadIdx.x] = v;
        __syncthreads();
        for (uint32_t d = 1; d < blockDim.x; d <<= 1) { uint64_t a = threadIdx.x >= d ? s[threadIdx.x - d] : 0; __syncthreads(); s[threadIdx.x] += a; __syncthreads(); }
        if (i < n) offs[i] = carry + s[threadIdx.x] - v;
        __syncthreads();
        if (threadIdx.x == blockDim.x - 1) carry += s[threadIdx.x];
        __syncthreads();
    }
    if (threadIdx.x == 0) offs[n] = carry;
}
static __global__ void k_hits_compact(BatchView B, const uint64_t* __restrict__ reg, const uint64_t* __restrict__ offs, uint32_t* __restrict__ hits, uint64_t cap) {
    uint32_t b = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (b >= B.nblocks) return;
    uint64_t lo = B.blk_word_off[b], hi = B.blk_word_off[b + 1];
    uint64_t out = offs[b];
    for (uint64_t w0 = lo; w0 < hi; w0 += 32) {
        uint64_t w = w0 + lane_id();
        uint64_t bits = w < hi ? reg[w] : 0;
        uint32_t n = __popcll(bits), incl = n;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) { uint32_t t = __shfl_up_sync(0xffffffffu, incl, d); if (lane_id() >= d) incl += t; }
        uint64_t pos = out + incl - n;
        uint32_t rbase = (uint32_t)(w - lo) * 64;
        while (bits) { int k = __ffsll((long long)bits) - 1; bits &= bits - 1; if (pos < cap) hits[pos] = rbase + k; pos++; }
        out += __shfl_sync(0xffffffffu, incl, 31);
    }
}

// ---- timestamps column: encoding.UnmarshalTimestamps on the device (vm/lib/encoding/encoding.go:173-250, nearest_delta2.go:57-90, ------------
// nearest_delta.go, int.go:173-280) and filterTime (lib/logstorage/filter_time.go:114-137) ------------------------------------------------------
// One CTA per block.  The sequential decoder becomes three data-parallel steps (tests/test_timestamps_model_cpu.py proves them equal to it,
// malformed input included): (1) a byte ends a varint iff its continuation bit is clear, so the index of a varint is the number of such bytes in
// front of it (ballot + popcount, CTA running sum) and every varint is assembled from its <= 10 bytes independently; (2) NearestDelta: values =
// first + inclusive scan of the deltas; NearestDelta2: one more inclusive scan in front (deltas of deltas -> deltas), all sums mod 2^64 like Go's
// int64; (3) DeltaConst / Const need no scan.  vals[0 .. rows) receives the timestamps.  Returns false (CTA-uniform) on malformed input:
// a varint longer than 10 bytes or overflowing 64 bits, too few / too many varints, bytes left over.
static __device__ unsigned long long cta_incl_scan_u64(unsigned long long v, unsigned long long* s_warp, unsigned long long* s_carry) {   // all threads of the CTA; carries across calls
    unsigned long long incl = v;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) { unsigned long long t = __shfl_up_sync(0xffffffffu, incl, d); if (lane_id() >= d) incl += t; }
    const uint32_t wid = threadIdx.x >> 5, nw = blockDim.x >> 5;
    if (lane_id() == 31) s_warp[wid] = incl;
    __syncthreads();
    unsigned long long pre = *s_carry;
    for (uint32_t k = 0; k < wid; k++) pre += s_warp[k];
    unsigned long long tot = 0;
    for (uint32_t k = 0; k < nw; k++) tot += s_warp[k];
    __syncthreads();
    if (threadIdx.x == 0) *s_carry += tot;
    __syncthreads();
    return pre + incl;
}
static __device__ bool ts_decode_block(const BatchView& B, uint32_t b, unsigned long long* __restrict__ vals) {
    __shared__ unsigned long long s_warp[32];
    __shared__ unsigned long long s_carry;
    __shared__ uint32_t s_cnt[32];
    __shared__ uint32_t s_ccarry;
    __shared__ int s_bad;
    const DevTimestamps t = B.ts[b];
    const uint32_t R = B.blk_rows[b], len = t.len;
    const uint8_t* raw = B.arena + t.off;
    const unsigned long long first = (unsigned long long)t.first;
    if (threadIdx.x == 0) { s_bad = 0; s_ccarry = 0; s_carry = 0; }
    __syncthreads();
    if (t.mt == MT_CONST) {
        for (uint32_t r = threadIdx.x; r < R; r += blockDim.x) vals[r] = first;
        return len == 0;
    }
    if (t.mt == MT_DELTA_CONST) {
        unsigned long long u = 0; bool ok = len >= 1 && len <= 10;
        if (ok) { for (uint32_t k = 0; k < len; k++) { const uint8_t c = raw[k]; if ((k + 1 < len) != (c >= 0x80)) ok = false; u |= (unsigned long long)(c & 0x7F) << (7 * k); } if (len == 10 && raw[9] > 1) ok = false; }
        const unsigned long long d = (u >> 1) ^ (0ull - (u & 1));
        for (uint32_t r = threadIdx.x; r < R; r += blockDim.x) vals[r] = first + (unsigned long long)r * d;
        return ok;
    }
    if (t.mt != MT_NEAREST_DELTA && t.mt != MT_NEAREST_DELTA2) return false;
    const uint32_t min_rows = t.mt == MT_NEAREST_DELTA2 ? 2u : 1u;
    if (R < min_rows) return false;
    const uint32_t need = R - 1;   // NearestDelta: one delta per row after the first; NearestDelta2: the first delta, then R - 2 deltas of deltas
    // (1) varints
    for (uint32_t base = 0; base < len; base += blockDim.x) {
        const uint32_t i = base + threadIdx.x;
        const uint8_t c = i < len ? raw[i] : 0x80;
        const bool is_end = i < len && c < 0x80;
        const uint32_t m = __ballot_sync(0xffffffffu, is_end);
        if (lane_id() == 0) s_cnt[threadIdx.x >> 5] = __popc(m);
        __syncthreads();
        uint32_t k = s_ccarry + __popc(m & ((1u << lane_id()) - 1));
        for (uint32_t w = 0; w < (threadIdx.x >> 5); w++) k += s_cnt[w];
        if (is_end) {
            uint32_t s0 = i, n = 1;
            while (s0 > 0 && raw[s0 - 1] >= 0x80 && n <= 10) { s0--; n++; }
            unsigned long long u = 0;
            for (uint32_t q = 0; q < n && q < 10; q++) u |= (unsigned long long)(raw[s0 + q] & 0x7F) << (7 * q);
            if (n > 10 || (n == 10 && c > 1) || k >= need) s_bad = 1;
            else vals[1 + k] = (u >> 1) ^ (0ull - (u & 1));
        }
        __syncthreads();
        if (threadIdx.x == 0) { uint32_t tot = 0; for (uint32_t w = 0; w < (blockDim.x >> 5); w++) tot += s_cnt[w]; s_ccarry += tot; }
        __syncthreads();
    }
    if (threadIdx.x == 0 && (s_ccarry != need || (len > 0 && raw[len - 1] >= 0x80))) s_bad = 1;
    __syncthreads();
    if (s_bad) return false;
    // (2) prefix sums, in place
    for (int pass = t.mt == MT_NEAREST_DELTA2 ? 0 : 1; pass < 2; pass++) {
        if (threadIdx.x == 0) s_carry = pass == 1 ? first : 0;
        __syncthreads();
        for (uint32_t base = 0; base < need; base += blockDim.x) {
            const uint32_t i = base + threadIdx.x;
            const unsigned long long v = i < need ? vals[1 + i] : 0;
            const unsigned long long sum = cta_incl_scan_u64(v, s_warp, &s_carry);
            if (i < need) vals[1 + i] = sum;
        }
        __syncthreads();
    }
    if (threadIdx.x == 0) vals[0] = first;
    __syncthreads();
    return true;
}

// _time filter on the blocks it only partly covers (the ACT_TIME work list of k_plan_leaf): decode, compare, one 32-bit half of a bitmap word per warp
static __global__ void __launch_bounds__(256) k_time_match(BatchView B, long long mn, long long mx, const uint32_t* __restrict__ row_blocks, const uint32_t* __restrict__ work_count,
                                                            unsigned long long* __restrict__ ts_vals, uint64_t* __restrict__ leaf_bm, unsigned long long* __restrict__ stats) {
    const uint32_t nwork = work_count[WC_ROW];
    for (uint32_t j = blockIdx.x; j < nwork; j += gridDim.x) {
        const uint32_t b = row_blocks[j], R = B.blk_rows[b];
        const uint64_t w0 = B.blk_word_off[b];
        unsigned long long* vals = ts_vals + w0 * 64;
        const bool ok = ts_decode_block(B, b, vals);
        if (!ok && threadIdx.x == 0) atomicMax(&stats[ST_ERROR], (unsigned long long)ERR_BAD_TIMESTAMPS);
        const uint32_t rows_padded = (R + 63) / 64 * 64;
        for (uint32_t base = 0; base < rows_padded; base += blockDim.x) {
            const uint32_t r = base + threadIdx.x;
            const long long v = r < R ? (long long)vals[r] : 0;
            const uint32_t m = __ballot_sync(0xffffffffu, ok && r < R && v >= mn && v <= mx);
            if (lane_id() == 0 && r < rows_padded) ((uint32_t*)(leaf_bm + w0))[r >> 5] = m;   // little-endian halves of the 64-bit words
        }
        __syncthreads();
    }
}

// ---- hit materialisation: the selected rows' values and timestamps as blockResult would yield them -------------------------------------------
// (lib/logstorage/block_result.go:491-507 initTimestampsInternal, :529-591 the per-type readers behind getValues; values_encoder.go:1367-1422)
// hit h = (hit_block[h], hit_row[h]) in block order, rows ascending (k_hits_compact2).
static __global__ void k_hits_compact2(BatchView B, const uint64_t* __restrict__ reg, const uint64_t* __restrict__ offs, uint32_t* __restrict__ hits, uint32_t* __restrict__ hit_block, uint64_t cap) {
    uint32_t b = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (b >= B.nblocks) return;
    uint64_t lo = B.blk_word_off[b], hi = B.blk_word_off[b + 1];
    uint64_t out = offs[b];
    for (uint64_t w0 = lo; w0 < hi; w0 += 32) {
        uint64_t w = w0 + lane_id();
        uint64_t bits = w < hi ? reg[w] : 0;
        uint32_t n = __popcll(bits), incl = n;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) { uint32_t t = __shfl_up_sync(0xffffffffu, incl, d); if (lane_id() >= d) incl += t; }
        uint64_t pos = out + incl - n;
        uint32_t rbase = (uint32_t)(w - lo) * 64;
        while (bits) { int k = __ffsll((long long)bits) - 1; bits &= bits - 1; if (pos < cap) { hits[pos] = rbase + k; hit_block[pos] = b; } pos++; }
        out += __shfl_sync(0xffffffffu, incl, 31);
    }
}
// blocks with hits -> work list: mode 0 = into the lens list those whose column `slot` is a strings column with per-row lens items, mode 1 = into
// the row list every block with hits (timestamps decode)
static __global__ void k_hit_blocks_list(BatchView B, const uint32_t* __restrict__ counts, int slot, int mode, uint32_t* __restrict__ list, uint32_t* __restrict__ work_count) {
    const uint32_t b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= B.nblocks || counts[b] == 0) return;
    if (mode == 0) {
        if (slot < 0) return;
        const DevColumn& c = B.cols[(uint64_t)b * B.nfields + slot];
        if (c.kind != COL_VALUES || c.vt != VT_STRING || c.lens_type >= 4 || c.data_const) return;
        list[atomicAdd(&work_count[WC_LENS], 1u)] = b;
    } else list[atomicAdd(&work_count[WC_ROW], 1u)] = b;
}
static __global__ void __launch_bounds__(256) k_ts_decode_list(BatchView B, const uint32_t* __restrict__ row_blocks, const uint32_t* __restrict__ work_count,
                                                                unsigned long long* __restrict__ ts_vals, unsigned long long* __restrict__ stats) {
    const uint32_t nwork = work_count[WC_ROW];
    for (uint32_t j = blockIdx.x; j < nwork; j += gridDim.x) {
        const uint32_t b = row_blocks[j];
        const bool ok = B.ts && B.ts[b].mt && ts_decode_block(B, b, ts_vals + B.blk_word_off[b] * 64);
        if (!ok && threadIdx.x == 0) atomicMax(&stats[ST_ERROR], (unsigned long long)(B.ts && B.ts[b].mt ? ERR_BAD_TIMESTAMPS : ERR_NO_TIMESTAMPS));
        __syncthreads();
    }
}
static __global__ void k_gather_ts(BatchView B, const uint32_t* __restrict__ hits, const uint32_t* __restrict__ hit_block, uint64_t nhits, const unsigned long long* __restrict__ ts_vals,
                                   long long* __restrict__ out) {
    const uint64_t h = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (h < nhits) out[h] = (long long)ts_vals[B.blk_word_off[hit_block[h]] * 64 + hits[h]];
}
// The value of column `slot` in one row as a string.  pass 0: lens[h] = its length; pass 1: the bytes go to out + offs[h].
static __global__ void k_gather_values(BatchView B, int slot, const uint32_t* __restrict__ hits, const uint32_t* __restrict__ hit_block, uint64_t nhits, const uint32_t* __restrict__ row_off8,
                                       int pass, uint32_t* __restrict__ lens_out, const uint64_t* __restrict__ offs, uint8_t* __restrict__ out, unsigned long long* __restrict__ stats) {
    const uint64_t h = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (h >= nhits) return;
    const uint32_t b = hit_block[h], r = hits[h];
    const uint8_t* src = nullptr; uint32_t len = 0;
    uint8_t buf[VL_FMT_F64_MAX];
    if (slot >= 0) {
        const DevColumn& c = B.cols[(uint64_t)b * B.nfields + slot];
        if (c.kind == COL_CONST) { src = B.hdr + c.meta_off; len = c.meta_len; }
        else if (c.kind == COL_VALUES) {
            const uint8_t* data = B.arena + c.data_off;
            if (c.vt == VT_STRING) {
                if (c.data_const) { src = data; len = (uint32_t)c.data_len; }
                else if (c.lens_type >= 4) { len = c.lens_const; src = data + (uint64_t)r * len; }
                else {
                    const uint8_t* lens = B.arena + c.lens_off;
                    uint32_t o = row_off8[(B.blk_word_off[b] << 3) + (r >> 3)];
                    for (uint32_t q = r & ~7u; q < r; q++) o += row_len(c, lens, q);
                    len = row_len(c, lens, r); src = data + o;
                }
                if ((uint64_t)(src - data) + len > c.data_len) { len = 0; atomicMax(&stats[ST_ERROR], (unsigned long long)ERR_LENS_MISMATCH); }
            } else if (c.vt == VT_DICT) {
                const uint32_t id = data[r];
                if (id >= c.dict_len) atomicMax(&stats[ST_ERROR], (unsigned long long)ERR_DICT_INDEX);
                else { const uint32_t* dof = (const uint32_t*)(B.hdr + c.meta_off); src = B.hdr + c.meta_off + 4 * (c.dict_len + 1) + dof[id]; len = dof[id + 1] - dof[id]; }
            } else {
                const uint32_t w = width_of_vt(c.vt);
                const uint64_t raw = load_fixed_be(data + (uint64_t)r * w, w);
                const int n = c.vt == VT_FLOAT64 ? fmt_f64(buf, raw) : encoded_to_string(c.vt, raw, buf);
                src = buf; len = n > 0 ? (uint32_t)n : 0;
            }
        }
    }
    if (pass == 0) { lens_out[h] = len; return; }
    uint8_t* d = out + offs[h];
    for (uint32_t k = 0; k < len; k++) d[k] = src[k];
}
// exclusive scan of u32 lengths into u64 offsets (offs[n] = total): tile sums, scan of the tile sums by one CTA, per-tile prefixes
#define VL_SCAN_TILE 2048
static __global__ void __launch_bounds__(256) k_scan_tiles(const uint32_t* __restrict__ v, uint64_t n, unsigned long long* __restrict__ tile_sums, unsigned long long* __restrict__ offs, int pass) {
    __shared__ unsigned long long s_w[8];
    const uint64_t base = (uint64_t)blockIdx.x * VL_SCAN_TILE + (uint64_t)threadIdx.x * 8;
    unsigned long long x[8], sum = 0;
#pragma unroll
    for (int k = 0; k < 8; k++) { x[k] = base + k < n ? v[base + k] : 0; sum += x[k]; }
    unsigned long long incl = sum;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) { unsigned long long t = __shfl_up_sync(0xffffffffu, incl, d); if (lane_id() >= d) incl += t; }
    if (lane_id() == 31) s_w[threadIdx.x >> 5] = incl;
    __syncthreads();
    unsigned long long pre = 0, tot = 0;
    for (uint32_t k = 0; k < 8; k++) { if (k < (threadIdx.x >> 5)) pre += s_w[k]; tot += s_w[k]; }
    if (pass == 0) { if (threadIdx.x == 0) tile_sums[blockIdx.x] = tot; return; }
    unsigned long long o = tile_sums[blockIdx.x] + pre + incl - sum;
#pragma unroll
    for (int k = 0; k < 8; k++) { if (base + k < n) offs[base + k] = o; o += x[k]; }
}
static __global__ void k_scan_tile_sums(unsigned long long* __restrict__ tile_sums, uint64_t ntiles, unsigned long long* __restrict__ total) {   // single CTA, exclusive, in place
    __shared__ unsigned long long s[1024];
    __shared__ unsigned long long carry;
    if (threadIdx.x == 0) carry = 0;
    __syncthreads();
    for (uint64_t base = 0; base < ntiles; base += blockDim.x) {
        const uint64_t i = base + threadIdx.x;
        const unsigned long long v = i < ntiles ? tile_sums[i] : 0;
        s[threadIdx.x] = v;
        __syncthreads();
        for (uint32_t d = 1; d < blockDim.x; d <<= 1) { unsigned long long a = threadIdx.x >= d ? s[threadIdx.x - d] : 0; __syncthreads(); s[threadIdx.x] += a; __syncthreads(); }
        if (i < ntiles) tile_sums[i] = carry + s[threadIdx.x] - v;
        __syncthreads();
        if (threadIdx.x == blockDim.x - 1) carry += s[threadIdx.x];
        __syncthreads();
    }
    if (threadIdx.x == 0) *total = carry;
}

// ---- two-column leaves: eq_field(), le_field() / lt_field() (filter_eq_field.go:60-237, filter_le_field.go:93-313) -------------------------------
// the encoded bytes of row r of a values column (strings: the row; typed: the fixed-width value; dict: the id byte); false when the lens items are off
static __device__ bool row_bytes(const BatchView& B, const DevColumn& c, uint32_t b, uint32_t r, const uint32_t* __restrict__ row_off8, const uint8_t** p, uint32_t* n) {
    const uint8_t* data = B.arena + c.data_off;
    if (c.data_const) { *p = data; *n = (uint32_t)c.data_len; return true; }
    uint64_t off; uint32_t len;
    if (c.lens_type >= 4) { len = c.lens_const; off = (uint64_t)r * len; }
    else {
        const uint8_t* lens = B.arena + c.lens_off;
        uint32_t o = row_off8[(B.blk_word_off[b] << 3) + (r >> 3)];
        for (uint32_t q = r & ~7u; q < r; q++) o += row_len(c, lens, q);
        off = o; len = row_len(c, lens, r);
    }
    if (off + len > c.data_len) return false;
    *p = data + off; *n = len;
    return true;
}
// the string form of a row's value as blockResult.getValues yields it: const value, "" for a missing field, dict entry, row bytes, text of a typed value
static __device__ bool row_string(const BatchView& B, const DevColumn* c, uint32_t b, uint32_t r, const uint32_t* __restrict__ row_off8, uint8_t* buf, const uint8_t** p, uint32_t* n) {
    *p = buf; *n = 0;
    if (!c || c->kind == COL_MISSING) return true;
    if (c->kind == COL_CONST) { *p = B.hdr + c->meta_off; *n = c->meta_len; return true; }
    const uint8_t* v; uint32_t vn;
    if (!row_bytes(B, *c, b, r, row_off8, &v, &vn)) return false;
    if (c->vt == VT_STRING) { *p = v; *n = vn; return true; }
    if (c->vt == VT_DICT) {
        if (vn != 1 || v[0] >= c->dict_len) return false;
        const uint32_t* dof = (const uint32_t*)(B.hdr + c->meta_off);
        *p = B.hdr + c->meta_off + 4 * (c->dict_len + 1) + dof[v[0]]; *n = dof[v[0] + 1] - dof[v[0]];
        return true;
    }
    if (vn != width_of_vt(c->vt)) return false;
    const uint64_t raw = load_fixed_be(v, vn);
    const int k = c->vt == VT_FLOAT64 ? fmt_f64(buf, raw) : encoded_to_string(c->vt, raw, buf);
    *n = k > 0 ? (uint32_t)k : 0;
    return true;
}
// leValuesString filter_le_field.go:283-297: numbers when both sides are numbers, else strings (bytewise, the shorter first on a tie)
static __device__ bool le_values_string(const uint8_t* a, uint32_t an, const uint8_t* b2, uint32_t bn, bool excl) {
    const double fa = mn::parse_math_number(a, an);
    if (fa == fa) { const double fb = mn::parse_math_number(b2, bn); if (fb == fb) return excl ? fa < fb : fa <= fb; }
    const uint32_t m = an < bn ? an : bn;
    int cmp = 0;
    for (uint32_t i = 0; i < m && !cmp; i++) cmp = (int)a[i] - (int)b2[i];
    if (!cmp) cmp = an < bn ? -1 : an > bn ? 1 : 0;
    return excl ? cmp < 0 : cmp <= 0;
}
// header-level decisions of a two-column leaf; one warp per block (lane 0 decides), work lists like k_plan_leaf
static __global__ void __launch_bounds__(256) k_plan_pair(DevProgram P, BatchView B, uint32_t leaf_idx, int slot_a, int slot_b, const uint64_t* __restrict__ reg, uint8_t* __restrict__ action,
                                                           uint64_t* __restrict__ payload, uint32_t* __restrict__ lens_a, uint32_t* __restrict__ lens_b, uint32_t* __restrict__ row_blocks,
                                                           uint32_t* __restrict__ work_count, unsigned long long* __restrict__ stats, uint8_t* __restrict__ need = nullptr) {
    // need != NULL: probe pass of a bloom-first upload (see k_plan_leaf): marks the values columns the row kernel would read, writes nothing else
    const uint32_t b = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (b >= B.nblocks) return;
    const DevLeaf& L = P.leaves[leaf_idx];
    const bool alive = block_alive_warp(reg, B, b);
    if (lane_id() != 0) return;
    uint8_t act = ACT_NONE; uint64_t mode = PAIR_STRINGS;
    if (alive && !L.always_none) {
        const bool le = L.kind == F_LE_FIELD, excl = L.pair_excl != 0;
        const DevColumn* ca = slot_a >= 0 ? &B.cols[(uint64_t)b * B.nfields + slot_a] : nullptr;
        const DevColumn* cb = slot_b >= 0 ? &B.cols[(uint64_t)b * B.nfields + slot_b] : nullptr;
        const int ka = ca ? ca->kind : COL_MISSING, kb = cb ? cb->kind : COL_MISSING;
        // a const column with an empty value is no column at all for getConstColumnValue (block_search.go:232-276 returns "" for both)
        const bool consta = ka == COL_CONST && ca->meta_len > 0, constb = kb == COL_CONST && cb->meta_len > 0;
        const bool vala = ka == COL_VALUES, valb = kb == COL_VALUES;
        if (consta && constb) {
            const uint8_t* x = B.hdr + ca->meta_off; const uint8_t* y = B.hdr + cb->meta_off;
            const bool m = le ? le_values_string(x, ca->meta_len, y, cb->meta_len, excl) : bytes_equal(x, ca->meta_len, y, cb->meta_len);
            act = m ? ACT_ALL : ACT_NONE;
        } else if (consta || constb) act = ACT_PAIR;                                      // one const: row strings
        else if (!vala && !valb) act = (le && excl) ? ACT_NONE : ACT_ALL;                  // both fields missing: "" against ""
        else if (!vala || !valb) act = ACT_PAIR;                                          // one missing: row strings
        else if (ca->vt != cb->vt || ca->vt == VT_STRING) act = ACT_PAIR;
        else { act = ACT_PAIR; mode = ca->vt == VT_DICT ? PAIR_DICT : PAIR_BINARY; }
        if (act == ACT_PAIR && need) {
            if (vala) need[(uint64_t)b * B.nfields + slot_a] = 1;
            if (valb) need[(uint64_t)b * B.nfields + slot_b] = 1;
            return;
        }
        if (act == ACT_PAIR && ((vala && ca->values_state != VALUES_STAGED) || (valb && cb->values_state != VALUES_STAGED))) {
            atomicMax(&stats[ST_ERROR], (unsigned long long)ERR_VALUES_ABSENT); act = ACT_NONE;
        }
        if (act == ACT_PAIR) {
            unsigned long long vb = 0, cols = 0;
            if (vala) { vb += lens_stored_bytes(*ca, B.blk_rows[b]) + ca->data_len; cols++; if (ca->lens_type < 4 && !ca->data_const) lens_a[atomicAdd(&work_count[WC_LENS], 1u)] = b; }
            if (valb) { vb += lens_stored_bytes(*cb, B.blk_rows[b]) + cb->data_len; cols++; if (cb->lens_type < 4 && !cb->data_const) lens_b[atomicAdd(&work_count[WC_LENS2], 1u)] = b; }
            row_blocks[atomicAdd(&work_count[WC_ROW], 1u)] = b;
            atomicAdd(&stats[ST_VALUES_BYTES], vb); atomicAdd(&stats[ST_COLUMNS_READ], cols);
        }
    }
    if (need) return;
    action[b] = act; payload[b] = mode;
}
static __device__ __noinline__ bool pair_match_row(const DevProgram& P, const BatchView& B, const DevLeaf& L, const DevColumn* ca, const DevColumn* cb, uint32_t b, uint32_t r, uint32_t mode,
                                                   const uint32_t* __restrict__ ro_a, const uint32_t* __restrict__ ro_b, unsigned long long* __restrict__ stats) {
    const bool le = L.kind == F_LE_FIELD, excl = L.pair_excl != 0;
    const uint8_t *x, *y; uint32_t xn, yn;
    if (mode == PAIR_BINARY) {
        if (!row_bytes(B, *ca, b, r, ro_a, &x, &xn) || !row_bytes(B, *cb, b, r, ro_b, &y, &yn)) { atomicMax(&stats[ST_ERROR], (unsigned long long)ERR_LENS_MISMATCH); return false; }
        if (!le) return bytes_equal(x, xn, y, yn);                                        // applyFilterBinValue: same type, same binary form
        if (ca->vt == VT_INT64 && xn == 8 && yn == 8) { const int64_t u = unzigzag64(ld_be64(x)), v = unzigzag64(ld_be64(y)); return excl ? u < v : u <= v; }
        if (ca->vt == VT_FLOAT64 && xn == 8 && yn == 8) { const double u = __longlong_as_double((long long)ld_be64(x)), v = __longlong_as_double((long long)ld_be64(y)); return excl ? u < v : u <= v; }
        return le_values_string(x, xn, y, yn, excl);   // uintN, ipv4, iso8601: their big-endian encodings go through leValuesString as they are (:246-252)
    }
    uint8_t bufa[VL_FMT_F64_MAX], bufb[VL_FMT_F64_MAX];
    if (!row_string(B, ca, b, r, ro_a, bufa, &x, &xn) || !row_string(B, cb, b, r, ro_b, bufb, &y, &yn)) { atomicMax(&stats[ST_ERROR], (unsigned long long)ERR_DICT_INDEX); return false; }
    return le ? le_values_string(x, xn, y, yn, excl) : bytes_equal(x, xn, y, yn);   // PAIR_DICT compares the entries, PAIR_STRINGS the string forms: same code
}
static __global__ void __launch_bounds__(256) k_row_pair(DevProgram P, BatchView B, uint32_t leaf_idx, int slot_a, int slot_b, const uint32_t* __restrict__ row_blocks, const uint32_t* __restrict__ work_count,
                                                          const uint64_t* __restrict__ payload, const uint64_t* __restrict__ reg, const uint32_t* __restrict__ ro_a, const uint32_t* __restrict__ ro_b,
                                                          uint64_t* __restrict__ leaf_bm, unsigned long long* __restrict__ stats) {
    const uint32_t nwork = work_count[WC_ROW];
    const DevLeaf& L = P.leaves[leaf_idx];
    for (uint32_t j = blockIdx.x; j < nwork; j += gridDim.x) {
        const uint32_t b = row_blocks[j], rows = B.blk_rows[b], mode = (uint32_t)payload[b];
        const DevColumn* ca = slot_a >= 0 ? &B.cols[(uint64_t)b * B.nfields + slot_a] : nullptr;
        const DevColumn* cb = slot_b >= 0 ? &B.cols[(uint64_t)b * B.nfields + slot_b] : nullptr;
        const uint64_t w_lo = B.blk_word_off[b], w_hi = B.blk_word_off[b + 1];
        for (uint64_t gw = w_lo + (threadIdx.x >> 5); gw < w_hi; gw += blockDim.x >> 5) {
            const uint64_t live = reg[gw];   // only rows that are still selected (bm.forEachSetBit)
            if (!live) { if (lane_id() == 0) leaf_bm[gw] = 0; continue; }
            const uint32_t r0 = (uint32_t)(gw - w_lo) * 64, ra = r0 + lane_id(), rb = ra + 32;
            bool ha = false, hb = false;
            if (ra < rows && (live >> lane_id() & 1)) ha = pair_match_row(P, B, L, ca, cb, b, ra, mode, ro_a, ro_b, stats);
            if (rb < rows && (live >> (32 + lane_id()) & 1)) hb = pair_match_row(P, B, L, ca, cb, b, rb, mode, ro_a, ro_b, stats);
            const uint32_t lo = __ballot_sync(0xffffffffu, ha), hi = __ballot_sync(0xffffffffu, hb);
            if (lane_id() == 0) leaf_bm[gw] = ((uint64_t)hi << 32) | lo;
        }
    }
}

// ---- digest of the result bitmaps (bench / tests; the oracle computes the same over its own bitmaps, oracle/vlo_api.cpp vlo_scan_generated) -------
// xor over the blocks [block_lo, block_hi) of XXH64(the block's bitmap words as bytes) * (2 * key + 1), key = key_base + block index in the batch.
static __global__ void k_bitmap_digest(BatchView B, const uint64_t* __restrict__ reg, uint32_t block_lo, uint32_t block_hi, uint64_t key_base, unsigned long long* __restrict__ out) {
    const uint32_t b = block_lo + blockIdx.x * blockDim.x + threadIdx.x;
    unsigned long long d = 0;
    if (b < block_hi) {
        const uint64_t lo = B.blk_word_off[b], hi = B.blk_word_off[b + 1];
        d = xxh64((const uint8_t*)(reg + lo), (uint32_t)((hi - lo) * 8)) * (2 * (key_base + b) + 1);
    }
#pragma unroll
    for (int s = 16; s; s >>= 1) d ^= __shfl_xor_sync(0xffffffffu, d, s);
    if (lane_id() == 0 && d) atomicXor(out, d);
}

}  // namespace vl
