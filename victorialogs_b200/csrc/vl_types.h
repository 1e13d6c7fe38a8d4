// POD layouts shared by the host program compiler (vl_program.h), the staging code (vl_engine.h) and the CUDA kernels (vl_kernels.cuh).
#pragma once
#include <stdint.h>

namespace vl {

enum { VT_STRING = 1, VT_DICT = 2, VT_UINT8 = 3, VT_UINT16 = 4, VT_UINT32 = 5, VT_UINT64 = 6, VT_FLOAT64 = 7, VT_IPV4 = 8, VT_ISO8601 = 9, VT_INT64 = 10, VT_MAX = 11 };
enum { F_NOOP = 0, F_PHRASE, F_PREFIX, F_EXACT, F_IN, F_REGEXP, F_AND, F_OR, F_NOT,
       F_EXACT_PREFIX = 9, F_LEN_RANGE = 10, F_STRING_RANGE = 11, F_IPV4_RANGE = 12, F_VALUE_TYPE = 13,
       F_ANY_CASE_PHRASE = 14, F_ANY_CASE_PREFIX = 15, F_SEQUENCE = 16, F_CONTAINS_ALL = 17, F_CONTAINS_ANY = 18,
       F_EQ_FIELD = 19, F_LE_FIELD = 20, F_RANGE = 21, F_TIME = 22 };
enum { VTYPE_CONST = 0, VTYPE_NO_SUCH = 255 };   // F_VALUE_TYPE: DevLeaf.aux0 = VT_* code of the wanted type, or one of these
enum { COL_MISSING = 0, COL_CONST = 1, COL_VALUES = 2 };
enum { VALUES_STAGED = 0,     // lens items and data are in the arena
       VALUES_DEFERRED = 1,   // phase 1 of a bloom-first upload: only the header payloads (bloom filter, dict) are on the device yet
       VALUES_ABSENT = 2 };   // the probe pass proved that no filter of the program reads this column's values in this block: they stayed on the host

// One (block, field) cell of a resident batch: the columnHeader fields the scan needs + arena offsets of the payloads
// (lib/logstorage/block_header.go:584-615).  Offsets are relative to the batch arena base.
struct DevColumn {
    uint8_t kind;          // COL_*
    uint8_t vt;            // VT_*
    uint8_t lens_type;     // uintBlockType 0..7 (lib/logstorage/encoding.go:177-187)
    uint8_t dict_len;
    uint8_t data_const;    // decode rule "every row = data" (encoding.go:113-120)
    uint8_t values_state;  // VALUES_*: bloom-first staging (vlscan_scan_batch) leaves the values of a column on the host while / when no filter can reach them
    uint8_t pad[2];
    uint32_t lens_const;   // the single item of a const lens block
    uint32_t bloom_words;
    uint64_t min_value, max_value;
    uint64_t lens_off;     // lens items (after the type byte)
    uint64_t data_off, data_len;
    uint64_t bloom_off;
    uint64_t meta_off;     // CONST: value bytes.  DICT: u32 offsets[dict_len+1] followed by the concatenated values
    uint32_t meta_len;     // CONST: value length. DICT: total bytes of the concatenated values
    uint32_t pad2;
};

// The timestamps column of one block of a resident batch: raw varint bytes in the arena (ZSTD types already inflated) + timestampsHeader
struct DevTimestamps {
    uint64_t off;          // arena offset of the encoded deltas
    uint32_t len;
    uint8_t mt;            // 0 none, else the plain marshal type: 2 delta const, 3 const, 5 nearest delta2, 6 nearest delta (encoding.go:20-43)
    uint8_t pad[3];
    int64_t first, max;    // minTimestamp (= first value), maxTimestamp
};
enum { MT_ZSTD_NEAREST_DELTA2 = 1, MT_DELTA_CONST = 2, MT_CONST = 3, MT_ZSTD_NEAREST_DELTA = 4, MT_NEAREST_DELTA2 = 5, MT_NEAREST_DELTA = 6 };

struct TypedNeedle {       // result of parsing a needle for one valueType (filter_exact.go:237-354, in_values.go:141-315)
    uint64_t val;          // value in the column's comparison domain: uint / zig-zag int64 / float64 bits / ipv4 / iso8601 ns
    int64_t sval;          // signed view for the min/max range check of int64 / iso8601; float64: unused
    uint8_t ok;
    uint8_t pad[7];
};

struct DevRegex {          // device image of CompiledRegex (vl_regex.h)
    uint32_t prefix_off, prefix_len;
    uint32_t sub_off, sub_len;         // substrDotStar / substrDotPlus literal
    uint8_t only_prefix, dot_star, dot_plus, sub_kind;   // sub_kind: 0 none, 1 substrDotStar, 2 substrDotPlus
    uint32_t nclasses, nstates;
    uint32_t bounds_off;               // int32[nclasses] in blob (4-byte aligned)
    uint32_t ascii_off;                // uint8[128]
    uint32_t trans_off;                // uint16[nstates*nclasses] (2-byte aligned)
    uint32_t accept_off;               // uint8[nstates]
    uint32_t tail_off, tail_len;       // suffix == `.*LITERAL` (dot-all): the automaton accepts iff LITERAL occurs in the remainder
};

struct DevLeaf {
    uint8_t kind;                      // F_PHRASE .. F_REGEXP, F_NOOP
    uint8_t starts_tok, ends_tok;      // needle boundary flags (filter_phrase.go:229-239)
    uint8_t f64_phrase_gate;           // phrase on float64: tryParseFloat64Exact ok || phrase in {".","+","-"} (filter_phrase.go:165-168)
    uint8_t f64_exact_form;            // phrase contains '.' strictly inside (filter_phrase.go:169-173)
    uint8_t f64_prefix_gate;           // prefix on float64 (filter_prefix.go:161-165)
    uint8_t in_has_empty;              // "" is one of the in() values
    uint8_t in_skip_sets;              // number of token sets > maxTokenSetsToInit (filter_in.go:206)
    int32_t field;                     // index into the program's field table
    uint32_t needle_off, needle_len;   // blob
    uint32_t hashes_off, nhashes;      // u64 table: bloom probe hashes of the leaf's tokens (6 per token)
    TypedNeedle typed[VT_MAX];         // phrase/exact/prefix needle parsed per valueType
    // in(): string values + per-type sets
    uint32_t in_count;                 // number of values
    uint32_t in_offs_off;              // blob: u32 offsets[in_count+1] (4-byte aligned), relative to in_blob_off
    uint32_t in_blob_off;
    uint32_t in_sets_off, in_nsets;    // u32 table: per token set {hashes_off, nhashes}
    uint32_t in_typed_off[VT_MAX];     // u64 table offset of the sorted typed set
    uint32_t in_typed_cnt[VT_MAX];
    int32_t regex;                     // index into the regex table or -1
    // strategy for plain string columns, decided once per leaf on the host:
    uint8_t str_strategy;              // STR_ROW: per-row matcher, STR_SCAN: row-agnostic substring scan, STR_ALL: every row matches
    uint8_t scan_mode;                 // SCAN_* verifier of the substring scan
    uint8_t always_none;               // the filter's own arguments exclude every row (minLen > maxLen, minValue > maxValue)
    uint8_t gates;                     // header-level gates decided on the host from the arguments alone (GATE_* bits)
    uint32_t scan_needle_off, scan_needle_len;   // blob: the literal the scan searches for
    // exact_prefix / len_range / string_range / ipv4_range / value_type
    uint64_t aux0, aux1;               // len_range: minLen, maxLen; ipv4_range: minValue, maxValue; value_type: wanted type code
    uint32_t needle2_off, needle2_len; // string_range: maxValue (needle = minValue).  i(...): the UPPER-cased phrase (needle = the lower-cased one)
    uint32_t hashes2_off, nhashes2;    // i(...): probe hashes of the upper-cased tokens (iso8601 columns, filter_any_case_phrase.go:119-126)
    uint32_t list_off, list_len;       // seq() / contains_all() / contains_any(): the phrases as (varuint length, bytes)* in the blob; in_count = how many
    int32_t field2;                    // eq_field / le_field: the other field (index into the program's field table)
    uint32_t pair_excl;                // le_field: 1 = lt_field (equal values excluded)
    // range(): the bounds per column class (filter_range.go:246-347,362-420): u64 lo/hi, i64 lo/hi, f64 min/max (bits), u32 lo/hi
    uint64_t rng_ulo, rng_uhi; int64_t rng_ilo, rng_ihi; uint64_t rng_fmin, rng_fmax; uint32_t rng_iplo, rng_iphi;
};
// DevLeaf.gates
enum { GATE_DIGIT_PREFIX = 1,          // exact_prefix: !(prefix < "0" || prefix > "9")
       GATE_SR_UINT = 2,               // string_range on uint / ipv4 / iso8601 text: !(min > "9" || max < "0")
       GATE_SR_INT = 4,                // string_range on int64 text (filter_string_range.go:213-217)
       GATE_SR_FLOAT = 8 };            // string_range on float64 text: !(min > "9" || max < "+")

struct DevPrepass {                    // one fieldTokens entry of an AND / OR node (filter_and.go:21-25)
    int32_t field;
    uint32_t ntokens;
    uint32_t tok_offs_off;             // blob: u32 offsets[ntokens+1] (4-byte aligned) relative to tok_blob_off
    uint32_t tok_blob_off;
    uint32_t hashes_off, nhashes;      // u64 table
};

struct DevProgram {
    const DevLeaf* leaves; const DevPrepass* prepass; const DevRegex* regexes;
    const uint8_t* blob; const uint64_t* u64s; const uint32_t* u32s;
};

// stats slots (device u64 array)
enum { ST_VALUES_BYTES = 0, ST_BLOOM_BYTES, ST_COLUMNS_READ, ST_BITMAP_BYTES, ST_ROWS_MATCHED, ST_BLOCKS_MATCHED, ST_ERROR, ST_SCAN_BYTES, ST_COUNT };
enum { ERR_NONE = 0, ERR_LENS_MISMATCH = 1, ERR_DICT_INDEX = 2, ERR_BAD_WIDTH = 3, ERR_UNSUPPORTED_FLOAT_TOSTRING = 4, ERR_BAD_LENS_TYPE = 5, ERR_NO_TIMESTAMPS = 6, ERR_BAD_TIMESTAMPS = 7, ERR_VALUES_ABSENT = 8 };

struct BatchView {
    const uint8_t* arena;         // values payloads: lens items, data, encoded timestamps (lens_off, data_off, DevTimestamps.off)
    const uint8_t* hdr;           // header payloads: bloom filters, const values, dict tables (bloom_off, meta_off).  The same buffer as `arena`
                                  // unless the batch was staged bloom-first (vlscan_scan_batch): then it is the phase-1 buffer
    const DevColumn* cols;        // [nblocks * nfields]
    const uint32_t* blk_rows;     // [nblocks]
    const uint64_t* blk_word_off; // [nblocks + 1]
    const uint32_t* word_block;   // [nwords] owning block of each bitmap word
    const DevTimestamps* ts;      // [nblocks] or NULL when the batch was staged without timestamps
    uint32_t nblocks, nfields;
    uint64_t nwords;
};

// An on-disk values column whose lens block the device regenerates: k_finish_ondisk_cols checks its header once it is there
struct OndiskCol { uint64_t col; uint64_t lens_total; uint64_t rows; };

enum { STR_ROW = 0, STR_SCAN = 1, STR_ALL = 2 };
// per (block, leaf) decision of the header dispatch
enum { ACT_NONE = 0, ACT_ALL = 1, ACT_DICT = 2, ACT_SCAN = 3, ACT_FIXED_EQ = 4, ACT_FIXED_IN = 5,
       ACT_ROW = 6,         // per-row matcher: the leaf's string predicate on the value (typed values through their text)
       ACT_ROW_EQ = 7,      // per-row matcher: binary equality with the payload (typed column whose layout is not the fixed-width one)
       ACT_ROW_IN = 8,      // per-row matcher: membership in the leaf's typed value set
       ACT_TIME = 9,        // _time filter that partly overlaps the block: decode the timestamps, compare per row
       ACT_PAIR = 10 };     // eq_field / le_field: two columns, row by row (payload: PAIR_* mode)
// how a two-column leaf compares the rows of a block (filter_eq_field.go:60-121, filter_le_field.go:93-154)
enum { PAIR_STRINGS = 0,   // the string forms of both values (const, missing = "", dict entry, text of a typed value)
       PAIR_BINARY = 1,    // same typed valueType on both sides: the encoded values themselves
       PAIR_DICT = 2 };    // both dict columns: the dictionary entries
// scan verifier modes of the row-agnostic substring kernel
enum { SCAN_PHRASE = 0, SCAN_PREFIX = 1, SCAN_CONTAINS = 2, SCAN_RX_DOTPLUS = 3, SCAN_RX_SUFFIX = 4, SCAN_RX_TAIL = 5 };

}  // namespace vl
