/*
 * oracle.cpp — CPU restatement of the reference's scan -> filter -> hash-group-by/aggregate path.
 *
 * >>> TEST INFRASTRUCTURE.  Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline /
 * >>> `--impl reference` legs may build, load or call anything under oracle/.  The product
 * >>> (heavydb_b200/, include/) never links or imports it.
 *
 * What it is: a plain scalar C++17 restatement of what heavyai/heavydb executes below
 * Executor::executeWorkUnit (QueryEngine/Execute.cpp:2144) with --cpu-only, for the subset
 * single table, quals = AND/OR tree of `column OP constant`, optional single-column GROUP BY,
 * targets in {group key, COUNT(*), COUNT(c), SUM(c), MIN(c), MAX(c), AVG(c)},
 * column types TINYINT/SMALLINT/INT/BIGINT/DOUBLE.  Each function cites the reference lines it follows
 * (paths relative to /root/reference).
 *
 * Parity pinning (SURVEY.md §8c): the whole reference executor cannot be built here (needs LLVM 14, Boost,
 * Thrift, TBB, a JVM).  The oracle is pinned instead by
 *   (1) the reference's own hash/probe runtime compiled verbatim from /root/reference into
 *       oracle/_ref/libref_groupby.so (QueryEngine/GroupByRuntime.cpp + MurmurHash.cpp) and compared against
 *       oracle_murmur3 / oracle_get_group_value (tests/test_oracle_ref.py), plus the probe constants
 *       MurmurHash3(&int64{12345},8,0)=342635441 and MurmurHash3(&int32{7},4,0)=1343918321;
 *   (2) the reference's SQL golden tests: table `test` of Tests/ExecuteTest.cpp:30063-30115 and the
 *       FilterAndSimpleAggregation / FilterAndGroupBy / GroupByKeylessAndNotKeyless query shapes, with expected
 *       values computed by SQLite exactly as the reference's own comparator does
 *       (ExecuteTest.cpp:383-520) — tests/test_oracle_golden.py;
 *   (3) the ResultSetTest generator pattern (Tests/ResultSetTestUtils.h:33-70, ResultSetTest.cpp:1081-1098)
 *       for iteration and reduction over hand-filled storages — tests/test_resultset_vectors.py.
 */
#include <pthread.h>
#include <sched.h>

#include <algorithm>
#include <atomic>
#include <cfloat>
#include <climits>
#include <cmath>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <limits>
#include <memory>
#include <string>
#include <thread>
#include <vector>

#include "../include/b2q.h" /* POD input structs of the boundary only */
#include "oracle_gen.h"

#define ORACLE_EXPORT extern "C" __attribute__((visibility("default")))

namespace {

/* ---- Shared/InlineNullValues.h:30-36 ---- */
constexpr int64_t kNullTinyint = INT8_MIN;
constexpr int64_t kNullSmallint = INT16_MIN;
constexpr int64_t kNullInt = INT32_MIN;
constexpr int64_t kNullBigint = INT64_MIN;
constexpr double kNullDouble = DBL_MIN; /* NULL_DOUBLE is the smallest NORMAL double */
constexpr float kNullFloat = FLT_MIN;   /* NULL_FLOAT (Shared/InlineNullValues.h) */
/* QueryEngine/GpuRtConstants.h: EMPTY_KEY_64 / EMPTY_KEY_32 */
constexpr int64_t kEmptyKey64 = std::numeric_limits<int64_t>::max();
constexpr int32_t kEmptyKey32 = std::numeric_limits<int32_t>::max();

struct Ti {
  int type{0};
  bool notnull{false};
  int scale{0}; /* SQLTypeInfo::get_scale() of a DECIMAL / NUMERIC */
};

/* dictionary-encoded strings are int32 ids on this path (sqltypes.h is_dict_encoded_string; treated like
 * is_int_and_no_bigger_than(ti, 4) by QueryMemoryDescriptor.cpp:803-804), TIME / TIMESTAMP / DATE are int64 (is_time()) */
bool is_string(int t) { return t == B2Q_kTEXT || t == B2Q_kVARCHAR || t == B2Q_kCHAR; }
bool is_time(int t) { return t == B2Q_kTIME || t == B2Q_kTIMESTAMP || t == B2Q_kDATE; }
/* DECIMAL / NUMERIC: value x 10^scale as int64 (sqltypes.h is_decimal(); every branch of the planner and of the row
 * function that is not is_fp() treats it like BIGINT; the scale only matters at read-out) */
bool is_decimal(int t) { return t == B2Q_kDECIMAL || t == B2Q_kNUMERIC; }
bool is_integer(int t) { return t == B2Q_kTINYINT || t == B2Q_kSMALLINT || t == B2Q_kINT || t == B2Q_kBIGINT || is_string(t) || is_time(t) || is_decimal(t); }
bool is_fp(int t) { return t == B2Q_kDOUBLE || t == B2Q_kFLOAT; }
/* inline_fp_null_val widened to double: a FLOAT value reaches every comparison through an exact fpext */
double fp_null_of(int t) { return t == B2Q_kFLOAT ? static_cast<double>(kNullFloat) : kNullDouble; }
int type_size(int t) { /* SQLTypeInfo::get_size() for the fixed-width subset */
  switch (t) {
    case B2Q_kTINYINT: return 1;
    case B2Q_kSMALLINT: return 2;
    case B2Q_kINT: case B2Q_kFLOAT: case B2Q_kTEXT: case B2Q_kVARCHAR: case B2Q_kCHAR: return 4; /* logical size of a dictionary id */
    case B2Q_kBIGINT: case B2Q_kTIME: case B2Q_kTIMESTAMP: case B2Q_kDATE: case B2Q_kDECIMAL: case B2Q_kNUMERIC: return 8;
    case B2Q_kDOUBLE: return 8;
    default: return -1;
  }
}
int64_t inline_int_null_val(int t) { /* Shared/InlineNullValues.h inline_int_null_val */
  switch (t) {
    case B2Q_kTINYINT: return kNullTinyint;
    case B2Q_kSMALLINT: return kNullSmallint;
    case B2Q_kINT: case B2Q_kTEXT: case B2Q_kVARCHAR: case B2Q_kCHAR: return kNullInt;
    case B2Q_kBIGINT: case B2Q_kTIME: case B2Q_kTIMESTAMP: case B2Q_kDATE: case B2Q_kDECIMAL: case B2Q_kNUMERIC: return kNullBigint;
    default: abort();
  }
}
double exp_to_scale(int scale) { /* Shared/sqltypes.h exp_to_scale */
  double d = 1;
  for (int i = 0; i < scale; ++i) d *= 10;
  return d;
}
int64_t bits_of(double d) {
  int64_t r;
  memcpy(&r, &d, 8);
  return r;
}
double double_of(int64_t b) {
  double r;
  memcpy(&r, &b, 8);
  return r;
}
int64_t align_to_int64(int64_t x) { return (x + 7) & ~int64_t(7); } /* BufferCompaction.h:42-45 */

struct OracleError {
  int code;
  std::string msg;
};
[[noreturn]] void fail(int code, const std::string& msg) { throw OracleError{code, msg}; }

/* ---------------------------------------------------------------------------------------------------
 * MurmurHash3 x86_32 — QueryEngine/MurmurHash3Inl.h:11-72 (restated; pinned against _ref and constants)
 * ------------------------------------------------------------------------------------------------- */
uint32_t rotl32(uint32_t x, int8_t r) { return (x << r) | (x >> (32 - r)); }
uint32_t murmur3(const void* key, int len, uint32_t seed) {
  const uint8_t* data = static_cast<const uint8_t*>(key);
  const int nblocks = len / 4;
  uint32_t h1 = seed;
  const uint32_t c1 = 0xcc9e2d51, c2 = 0x1b873593;
  for (int i = 0; i < nblocks; ++i) {
    uint32_t k1;
    memcpy(&k1, data + 4 * i, 4);
    k1 *= c1;
    k1 = rotl32(k1, 15);
    k1 *= c2;
    h1 ^= k1;
    h1 = rotl32(h1, 13);
    h1 = h1 * 5 + 0xe6546b64;
  }
  const uint8_t* tail = data + nblocks * 4;
  uint32_t k1 = 0;
  switch (len & 3) {
    case 3: k1 ^= tail[2] << 16; /* fallthrough */
    case 2: k1 ^= tail[1] << 8;  /* fallthrough */
    case 1:
      k1 ^= tail[0];
      k1 *= c1;
      k1 = rotl32(k1, 15);
      k1 *= c2;
      h1 ^= k1;
  }
  h1 ^= static_cast<uint32_t>(len);
  h1 ^= h1 >> 16;
  h1 *= 0x85ebca6b;
  h1 ^= h1 >> 13;
  h1 *= 0xc2b2ae35;
  h1 ^= h1 >> 16;
  return h1;
}

/* ---------------------------------------------------------------------------------------------------
 * Baseline-hash group lookup — QueryEngine/GroupByRuntime.cpp:20-48 (key_hash, get_group_value) with the CPU
 * get_matching_group_value of QueryEngine/RuntimeFunctions.cpp:1953-2005 (match or claim an EMPTY slot).
 * Row-wise layout: [key: key_count * key_width bytes, padded to 8][slots...], row_size_quad int64 per row.
 * Returns pointer to the first slot of the row, or nullptr when the table is full.
 * ------------------------------------------------------------------------------------------------- */
template <typename T>
int64_t* get_matching_group_value_t(int64_t* groups_buffer, uint32_t h, const T* key, uint32_t key_count,
                                    uint32_t row_size_quad) {
  auto off = static_cast<uint64_t>(h) * row_size_quad;
  auto row_ptr = reinterpret_cast<T*>(groups_buffer + off);
  const T empty = sizeof(T) == 4 ? static_cast<T>(kEmptyKey32) : static_cast<T>(kEmptyKey64);
  if (*row_ptr == empty) {
    memcpy(row_ptr, key, key_count * sizeof(T));
    auto row_ptr_i8 = reinterpret_cast<int8_t*>(row_ptr + key_count);
    return reinterpret_cast<int64_t*>(align_to_int64(reinterpret_cast<int64_t>(row_ptr_i8)));
  }
  if (memcmp(row_ptr, key, key_count * sizeof(T)) == 0) {
    auto row_ptr_i8 = reinterpret_cast<int8_t*>(row_ptr + key_count);
    return reinterpret_cast<int64_t*>(align_to_int64(reinterpret_cast<int64_t>(row_ptr_i8)));
  }
  return nullptr;
}

int64_t* get_matching_group_value(int64_t* groups_buffer, uint32_t h, const int64_t* key, uint32_t key_count,
                                  uint32_t key_width, uint32_t row_size_quad) {
  switch (key_width) {
    case 4:
      return get_matching_group_value_t(groups_buffer, h, reinterpret_cast<const int32_t*>(key), key_count,
                                        row_size_quad);
    case 8:
      return get_matching_group_value_t(groups_buffer, h, key, key_count, row_size_quad);
    default:
      return nullptr;
  }
}

int64_t* get_group_value(int64_t* groups_buffer, uint32_t entry_count, const int64_t* key, uint32_t key_count,
                         uint32_t key_width, uint32_t row_size_quad) {
  uint32_t h = murmur3(key, key_width * key_count, 0) % entry_count;
  int64_t* m = get_matching_group_value(groups_buffer, h, key, key_count, key_width, row_size_quad);
  if (m) return m;
  uint32_t h_probe = (h + 1) % entry_count;
  while (h_probe != h) {
    m = get_matching_group_value(groups_buffer, h_probe, key, key_count, key_width, row_size_quad);
    if (m) return m;
    h_probe = (h_probe + 1) % entry_count;
  }
  return nullptr;
}

/* get_matching_group_value_columnar + get_group_value_columnar (GroupByRuntime.cpp:136-157 and the matcher in
 * RuntimeFunctions.cpp): one 8-byte key per entry in the leading key column; returns the entry index or -1. */
int64_t get_group_value_columnar_slot(int64_t* groups_buffer, uint32_t entry_count, int64_t key) {
  const uint32_t h = murmur3(&key, 8, 0) % entry_count;
  uint32_t probe = h;
  do {
    if (groups_buffer[probe] == key) return probe;
    if (groups_buffer[probe] == kEmptyKey64) { groups_buffer[probe] = key; return probe; }
    probe = (probe + 1) % entry_count;
  } while (probe != h);
  return -1;
}

/* ---------------------------------------------------------------------------------------------------
 * Aggregate update functions — QueryEngine/RuntimeFunctions.cpp:362 (agg_count), :1151-1173 (agg_sum/max/min/id),
 * :1313-1431 (*_skip_val), :1439-1473 (double), :1558-1593 (fp skip_val)
 * ------------------------------------------------------------------------------------------------- */
void agg_count(int64_t* agg) { *reinterpret_cast<uint64_t*>(agg) += 1; }
void agg_sum(int64_t* agg, int64_t val) { /* wraps silently, like the reference (:1151-1155) */
  *agg = static_cast<int64_t>(static_cast<uint64_t>(*agg) + static_cast<uint64_t>(val));
}
void agg_max(int64_t* agg, int64_t val) { *agg = std::max(*agg, val); }
void agg_min(int64_t* agg, int64_t val) { *agg = std::min(*agg, val); }
void agg_id(int64_t* agg, int64_t val) { *agg = val; }
void agg_sum_skip_val(int64_t* agg, int64_t val, int64_t skip_val) { /* :1313-1325 */
  const auto old = *agg;
  if (val != skip_val) {
    if (old != skip_val) {
      agg_sum(agg, val);
    } else {
      *agg = val;
    }
  }
}
void agg_count_skip_val(int64_t* agg, int64_t val, int64_t skip_val) { /* :1363-1369 */
  if (val != skip_val) agg_count(agg);
}
void agg_max_skip_val(int64_t* agg, int64_t val, int64_t skip_val) { /* DEF_SKIP_AGG :1405-1416 */
  if (val != skip_val) {
    const int64_t old_agg = *agg;
    if (old_agg != skip_val) agg_max(agg, val); else *agg = val;
  }
}
void agg_min_skip_val(int64_t* agg, int64_t val, int64_t skip_val) {
  if (val != skip_val) {
    const int64_t old_agg = *agg;
    if (old_agg != skip_val) agg_min(agg, val); else *agg = val;
  }
}
void agg_sum_double(int64_t* agg, double val) { *agg = bits_of(double_of(*agg) + val); } /* :1444-1448 */
void agg_max_double(int64_t* agg, double val) { *agg = bits_of(std::max(double_of(*agg), val)); }
void agg_min_double(int64_t* agg, double val) { *agg = bits_of(std::min(double_of(*agg), val)); }
/* DEF_SKIP_AGG for doubles (:1558-1570): `val != skip_val` is an fp compare, `old_agg` is compared bitwise */
void agg_sum_double_skip_val(int64_t* agg, double val, double skip_val) {
  if (val != skip_val) {
    if (*agg != bits_of(skip_val)) agg_sum_double(agg, val); else *agg = bits_of(val);
  }
}
void agg_max_double_skip_val(int64_t* agg, double val, double skip_val) {
  if (val != skip_val) {
    if (*agg != bits_of(skip_val)) agg_max_double(agg, val); else *agg = bits_of(val);
  }
}
void agg_min_double_skip_val(int64_t* agg, double val, double skip_val) {
  if (val != skip_val) {
    if (*agg != bits_of(skip_val)) agg_min_double(agg, val); else *agg = bits_of(val);
  }
}
void agg_count_double_skip_val(int64_t* agg, double val, double skip_val) { /* :1541-1547 */
  if (val != skip_val) agg_count(agg);
}

/* ---------------------------------------------------------------------------------------------------
 * Column decode — QueryEngine/DecodersImpl.h:30-61 (fixed_width_int_decode: sign-extending load),
 * :112-136 (fixed_width_double_decode)
 * ------------------------------------------------------------------------------------------------- */
int64_t fixed_width_int_decode(const int8_t* byte_stream, int byte_width, int64_t pos) {
  switch (byte_width) {
    case 1: return static_cast<int64_t>(byte_stream[pos]);
    case 2: { int16_t v; memcpy(&v, byte_stream + pos * 2, 2); return v; }
    case 4: { int32_t v; memcpy(&v, byte_stream + pos * 4, 4); return v; }
    case 8: { int64_t v; memcpy(&v, byte_stream + pos * 8, 8); return v; }
    default: abort();
  }
}
double fixed_width_double_decode(const int8_t* byte_stream, int64_t pos) {
  double v;
  memcpy(&v, byte_stream + pos * 8, 8);
  return v;
}

/* Hash join (one INNER level): the joined inner table's columns are addressed as columns n_outer.. of a combined
 * ("virtual") table; their row position is the matching inner row (the join loop's iterator, IRCodegen.cpp
 * buildJoinLoops), not the outer position.  Set per outer row by run_fragment; one row loop per thread. */
struct JoinRowCtx {
  int n_outer{INT32_MAX};
  int64_t inner_pos{0}; /* -1: LEFT join without a match => every inner column reads NULL (codegenOuterJoinNullPlaceholder) */
};
thread_local JoinRowCtx g_join_row;
inline int64_t row_pos_of(int c, int64_t pos) { return c >= g_join_row.n_outer ? g_join_row.inner_pos : pos; }
inline bool outer_join_null(int c) { return c >= g_join_row.n_outer && g_join_row.inner_pos < 0; }

/* Physical element width of column c: narrower than the logical type under `ENCODING FIXED(bits)`. */
int phys_width(const B2QTableInfo& tbl, int c) {
  if (tbl.col_encoded_sizes && tbl.col_encoded_sizes[c] > 0) return tbl.col_encoded_sizes[c];
  if (tbl.col_encoded_sizes && tbl.col_encoded_sizes[c] < 0) return -tbl.col_encoded_sizes[c]; /* DATE ENCODING DAYS(32|16) */
  return type_size(tbl.col_types[c].type);
}
/* kENCODING_DATE_IN_DAYS (the default encoding of DATE columns): the chunk holds int32 / int16 days since the epoch */
bool is_date_in_days(const B2QTableInfo& tbl, int c) { return tbl.col_encoded_sizes && tbl.col_encoded_sizes[c] < 0; }
constexpr int64_t kSecsPerDay = 86400;
/* FixedWidthInt::codegenDecode (sign-extending load, DecodersImpl.h:30-61) followed by
 * CodeGenerator::codgenAdjustFixedEncNull (ColumnIR.cpp:456-500): the physical width's minimum is NULL and becomes the
 * logical type's sentinel (only for nullable columns, ColumnIR.cpp:286-291). */
int64_t decode_int_column(const B2QTableInfo& tbl, const B2QFragmentInfo& fr, int c, int64_t pos) {
  if (outer_join_null(c)) return inline_int_null_val(tbl.col_types[c].type);
  pos = row_pos_of(c, pos);
  const int pw = phys_width(tbl, c);
  const int lw = type_size(tbl.col_types[c].type);
  if (is_string(tbl.col_types[c].type) && pw < lw) {
    /* FixedWidthUnsigned (ColumnIR.cpp:59-67, fixed_width_unsigned_decode DecodersImpl.h:63-88); NULL is the maximum
     * of the unsigned type (inline_fixed_encoding_null_val, InlineNullValues.h:173-182) */
    const uint8_t* b = static_cast<const uint8_t*>(fr.col_buffers[c]);
    int64_t u;
    if (pw == 1) u = b[pos]; else { uint16_t x; memcpy(&x, b + 2 * pos, 2); u = x; }
    if (!tbl.col_types[c].notnull && u == (pw == 1 ? 255 : 65535)) u = inline_int_null_val(tbl.col_types[c].type);
    return u;
  }
  int64_t v = fixed_width_int_decode(static_cast<const int8_t*>(fr.col_buffers[c]), pw, pos);
  if (is_date_in_days(tbl, c)) {
    /* FixedWidthSmallDate (ColumnIR.cpp:73-81), fixed_width_small_date_decode (DecodersImpl.h:138-146): the physical
     * minimum is NULL whatever the column's nullability, everything else is days * 86400 */
    const int64_t phys_null = pw == 2 ? INT16_MIN : INT32_MIN;
    return v == phys_null ? inline_int_null_val(tbl.col_types[c].type) : v * kSecsPerDay;
  }
  if (pw < lw && !tbl.col_types[c].notnull) {
    const int64_t phys_null = pw == 1 ? INT8_MIN : pw == 2 ? INT16_MIN : INT32_MIN;
    if (v == phys_null) v = inline_int_null_val(tbl.col_types[c].type);
  }
  return v;
}

/* fixed_width_double_decode / fixed_width_float_decode (DecodersImpl.h:112-136); a float is returned fpext-ed */
double decode_double_column(int type, const B2QFragmentInfo& fr, int c, int64_t pos) {
  if (outer_join_null(c)) return fp_null_of(type);
  if (type == B2Q_kFLOAT) {
    float f;
    memcpy(&f, static_cast<const int8_t*>(fr.col_buffers[c]) + row_pos_of(c, pos) * 4, 4);
    return f;
  }
  return fixed_width_double_decode(static_cast<const int8_t*>(fr.col_buffers[c]), row_pos_of(c, pos));
}
int64_t float_bits(float f) { int32_t b; memcpy(&b, &f, 4); return b; } /* int32 image, sign-extended: how get_agg_initial_val returns 4-byte patterns */

/* ===================================================================================================
 * Planner
 * ================================================================================================= */
struct Target {
  /* Shared/TargetInfo.h:49-78 */
  bool is_agg{false};
  int agg_kind{B2Q_kMIN};
  Ti sql_type;
  Ti agg_arg_type; /* type 0 == kNULLT */
  bool skip_null_val{false};
  /* ours */
  int arg_col{-1};
  Ti arg_ti;      /* argument expression's own type info */
  int first_slot{0};
  bool arg_constrained_not_null{false}; /* constrained_not_null(agg_arg(target_expr), ra_exe_unit.quals) */
  /* is_distinct_target: CountDistinctDescriptor{Bitmap, min_val, bucket_size, bitmap_sz_bits} (CountDistinctDescriptor.h) */
  bool is_distinct{false};
  int64_t cd_min{0}, cd_bits{0}, cd_bucket{0};
  int64_t cd_tail{0}; /* ours: byte offset (past p.buffer_size) of this target's per-entry bitmaps while the query runs */
};

struct Range { /* ExpressionRange (Integer or Double or Invalid) */
  enum Kind { Invalid, Integer, Double } kind{Invalid};
  int64_t imin{0}, imax{-1}, bucket{0};
  double fmin{0}, fmax{-1};
  bool has_nulls{false};
};

struct KeyCol { /* one GROUP BY column of a multi-column perfect hash */
  int col{-1};
  int64_t min{0}, max{-1}, card{0}, mult{1}, bucket{0};
  bool has_nulls{false};
};

struct Plan {
  B2QPlan p{};
  std::vector<Target> targets;
  std::vector<Ti> slot_compact_ti;
  std::vector<KeyCol> keys; /* size > 1: multi-column perfect hash */
  /* join level: probe parameters (the table itself is built per execution) */
  bool join{false};
  int join_outer_col{-1}, join_inner_vcol{-1}; /* virtual column ids */
  bool join_outer_nullable{false};
  bool join_left{false};
  std::shared_ptr<std::vector<int32_t>> join_buff;
  /* estimator query (QueryDescriptionType::Estimator): the argument tuple's (virtual) column ids */
  std::vector<int> estimator_cols;
  /* COUNT(DISTINCT): bytes of bitmaps kept behind the result buffer while the query runs (the reference keeps them in the
   * row set memory owner and a pointer in the slot; the slot here receives the set size when the query is done) */
  int64_t cd_total{0};
};

const B2QExpr& expr_at(const B2QExecUnit& u, int idx) {
  if (idx < 0 || idx >= u.num_exprs) fail(B2Q_ERR_INVALID_ARGUMENT, "expr index out of range");
  return u.exprs[idx];
}
Ti ti_of(const B2QTypeInfo& t) { return Ti{t.type, t.notnull != 0, t.scale}; }

/* OutputBufferInitialization.cpp:301-324 constrained_not_null: some member of ra_exe_unit.quals (NOT simple_quals) is,
 * at its top level, `expr IS NOT NULL` — which reaches the executor as UOper(kNOT, UOper(kISNULL, expr)) — over an
 * operand equal to `expr` (ColumnVar::operator==: same table / column / rte_idx). */
bool constrained_not_null(const B2QExecUnit& u, int arg_expr_idx) {
  if (arg_expr_idx < 0) return false;
  const B2QExpr& arg = expr_at(u, arg_expr_idx);
  for (int i = 0; i < u.num_quals; ++i) {
    const B2QExpr* uoper = &expr_at(u, u.quals[i]);
    if (uoper->kind != B2Q_EXPR_UOPER) continue;
    bool is_negated = false;
    if (uoper->op == B2Q_kNOT) {
      const B2QExpr& operand = expr_at(u, uoper->left);
      if (operand.kind != B2Q_EXPR_UOPER) continue;
      uoper = &operand;
      is_negated = true;
    }
    if (is_negated && uoper->op == B2Q_kISNULL) { /* kISNOTNULL itself never reaches this boundary */
      const B2QExpr& operand = expr_at(u, uoper->left);
      if (operand.kind == B2Q_EXPR_COLUMN_VAR && arg.kind == B2Q_EXPR_COLUMN_VAR && operand.col_id == arg.col_id &&
          operand.rte_idx == arg.rte_idx)
        return true;
    }
  }
  return false;
}

/* Shared/TargetInfo.cpp:25-78 get_target_info_impl */
Target get_target_info(const B2QExecUnit& u, int expr_idx, bool bigint_count) {
  const B2QExpr& e = expr_at(u, expr_idx);
  Target t;
  const bool notnull = e.ti.notnull != 0;
  if (e.kind != B2Q_EXPR_AGG) {
    if (e.kind != B2Q_EXPR_COLUMN_VAR) fail(B2Q_ERR_UNSUPPORTED, "non-aggregate target must be a ColumnVar");
    t.is_agg = false;
    t.agg_kind = B2Q_kMIN;
    t.sql_type = ti_of(e.ti); /* get_logical_type_info: identity for the numeric subset */
    t.agg_arg_type = Ti{0, false};
    t.skip_null_val = false;
    t.arg_col = e.col_id;
    t.arg_ti = ti_of(e.ti);
    return t;
  }
  t.is_agg = true;
  t.agg_kind = e.op;
  if (e.ival != 0 && (e.op != B2Q_kCOUNT || e.left < 0)) fail(B2Q_ERR_UNSUPPORTED, "DISTINCT is restated for COUNT(DISTINCT column) only");
  t.is_distinct = e.ival != 0;
  if (e.left < 0) {
    if (e.op != B2Q_kCOUNT) fail(B2Q_ERR_INVALID_ARGUMENT, "only COUNT may have no argument");
    t.sql_type = Ti{bigint_count ? B2Q_kBIGINT : B2Q_kINT, notnull};
    t.agg_arg_type = Ti{0, false};
    t.skip_null_val = false;
    return t;
  }
  const B2QExpr& arg = expr_at(u, e.left);
  if (arg.kind != B2Q_EXPR_COLUMN_VAR) fail(B2Q_ERR_UNSUPPORTED, "aggregate argument must be a ColumnVar");
  const Ti arg_ti = ti_of(arg.ti);
  t.arg_col = arg.col_id;
  t.arg_ti = arg_ti;
  t.arg_constrained_not_null = constrained_not_null(u, e.left); /* evaluated where the reference evaluates it; kept here once */
  if (is_string(arg_ti.type) && e.op != B2Q_kCOUNT) fail(B2Q_ERR_UNSUPPORTED, "only COUNT of a dictionary-encoded string is on this path");
  if (is_time(arg_ti.type) && (e.op == B2Q_kSUM || e.op == B2Q_kAVG)) fail(B2Q_ERR_UNSUPPORTED, "SUM / AVG of a TIME / TIMESTAMP / DATE");
  if (e.op == B2Q_kAVG) {
    t.sql_type = (is_integer(arg_ti.type) && !is_decimal(arg_ti.type)) ? Ti{B2Q_kBIGINT, arg_ti.notnull} : arg_ti; /* SQLTypeInfo::is_integer() is false for a DECIMAL: AVG keeps the scale for pair_to_double */
    t.agg_arg_type = arg_ti;
    t.skip_null_val = !arg_ti.notnull;
    return t;
  }
  t.sql_type = (e.op == B2Q_kCOUNT) ? Ti{bigint_count ? B2Q_kBIGINT : B2Q_kINT, notnull} : ti_of(e.ti);
  t.agg_arg_type = arg_ti;
  t.skip_null_val = !arg_ti.notnull;
  return t;
}

bool is_agg_domain_range_equivalent(int agg_kind) { return agg_kind == B2Q_kMIN || agg_kind == B2Q_kMAX; }

/* Shared/SqlTypesLayout.h:37-63 get_compact_type */
Ti get_compact_type(const Target& t) {
  if (!t.is_agg) return t.sql_type;
  if (t.agg_arg_type.type == 0) return t.sql_type;
  if (is_agg_domain_range_equivalent(t.agg_kind)) return t.agg_arg_type;
  Ti m = t.sql_type;
  m.notnull = t.agg_arg_type.notnull;
  return m;
}

/* ExpressionRange.cpp:521-632 getLeafColumnRange, then :144-200 apply_simple_quals when asked */
Range leaf_column_range(const B2QTableInfo& tbl, int col_id) {
  Range r;
  if (col_id < 0 || col_id >= tbl.num_cols) fail(B2Q_ERR_INVALID_ARGUMENT, "column id out of range");
  const int type = tbl.col_types[col_id].type;
  int64_t total = 0;
  for (int f = 0; f < tbl.num_fragments; ++f) total += tbl.fragments[f].num_tuples;
  const bool fp = is_fp(type);
  r.kind = fp ? Range::Double : Range::Integer;
  if (total == 0) { /* :567-575 empty table => [0,-1] */
    r.imin = 0; r.imax = -1; r.fmin = 0; r.fmax = -1; r.has_nulls = false;
    return r;
  }
  bool first = true;
  for (int f = 0; f < tbl.num_fragments; ++f) {
    const auto& fr = tbl.fragments[f];
    if (fr.num_tuples == 0) continue; /* isEmptyPhysicalFragment */
    const auto& st = fr.col_stats[col_id];
    if (first) {
      r.imin = st.int_min; r.imax = st.int_max; r.fmin = st.fp_min; r.fmax = st.fp_max;
      first = false;
    } else {
      r.imin = std::min(r.imin, st.int_min); r.imax = std::max(r.imax, st.int_max);
      r.fmin = std::min(r.fmin, st.fp_min); r.fmax = std::max(r.fmax, st.fp_max);
    }
  }
  for (int f = 0; f < tbl.num_fragments; ++f) {
    if (tbl.fragments[f].col_stats[col_id].has_nulls) { r.has_nulls = true; break; }
  }
  if (!fp && r.imax < r.imin) { /* :617-621 only nulls */
    r.imin = 0; r.imax = -1;
  }
  /* :622-624: DATE columns carry the day bucket (get_conservative_datetrunc_bucket(dtDAY)) */
  r.bucket = type == B2Q_kDATE ? kSecsPerDay : 0;
  return r;
}

void apply_simple_quals(const B2QExecUnit& u, int key_col_id, Range& r) { /* ExpressionRange.cpp:144-200, :95-123 */
  for (int i = 0; i < u.num_simple_quals; ++i) {
    const B2QExpr& q = expr_at(u, u.simple_quals[i]);
    if (q.kind != B2Q_EXPR_BIN_OPER) continue;
    const B2QExpr& l = expr_at(u, q.left);
    const B2QExpr& c = expr_at(u, q.right);
    if (l.kind != B2Q_EXPR_COLUMN_VAR || l.col_id != key_col_id || c.kind != B2Q_EXPR_CONSTANT) continue;
    /* an int column against an fp literal is CAST(col AS DOUBLE) OP lit in the reference; such casts do not pass
     * BinOper::normalize_simple_predicate, so the qual never reaches apply_simple_quals */
    if (is_fp(c.ti.type) != (r.kind == Range::Double)) continue;
    if (r.kind == Range::Double) {
      const double v = is_fp(c.ti.type) ? c.dval : static_cast<double>(c.ival);
      switch (q.op) {
        case B2Q_kGT: case B2Q_kGE: r.fmin = std::max(r.fmin, v); break;
        case B2Q_kLT: case B2Q_kLE: r.fmax = std::min(r.fmax, v); break;
        case B2Q_kEQ: r.fmin = std::max(r.fmin, v); r.fmax = std::min(r.fmax, v); break;
        default: break;
      }
    } else if (r.kind == Range::Integer) {
      const int64_t v = is_fp(c.ti.type) ? static_cast<int64_t>(c.dval) : c.ival;
      switch (q.op) {
        case B2Q_kGT: r.imin = std::max(r.imin, static_cast<int64_t>(static_cast<uint64_t>(v) + 1)); break; /* apply_int_qual's const_val + 1 wraps for INT64_MAX: the same value without the signed-overflow UB */
        case B2Q_kGE: r.imin = std::max(r.imin, v); break;
        case B2Q_kLT: r.imax = std::min(r.imax, static_cast<int64_t>(static_cast<uint64_t>(v) - 1)); break;
        case B2Q_kLE: r.imax = std::min(r.imax, v); break;
        case B2Q_kEQ: r.imin = std::max(r.imin, v); r.imax = std::min(r.imax, v); break;
        default: break;
      }
    }
  }
}

/* QueryEngine/OutputBufferInitialization.cpp:124-262 get_agg_initial_val (numeric subset) */
int64_t get_agg_initial_val(int agg, const Ti& ti, bool enable_compaction, unsigned min_byte_width_to_compact) {
  const unsigned byte_width = enable_compaction
                                  ? std::max(static_cast<unsigned>(type_size(ti.type)), min_byte_width_to_compact)
                                  : 8u;
  const bool fp = is_fp(ti.type);
  auto int_max_of = [](unsigned w) -> int64_t {
    switch (w) { case 1: return INT8_MAX; case 2: return INT16_MAX; case 4: return INT32_MAX; default: return INT64_MAX; }
  };
  auto int_min_of = [](unsigned w) -> int64_t {
    switch (w) { case 1: return INT8_MIN; case 2: return INT16_MIN; case 4: return INT32_MIN; default: return INT64_MIN; }
  };
  if (ti.type == B2Q_kFLOAT) { /* byte_width 4 (float_argument_input, OutputBufferInitialization.cpp:66-76, :141-247): int32 patterns */
    switch (agg) {
      case B2Q_kSUM: return ti.notnull ? float_bits(0.f) : float_bits(kNullFloat);
      case B2Q_kAVG: case B2Q_kCOUNT: return 0;
      case B2Q_kMIN: return ti.notnull ? float_bits(std::numeric_limits<float>::max()) : float_bits(kNullFloat);
      case B2Q_kMAX: return ti.notnull ? float_bits(-std::numeric_limits<float>::max()) : float_bits(kNullFloat);
      default: abort();
    }
  }
  switch (agg) {
    case B2Q_kSUM:
      if (!ti.notnull) return fp ? bits_of(kNullDouble) : inline_int_null_val(ti.type);
      return fp ? bits_of(0.0) : 0;
    case B2Q_kAVG:
    case B2Q_kCOUNT:
      return 0;
    case B2Q_kMIN:
      if (fp) return ti.notnull ? bits_of(DBL_MAX) : bits_of(kNullDouble);
      return ti.notnull ? int_max_of(byte_width) : inline_int_null_val(ti.type);
    case B2Q_kMAX:
      if (fp) return ti.notnull ? bits_of(-DBL_MAX) : bits_of(kNullDouble);
      return ti.notnull ? int_min_of(byte_width) : inline_int_null_val(ti.type);
    default:
      abort();
  }
}

/* GroupByAndAggregate.cpp:489-648 get_keyless_info */
void get_keyless_info(const B2QExecUnit& u, const B2QTableInfo& tbl, const std::vector<Target>& targets,
                      bool is_group_by, bool& keyless_out, int32_t& index_out) {
  bool keyless = true, found = false;
  int32_t index = 0;
  for (const auto& agg_info : targets) {
    const Ti chosen_type = get_compact_type(agg_info);
    if (!found && agg_info.is_agg && !agg_info.is_distinct) { /* !is_distinct_target(agg_info) */
      const bool has_arg = agg_info.arg_col >= 0;
      switch (agg_info.agg_kind) {
        case B2Q_kAVG:
          ++index;
          if (has_arg && !agg_info.arg_ti.notnull) {
            const Range er = leaf_column_range(tbl, agg_info.arg_col);
            if (er.kind == Range::Invalid || er.has_nulls) break;
          }
          found = true;
          break;
        case B2Q_kCOUNT:
          if (has_arg && !agg_info.arg_ti.notnull) {
            const Range er = leaf_column_range(tbl, agg_info.arg_col);
            if (er.kind == Range::Invalid || er.has_nulls) break;
          }
          found = true;
          break;
        case B2Q_kSUM: {
          const Range er = leaf_column_range(tbl, agg_info.arg_col);
          Ti arg_ti = agg_info.arg_ti;
          if (agg_info.arg_constrained_not_null) arg_ti.notnull = true; /* GroupByAndAggregate.cpp:531-533 */
          if (!arg_ti.notnull) {
            if (er.kind != Range::Invalid && !er.has_nulls) found = true;
          } else {
            if (er.kind == Range::Double) {
              if (er.fmax < 0 || er.fmin > 0) found = true;
            } else if (er.kind == Range::Integer) {
              if (er.imax < 0 || er.imin > 0) found = true;
            }
          }
          break;
        }
        case B2Q_kMIN: {
          const Range er = leaf_column_range(tbl, agg_info.arg_col);
          const int64_t init_max = get_agg_initial_val(agg_info.agg_kind, chosen_type, is_group_by, 8);
          if (er.kind == Range::Double) {
            if (er.fmax < double_of(init_max)) found = true;
          } else if (er.kind == Range::Integer) {
            if (er.imax < init_max) found = true;
          }
          break;
        }
        case B2Q_kMAX: {
          const Range er = leaf_column_range(tbl, agg_info.arg_col);
          if (er.kind == Range::Invalid || er.has_nulls) break;
          const int64_t init_min = get_agg_initial_val(agg_info.agg_kind, chosen_type, is_group_by, 8);
          if (er.kind == Range::Double) {
            if (er.fmin > double_of(init_min)) found = true;
          } else if (er.kind == Range::Integer) {
            if (er.imin > init_min) found = true;
          }
          break;
        }
        default:
          keyless = false;
          break;
      }
    }
    if (!keyless) break;
    if (!found) ++index;
  }
  keyless_out = keyless && found;
  index_out = index;
}

constexpr int64_t kMaxBufferSize = int64_t(1) << 30;   /* GroupByAndAggregate.cpp:57 */

/* inner_tuples: the rows of a join level's inner table, which `tbl` (the combined input) does not carry */
Plan make_plan_single(const B2QExecUnit& u, const B2QTableInfo& tbl, const B2QExecutionOptions& eo,
                      size_t max_groups_buffer_entry_guess, bool has_cardinality_estimation, uint64_t inner_tuples = 0) {
  if (u.has_union_all || u.has_window_function)
    fail(B2Q_ERR_UNSUPPORTED, "union / window functions are outside this path");
  if (u.has_estimator) {
    /* RelAlgExecutionUnit::createNdvExecutionUnit (CardinalityEstimator.cpp:94-116): no groupby_exprs, no targets,
     * estimator = NDVEstimator / LargeNDVEstimator over the GROUP BY tuple; QueryMemoryDescriptor::init returns the
     * Estimator descriptor with entry_count 1 (QueryMemoryDescriptor.cpp:270-300) */
    if (u.has_estimator != 1 && u.has_estimator != 2) fail(B2Q_ERR_INVALID_ARGUMENT, "estimator kind");
    if (u.num_groupby_exprs || u.num_target_exprs || u.num_order_entries || u.has_limit || u.offset)
      fail(B2Q_ERR_INVALID_ARGUMENT, "an estimator unit has no groupby_exprs, targets or sort_info");
    if (u.num_estimator_args <= 0 || u.num_estimator_args > B2Q_MAX_GROUP_COLS) fail(B2Q_ERR_UNSUPPORTED, "estimator argument count");
    Plan plan;
    B2QPlan& p = plan.p;
    p.query_desc_type = B2Q_Estimator;
    p.entry_count = 1;
    p.key_col_id = -1;
    p.idx_target_as_key = -1;
    p.effective_key_width = 8;
    p.join_outer_col = p.join_inner_col = -1;
    p.buffer_size = (u.has_estimator == 2 ? int64_t(256) : int64_t(1)) * 1024 * 1024; /* Estimator::getBufferSize() */
    for (int i = 0; i < u.num_estimator_args; ++i) {
      const B2QExpr& e = expr_at(u, u.estimator_args[i]);
      if (e.kind != B2Q_EXPR_COLUMN_VAR) fail(B2Q_ERR_UNSUPPORTED, "estimator argument must be a ColumnVar");
      if (e.col_id < 0 || e.col_id >= tbl.num_cols) fail(B2Q_ERR_INVALID_ARGUMENT, "column id out of range");
      if (!is_integer(tbl.col_types[e.col_id].type)) fail(B2Q_ERR_UNSUPPORTED, "estimator over a floating-point key");
      if (is_date_in_days(tbl, e.col_id)) fail(B2Q_ERR_UNSUPPORTED, "estimator over a days-encoded DATE is outside the product path");
      plan.estimator_cols.push_back(e.col_id);
      p.group_col_ids[i] = e.col_id;
      p.group_col_widths[i] = static_cast<int8_t>(type_size(tbl.col_types[e.col_id].type));
    }
    p.num_group_cols = u.num_estimator_args;
    return plan;
  }
  if (u.num_order_entries < 0 || u.num_order_entries > 8) fail(B2Q_ERR_UNSUPPORTED, "more ORDER BY entries than the path carries");
  for (int i = 0; i < u.num_order_entries; ++i)
    if (u.order_entries[i].tle_no < 1 || u.order_entries[i].tle_no > u.num_target_exprs) fail(B2Q_ERR_INVALID_ARGUMENT, "order entry refers to a target that does not exist");
  if (u.offset < 0 || (u.has_limit && u.limit < 0)) fail(B2Q_ERR_INVALID_ARGUMENT, "negative LIMIT / OFFSET");
  for (int i = 0; i < u.num_order_entries; ++i) /* ResultSet::sort orders dictionary strings through the dictionary (ResultSet.cpp:1431-1446) */
    if (is_string(expr_at(u, u.target_exprs[u.order_entries[i].tle_no - 1]).ti.type)) fail(B2Q_ERR_UNSUPPORTED, "ORDER BY a dictionary-encoded string needs the dictionary");
  /* a DECIMAL compares as its scaled integer: both sides must already be at one scale, which is what the analyzer's
   * common_numeric_type + folded constant casts leave when the types agree (Analyzer.cpp BinOper::normalize); anything
   * else reaches the executor as a CAST node, which is outside this path */
  for (int i = 0; i < u.num_exprs; ++i) {
    const B2QExpr& e = u.exprs[i];
    if (e.kind != B2Q_EXPR_BIN_OPER || e.op == B2Q_kAND || e.op == B2Q_kOR || e.left < 0 || e.right < 0 || e.left >= u.num_exprs || e.right >= u.num_exprs) continue;
    const B2QTypeInfo& a = u.exprs[e.left].ti, &b = u.exprs[e.right].ti;
    if ((is_decimal(a.type) || is_decimal(b.type)) && !(is_decimal(a.type) && is_decimal(b.type) && a.scale == b.scale))
      fail(B2Q_ERR_UNSUPPORTED, "DECIMAL compared with a value of another type / scale needs the analyzer's cast");
  }
  if (u.num_groupby_exprs > B2Q_MAX_GROUP_COLS) fail(B2Q_ERR_UNSUPPORTED, "more GROUP BY columns than the path carries");
  if (u.num_target_exprs <= 0 || u.num_target_exprs > B2Q_MAX_TARGETS)
    fail(B2Q_ERR_INVALID_ARGUMENT, "bad target count");
  for (int c = 0; c < tbl.num_cols; ++c) {
    const bool is_deleted_col = tbl.deleted_column_plus1 == c + 1;
    if (tbl.col_types[c].type == B2Q_kBOOLEAN) { if (!is_deleted_col) fail(B2Q_ERR_UNSUPPORTED, "BOOLEAN is only supported as the deleted-rows column"); continue; }
    if (type_size(tbl.col_types[c].type) < 0) fail(B2Q_ERR_UNSUPPORTED, "column type outside the numeric / time / dictionary-string subset");
    if (tbl.col_encoded_sizes && tbl.col_encoded_sizes[c]) {
      const int e = tbl.col_encoded_sizes[c];
      if (e < 0) {
        if (tbl.col_types[c].type != B2Q_kDATE || (e != -4 && e != -2)) fail(B2Q_ERR_UNSUPPORTED, "ENCODING DAYS needs a DATE column and 32 or 16 bits");
      } else if (!is_integer(tbl.col_types[c].type) || (e != 1 && e != 2 && e != 4) || e >= type_size(tbl.col_types[c].type))
        fail(B2Q_ERR_UNSUPPORTED, "ENCODING FIXED needs an integer column and a physical width below the logical one");
    }
  }

  Plan plan;
  B2QPlan& p = plan.p;
  const bool bigint_count = eo.bigint_count != 0;
  const bool is_group_by = u.num_groupby_exprs >= 1;
  const bool multi_key = u.num_groupby_exprs > 1;

  for (int i = 0; i < u.num_target_exprs; ++i) plan.targets.push_back(get_target_info(u, u.target_exprs[i], bigint_count));
  bool any_agg = false;
  for (auto& t : plan.targets) any_agg |= t.is_agg;
  if (!any_agg) fail(B2Q_ERR_UNSUPPORTED, "projection queries are outside this path");
  for (int i = 0; i < u.num_order_entries; ++i) {
    const int tle = u.order_entries[i].tle_no;
    if (tle >= 1 && tle <= static_cast<int>(plan.targets.size()) && get_compact_type(plan.targets[tle - 1]).type == B2Q_kFLOAT)
      fail(B2Q_ERR_UNSUPPORTED, "ORDER BY a FLOAT target is outside the product path");
  }

  /* GroupByAndAggregate::getBaselineThreshold (:222-230): device_type is GPU on this path, so COUNT(DISTINCT) targets divide
   * g_baseline_groupby_threshold (1e6) by four */
  bool any_count_distinct = false;
  for (const auto& t : plan.targets) any_count_distinct |= t.is_distinct;
  const int64_t baseline_threshold = any_count_distinct ? 1000000 / 4 : 1000000;

  /* ---- hash type: GroupByAndAggregate::getColRangeInfo (:232-365) + get_expr_range_info (:181-218) ---- */
  int key_col = -1;
  Range key_range;
  if (multi_key) {
    /* getColRangeInfo, groupby_exprs.size() != 1 (GroupByAndAggregate.cpp:240-280): every column must have a valid
     * integer range; cardinality = product of the bucketed cardinalities; zero or > g_baseline_groupby_threshold
     * (1e6, Execute.cpp:111) => baseline hash, which for several key columns is outside this path. */
    int64_t cardinality = 1;
    bool has_nulls = false;
    for (int i = 0; i < u.num_groupby_exprs; ++i) {
      const B2QExpr& g = expr_at(u, u.groupby_exprs[i]);
      if (g.kind != B2Q_EXPR_COLUMN_VAR) fail(B2Q_ERR_UNSUPPORTED, "GROUP BY expression must be a ColumnVar");
      if (is_fp(tbl.col_types[g.col_id].type)) fail(B2Q_ERR_UNSUPPORTED, "multi-column baseline hash (fp key) is outside this path");
      Range r = leaf_column_range(tbl, g.col_id);
      apply_simple_quals(u, g.col_id, r);
      if (r.kind != Range::Integer || r.imin > r.imax) fail(B2Q_ERR_UNSUPPORTED, "multi-column baseline hash is outside this path");
      KeyCol k;
      k.col = g.col_id; k.min = r.imin; k.max = r.imax; k.has_nulls = r.has_nulls; k.bucket = r.bucket;
      int64_t span;
      const bool span_ovf = __builtin_sub_overflow(r.imax, r.imin, &span);
      if (!span_ovf && r.bucket) span /= r.bucket; /* getBucketedCardinality (:367-375) */
      if (span_ovf || __builtin_add_overflow(span, int64_t(1 + (r.has_nulls ? 1 : 0)), &k.card))
        fail(B2Q_ERR_UNSUPPORTED, "multi-column baseline hash is outside this path");
      k.mult = cardinality;
      if (__builtin_mul_overflow(cardinality, k.card, &cardinality)) fail(B2Q_ERR_UNSUPPORTED, "multi-column baseline hash is outside this path");
      has_nulls |= r.has_nulls;
      plan.keys.push_back(k);
      p.group_col_ids[i] = g.col_id;
      p.group_col_widths[i] = static_cast<int8_t>(type_size(tbl.col_types[g.col_id].type));
    }
    if (!cardinality || cardinality > baseline_threshold) fail(B2Q_ERR_UNSUPPORTED, "multi-column baseline hash is outside this path");
    p.query_desc_type = B2Q_GroupByPerfectHash;
    p.min_val = 0; p.max_val = cardinality; p.bucket = 0; p.has_nulls = has_nulls;
    key_col = plan.keys[0].col;
    p.group_col_width = p.group_col_widths[0];
  } else if (is_group_by) {
    const B2QExpr& g = expr_at(u, u.groupby_exprs[0]);
    if (g.kind != B2Q_EXPR_COLUMN_VAR) fail(B2Q_ERR_UNSUPPORTED, "GROUP BY expression must be a ColumnVar");
    key_col = g.col_id;
    key_range = leaf_column_range(tbl, key_col);
    apply_simple_quals(u, key_col, key_range);
    p.group_col_width = type_size(tbl.col_types[key_col].type);
    int hash_type;
    int64_t cmin = 0, cmax = 0, cbucket = 0;
    bool chas_nulls = false;
    if (key_range.kind == Range::Integer) {
      if (key_range.imin > key_range.imax) { /* :193-196 */
        hash_type = B2Q_GroupByBaselineHash; cmin = 0; cmax = -1; chas_nulls = key_range.has_nulls;
      } else {
        hash_type = B2Q_GroupByPerfectHash;
        cmin = key_range.imin; cmax = key_range.imax; cbucket = key_range.bucket; chas_nulls = key_range.has_nulls;
      }
    } else { /* Float/Double/Invalid => baseline (:203-212) */
      hash_type = B2Q_GroupByBaselineHash;
      if (key_range.kind == Range::Double && key_range.fmin > key_range.fmax) { cmax = -1; chas_nulls = key_range.has_nulls; }
    }
    if (hash_type == B2Q_GroupByPerfectHash) {
      /* :298-304 max_entry_count, :131-139 is_column_range_too_big_for_perfect_hash */
      const int64_t col_count = u.num_groupby_exprs + u.num_target_exprs;
      int64_t max_entry_count = kMaxBufferSize / (col_count * static_cast<int64_t>(sizeof(int64_t)));
      if (any_count_distinct) max_entry_count = std::min(max_entry_count, baseline_threshold); /* :307-309 */
      bool too_big;
      int64_t diff;
      if (__builtin_sub_overflow(cmax, cmin, &diff)) too_big = true; else too_big = diff >= max_entry_count;
      if (is_string(tbl.col_types[key_col].type) && !cbucket) {
        /* :311-356 dictionary ids are dense, so a too-big range stays perfect hash unless a filter can be expected to
         * thin it out: with filters and no sort, baseline when there is no estimate yet or 2 * estimate < range */
        const bool has_filters = u.num_quals > 0 || u.num_simple_quals > 0;
        if (has_filters && too_big && u.num_order_entries != 0) {
          /* :329-341 with a sort the original range is kept — except with COUNT(DISTINCT): "always use baseline hash for column
           * range too big for perfect hash with count distinct descriptors" */
          if (any_count_distinct) hash_type = B2Q_GroupByBaselineHash;
        } else if (has_filters && too_big) {
          int64_t twice;
          const bool less = has_cardinality_estimation &&
                            !__builtin_mul_overflow(static_cast<int64_t>(max_groups_buffer_entry_guess), int64_t(2), &twice) && twice < diff;
          if (!has_cardinality_estimation || less) hash_type = B2Q_GroupByBaselineHash; /* min/max kept */
        }
      } else if (too_big && !cbucket) hash_type = B2Q_GroupByBaselineHash; /* :357-363, min/max kept */
    }
    p.query_desc_type = hash_type;
    p.min_val = cmin; p.max_val = cmax; p.bucket = cbucket; p.has_nulls = chas_nulls;
  } else {
    p.query_desc_type = B2Q_NonGroupedAggregate;
    p.group_col_width = 0;
  }
  p.key_col_id = key_col;
  p.num_group_cols = u.num_groupby_exprs;
  if (!multi_key && is_group_by) { p.group_col_ids[0] = key_col; p.group_col_widths[0] = static_cast<int8_t>(p.group_col_width); }

  /* ---- keyless: initQueryMemoryDescriptorImpl :943-947 ---- */
  bool keyless = false;
  int32_t keyless_index = -1;
  if (is_group_by && p.query_desc_type == B2Q_GroupByPerfectHash)
    get_keyless_info(u, tbl, plan.targets, is_group_by, keyless, keyless_index);

  /* ---- slots: ColSlotContext ctor (ColSlotContext.cpp:35-101) ---- */
  std::vector<int8_t> logical;
  for (size_t ti = 0; ti < plan.targets.size(); ++ti) {
    auto& t = plan.targets[ti];
    t.first_slot = static_cast<int>(logical.size());
    const Ti chosen = get_compact_type(t);
    logical.push_back(static_cast<int8_t>(type_size(chosen.type)));
    plan.slot_compact_ti.push_back(chosen);
    if (t.is_agg && t.agg_kind == B2Q_kAVG) {
      logical.push_back(8);
      plan.slot_compact_ti.push_back(Ti{B2Q_kBIGINT, true});
    }
  }
  if (logical.size() > B2Q_MAX_SLOTS) fail(B2Q_ERR_UNSUPPORTED, "too many slots");

  /* ---- pick_target_compact_width (QueryMemoryDescriptor.cpp:748-842), crt_min_byte_width = 8 ---- */
  int8_t min_slot_size;
  {
    const int8_t crt_min_byte_width = 8;
    if (bigint_count) {
      min_slot_size = 8;
    } else {
      int8_t compact_width = 0;
      /* :775-778: `groupby_exprs.size() != 1 || !groupby_exprs.front()` — the non-grouped unit ({nullptr}) AND every multi-column
       * GROUP BY keep the 8-byte slots; only a single-column GROUP BY can compact to 4 */
      if (!is_group_by || u.num_groupby_exprs != 1) compact_width = crt_min_byte_width;
      if (!compact_width) {
        for (int i = 0; i < u.num_target_exprs; ++i) {
          const B2QExpr& e = expr_at(u, u.target_exprs[i]);
          if (e.kind == B2Q_EXPR_AGG && e.left >= 0) { compact_width = crt_min_byte_width; break; }
          if (e.kind == B2Q_EXPR_AGG) continue; /* COUNT(*) */
          if (is_integer(e.ti.type) && type_size(e.ti.type) <= 4) continue; /* is_int_and_no_bigger_than(ti,4) */
          compact_width = crt_min_byte_width;
          break;
        }
      }
      if (!compact_width) {
        /* :826-830: the tuples of every table in query_infos, the inner table of a join level included */
        uint64_t total_tuples = inner_tuples;
        for (int f = 0; f < tbl.num_fragments; ++f) total_tuples += tbl.fragments[f].num_tuples;
        min_slot_size = total_tuples <= std::numeric_limits<uint32_t>::max() ? 4 : crt_min_byte_width;
      } else {
        for (int i = 0; i < u.num_target_exprs; ++i) /* get_col_byte_widths(target_exprs) */
          compact_width = std::max<int8_t>(compact_width, static_cast<int8_t>(type_size(expr_at(u, u.target_exprs[i]).ti.type)));
        min_slot_size = compact_width;
      }
    }
  }

  /* ---- QueryMemoryDescriptor::init (:240-444) ---- */
  p.num_targets = static_cast<int32_t>(plan.targets.size());
  /* QueryMemoryDescriptor ctor (:510-536): no GPU sort on this path, so output_columnar_ is the hint for every
   * descriptor type we plan (no count-distinct / quantile / mode targets here) */
  p.output_columnar = eo.output_columnar_hint ? 1 : 0;
  p.interleaved_bins_on_gpu = 0;
  p.keyless_hash = 0;
  p.idx_target_as_key = -1;
  p.effective_key_width = 8;
  std::vector<bool> slot_is_key_ref(logical.size(), false); /* target_groupby_indices != -1 => 0-width slot */
  if (!is_group_by) {
    p.entry_count = 1;
  } else if (p.query_desc_type == B2Q_GroupByPerfectHash) {
    /* keyless_hash (:327-333): no sort hint, no bucket, no baseline sort in this path */
    p.keyless_hash = (!p.bucket && keyless) ? 1 : 0;
    p.idx_target_as_key = keyless_index;
    if (multi_key) {
      p.entry_count = p.max_val; /* col range info max contains the expected cardinality (QueryMemoryDescriptor.cpp:339-342) */
    } else {
      /* getBucketedCardinality (:367-375) */
      int64_t card;
      if (__builtin_sub_overflow(p.max_val, p.min_val, &card)) fail(B2Q_ERR_UNSUPPORTED, "DATE key range wider than int64 (undefined in the reference)");
      if (p.bucket) card /= p.bucket;
      card += 1 + (p.has_nulls ? 1 : 0);
      p.entry_count = std::max<int64_t>(card, 1);
    }
    /* interleaved_bins_on_gpu (:364-369) is a GPU-layout detail of the reference; the CPU path never has it */
  } else { /* baseline (:380-398) */
    if (is_date_in_days(tbl, key_col)) fail(B2Q_ERR_UNSUPPORTED, "baseline hash over a days-encoded DATE key is outside the product path");
    if (!has_cardinality_estimation) fail(B2Q_ERR_CARDINALITY_ESTIMATION_REQUIRED, "baseline hash needs a cardinality estimate");
    p.entry_count = static_cast<int64_t>(max_groups_buffer_entry_guess);
    if (p.entry_count <= 0) fail(B2Q_ERR_INVALID_ARGUMENT, "entry guess must be positive");
    /* target_expr_group_by_indices: targets that ARE the group key get 0-width slots */
    for (size_t ti = 0; ti < plan.targets.size(); ++ti) {
      const auto& t = plan.targets[ti];
      if (!t.is_agg && t.arg_col == key_col) slot_is_key_ref[t.first_slot] = true;
    }
    /* pick_baseline_key_width (:112-147) */
    int8_t kw = 4;
    {
      const Range er = leaf_column_range(tbl, key_col); /* no simple quals here (getExpressionRange w/o quals) */
      int8_t w;
      if (er.kind == Range::Invalid) w = 8;
      else if (er.kind == Range::Integer) {
        if (p.group_col_width == 8 && er.has_nulls) w = 8;
        else {
          /* is_valid_int32_range (QueryMemoryDescriptor.cpp:40-42): min > INT32_MIN && max < EMPTY_KEY_32 - 1 */
          const bool ok = er.imin > static_cast<int64_t>(INT32_MIN) && er.imax < static_cast<int64_t>(kEmptyKey32) - 1;
          w = ok ? 4 : 8;
        }
      } else w = 8;
      kw = std::max(kw, w);
    }
    p.effective_key_width = p.output_columnar ? 8 : kw; /* group_col_compact_width = output_columnar ? 8 : pick_baseline_key_width (:391-393) */
    p.min_val = 0; p.max_val = 0; p.bucket = 0; p.has_nulls = 0; /* actual_col_range_info reset (:396-397) */
  }

  /* padded widths: setAllSlotsPaddedSize(min_slot_size); 0-width for key-ref slots (addSlotForColumn(0,0)) */
  p.num_slots = static_cast<int32_t>(logical.size());
  for (size_t s = 0; s < logical.size(); ++s) {
    if (slot_is_key_ref[s]) { p.slot_logical_width[s] = 0; p.slot_padded_width[s] = 0; continue; }
    p.slot_logical_width[s] = logical[s];
    p.slot_padded_width[s] = min_slot_size;
    if (logical[s] > min_slot_size) fail(B2Q_ERR_UNSUPPORTED, "slot wider than compact width (ColSlotContext::validate)");
  }
  /* TargetExprCodegenBuilder::operator() (:614-621): non-grouped + slot < 8 => CompilationRetryNoCompaction;
   * the retry (Execute.cpp:2260) re-plans with 8-byte slots.  Non-grouped already forces 8 above. */

  /* ---- row size / offsets: getRowSize (:848-860), getColOffInBytes (:918-955), ColSlotContext alignment ---- */
  if (p.output_columnar) {
    /* columnar: [key columns: align8(max(width,8) * N) each, absent if keyless][slot columns: align8(w * N) each]
     * (getPrependedGroupBufferSizeInBytes :987-997, getColOffInBytes :920-944, getBufferSizeBytes :1084-1111) */
    if (is_group_by && !p.keyless_hash && p.group_col_widths[0] != 8)
      /* ResultSetStorage::isEmptyEntryColumnar (ResultSetIteration.cpp:2533-2543) indexes the first key column by
       * groupColWidth(0) — the COLUMN's width — although the column is stored as int64 (initColumnarGroups,
       * QueryMemoryInitializer.cpp:729-735): with a narrower key the reference's own reader and reduce misjudge
       * emptiness.  There is no well-defined result to match, so the layout is refused on both sides. */
      fail(B2Q_ERR_UNSUPPORTED, "columnar output with a stored GROUP BY key narrower than 8 bytes (reference reader reads it at the column's width)");
    int64_t off = 0;
    if (is_group_by && !p.keyless_hash) off = static_cast<int64_t>(u.num_groupby_exprs) * align_to_int64(8 * p.entry_count);
    for (int s = 0; s < p.num_slots; ++s) {
      p.slot_offset[s] = off;
      off += align_to_int64(static_cast<int64_t>(p.slot_padded_width[s]) * p.entry_count);
    }
    p.row_size = 0;
    for (int s = 0; s < p.num_slots; ++s) p.row_size += p.slot_padded_width[s]; /* getColsSize(); informational for columnar */
    p.row_size = align_to_int64(p.row_size);
    p.buffer_size = off;
  } else {
    int64_t off = 0;
    if (is_group_by && !p.keyless_hash) off = align_to_int64(static_cast<int64_t>(u.num_groupby_exprs) * p.effective_key_width);
    const int64_t key_bytes = off;
    int64_t cols = 0;
    for (int s = 0; s < p.num_slots; ++s) {
      const int w = p.slot_padded_width[s];
      if (w == 8) cols = align_to_int64(cols);
      p.slot_offset[s] = key_bytes + cols;
      cols += w;
    }
    p.row_size = align_to_int64(key_bytes + cols);
    p.buffer_size = p.row_size * p.entry_count;
  }

  /* ---- init vals: init_agg_val_vec (OutputBufferInitialization.cpp:26-86, :264-293) ---- */
  {
    int8_t compact_byte_width = 8; /* ColSlotContext::getCompactByteWidth: first non-zero padded size */
    for (int s = 0; s < p.num_slots; ++s) if (p.slot_padded_width[s]) { compact_byte_width = p.slot_padded_width[s]; break; }
    int s = 0;
    for (auto t : plan.targets) { /* by value: set_notnull only affects the init computation (:283-288) */
      if (t.arg_col >= 0 && t.is_agg && p.query_desc_type == B2Q_NonGroupedAggregate &&
          (t.agg_kind == B2Q_kMIN || t.agg_kind == B2Q_kMAX || t.agg_kind == B2Q_kSUM || t.agg_kind == B2Q_kAVG)) {
        t.sql_type.notnull = false; t.agg_arg_type.notnull = false; t.skip_null_val = true; /* set_notnull(target,false) */
      } else if (t.arg_col >= 0 && t.is_agg && t.arg_constrained_not_null) { /* :287-289 set_notnull(target, true) */
        t.sql_type.notnull = true; t.agg_arg_type.notnull = true; t.skip_null_val = false;
      }
      if (!t.is_agg) {
        p.init_vals[s] = 0;
        ++s;
        continue;
      }
      Ti init_ti = get_compact_type(t);
      if (!is_group_by) init_ti.notnull = false;
      p.init_vals[s++] = get_agg_initial_val(t.agg_kind, init_ti, is_group_by, compact_byte_width);
      if (t.agg_kind == B2Q_kAVG) p.init_vals[s++] = 0;
    }
  }

  /* ---- skip_null_val as the code generator sees it (TargetExprBuilder.cpp:648-662) + public target infos ---- */
  for (size_t i = 0; i < plan.targets.size(); ++i) {
    auto& t = plan.targets[i];
    if (t.arg_col >= 0 && t.is_agg && p.query_desc_type == B2Q_NonGroupedAggregate) t.skip_null_val = true;
    else if (t.arg_col >= 0 && t.is_agg && t.arg_constrained_not_null) t.skip_null_val = false; /* TargetExprBuilder.cpp:690-692 */
    B2QTargetInfo& o = p.targets[i];
    o.is_agg = t.is_agg; o.agg_kind = t.agg_kind;
    o.sql_type = B2QTypeInfo{t.sql_type.type, t.sql_type.notnull, t.sql_type.scale};
    o.agg_arg_type = B2QTypeInfo{t.agg_arg_type.type, t.agg_arg_type.notnull, t.agg_arg_type.scale};
    o.skip_null_val = t.skip_null_val; o.is_distinct = t.is_distinct ? 1 : 0; o.arg_col_id = t.arg_col; o.first_slot = t.first_slot;
  }
  /* ---- init_count_distinct_descriptors (GroupByAndAggregate.cpp:650-855) for COUNT(DISTINCT column) on the GPU:
   * arg_range_info = get_expr_range_info (:181-218: the column's chunk-stats range narrowed by the simple quals);
   * empty range -> Bitmap of 64 bits at min 0 (:735-744); integer range -> Bitmap of get_bucketed_cardinality_without_nulls
   * bits (:379-395) unless that is <= 0 or >= g_bitmap_memory_limit (8e9, QueryMemoryInitializer.cpp:28) or the bitmaps of
   * the whole group range would reach the limit (:755-832) — then the std::set implementation or an exception; fp / invalid
   * ranges are the set implementation from the start.  Sets do not run on the reference's GPU (QueryMustRunOnCpu), so they
   * are refused.  check_total_bitmap_memory (QueryMemoryInitializer.cpp:40-66) bounds bytes per group x entry count. ---- */
  {
    const int64_t limit = 8000000000ll;
    int64_t bytes_per_group = 0, tail = p.buffer_size;
    for (size_t i = 0; i < plan.targets.size(); ++i) {
      auto& t = plan.targets[i];
      p.count_distinct_min[i] = p.count_distinct_bits[i] = 0;
      if (!t.is_distinct) continue;
      if (is_fp(tbl.col_types[t.arg_col].type)) fail(B2Q_ERR_UNSUPPORTED, "COUNT(DISTINCT) of a floating-point column: set implementation, CPU only");
      if (is_date_in_days(tbl, t.arg_col)) fail(B2Q_ERR_UNSUPPORTED, "COUNT(DISTINCT) of a days-encoded DATE is outside the product path");
      Range r = leaf_column_range(tbl, t.arg_col);
      apply_simple_quals(u, t.arg_col, r);
      if (r.kind != Range::Integer) fail(B2Q_ERR_UNSUPPORTED, "COUNT(DISTINCT): no integer range: set implementation, CPU only");
      if (r.imin > r.imax) { t.cd_min = 0; t.cd_bucket = r.bucket; t.cd_bits = 64; }
      else {
        uint64_t size = static_cast<uint64_t>(r.imax) - static_cast<uint64_t>(r.imin);
        if (r.bucket) size /= static_cast<uint64_t>(r.bucket);
        const int64_t bits = size >= static_cast<uint64_t>(std::numeric_limits<int64_t>::max()) ? 0 : static_cast<int64_t>(size + 1);
        if (bits <= 0 || limit <= bits) fail(B2Q_ERR_UNSUPPORTED, "COUNT(DISTINCT): range too wide for a bitmap: set implementation, CPU only");
        const int64_t padded = align_to_int64((bits + 7) / 8);
        int64_t groups = 1;
        if (is_group_by) groups = p.max_val >= p.min_val ? (p.max_val - p.min_val + 1) / std::max<int64_t>(p.bucket, 1) : 0;
        if (groups > 0 && padded >= (limit + groups - 1) / groups) fail(B2Q_ERR_UNSUPPORTED, "COUNT(DISTINCT): bitmaps over the group range reach g_bitmap_memory_limit: set implementation or an error");
        t.cd_min = r.imin; t.cd_bucket = r.bucket; t.cd_bits = bits;
      }
      const int64_t padded = align_to_int64((t.cd_bits + 7) / 8);
      bytes_per_group += padded;
      t.cd_tail = tail;
      tail += padded * std::max<int64_t>(p.entry_count, 1);
      p.count_distinct_min[i] = t.cd_min;
      p.count_distinct_bits[i] = t.cd_bits;
    }
    if (bytes_per_group && p.entry_count > 0 && bytes_per_group >= (limit + p.entry_count - 1) / p.entry_count)
      fail(B2Q_ERR_OUT_OF_GPU_MEM, "COUNT(DISTINCT) bitmaps reach g_bitmap_memory_limit (OutOfHostMemory)");
    plan.cd_total = tail - p.buffer_size;
  }
  p.kernel = 0;
  p.join_outer_col = p.join_inner_col = -1;
  return plan;
}

/* ---- one INNER hash-join level -------------------------------------------------------------------------------
 * The unit is rewritten over a combined table: columns [0, n_outer) are the outer table's, [n_outer, n_outer +
 * n_inner) the inner table's (ColumnVar rte_idx 1); every fragment of the combined table pairs one outer fragment
 * with the (single, concatenated) inner fragment. */
struct JoinedInput {
  bool active{false};
  std::vector<B2QExpr> exprs;
  B2QExecUnit u{};
  std::vector<B2QTypeInfo> col_types;
  std::vector<int8_t> enc;
  std::vector<std::vector<const void*>> bufs;
  std::vector<std::vector<B2QChunkStats>> stats;
  std::vector<B2QFragmentInfo> frags;
  B2QTableInfo t{};
  int n_outer{0};
  int outer_col{-1}, inner_vcol{-1};
  bool left{false};
};

void build_joined_input(const B2QExecUnit& u, const B2QTableInfo& outer, JoinedInput& ji) {
  if (u.num_join_quals != 1) fail(B2Q_ERR_UNSUPPORTED, "more than one join level is outside this path");
  if (u.join_type != 0 && u.join_type != 1) fail(B2Q_ERR_UNSUPPORTED, "only INNER and LEFT joins are on this path");
  const bool left = u.join_type == 1;
  if (!u.inner_table) fail(B2Q_ERR_INVALID_ARGUMENT, "join without an inner table");
  const B2QTableInfo& inner = *u.inner_table;
  if (inner.num_fragments > 1) fail(B2Q_ERR_INVALID_ARGUMENT, "the inner table must come as one concatenated fragment (getAllTableColumnFragments)");
  if (inner.deleted_column_plus1) fail(B2Q_ERR_UNSUPPORTED, "inner table with a deleted-rows column");
  if (inner.memory_level != B2Q_CPU_LEVEL) fail(B2Q_ERR_INVALID_ARGUMENT, "oracle needs host column buffers");
  ji.active = true;
  ji.n_outer = outer.num_cols;
  const int n_inner = inner.num_cols;
  ji.exprs.assign(u.exprs, u.exprs + u.num_exprs);
  for (auto& e : ji.exprs) {
    if (e.kind != B2Q_EXPR_COLUMN_VAR) continue;
    if (e.rte_idx == 1) {
      if (e.col_id < 0 || e.col_id >= n_inner) fail(B2Q_ERR_INVALID_ARGUMENT, "inner column id out of range");
      /* RelAlgTranslator hands a LEFT join's inner columns over as nullable; a NOT NULL one would mis-plan */
      if (left && e.ti.notnull) fail(B2Q_ERR_INVALID_ARGUMENT, "LEFT join: inner ColumnVars must be nullable");
      e.col_id += ji.n_outer;
      e.rte_idx = 0;
    } else if (e.rte_idx != 0) fail(B2Q_ERR_UNSUPPORTED, "rte_idx beyond one join level");
  }
  ji.u = u;
  ji.u.exprs = ji.exprs.data();
  ji.u.num_join_quals = 0;
  ji.u.inner_table = nullptr;
  /* the qual: ColumnVar = ColumnVar, one side per table (normalizeColumnPairs, HashJoin.cpp) */
  const B2QExpr& q = expr_at(ji.u, u.join_qual);
  if (q.kind != B2Q_EXPR_BIN_OPER || q.op != B2Q_kEQ) fail(B2Q_ERR_UNSUPPORTED, "join qual must be an equality");
  const B2QExpr& a = expr_at(ji.u, q.left);
  const B2QExpr& b = expr_at(ji.u, q.right);
  if (a.kind != B2Q_EXPR_COLUMN_VAR || b.kind != B2Q_EXPR_COLUMN_VAR) fail(B2Q_ERR_UNSUPPORTED, "join qual must compare two ColumnVars");
  const bool a_inner = a.col_id >= ji.n_outer, b_inner = b.col_id >= ji.n_outer;
  if (a_inner == b_inner) fail(B2Q_ERR_UNSUPPORTED, "join qual must compare an outer with an inner column");
  ji.outer_col = a_inner ? b.col_id : a.col_id;
  ji.inner_vcol = a_inner ? a.col_id : b.col_id;
  /* combined table */
  ji.col_types.assign(outer.col_types, outer.col_types + outer.num_cols);
  ji.col_types.insert(ji.col_types.end(), inner.col_types, inner.col_types + n_inner);
  if (left) for (int c = 0; c < n_inner; ++c) ji.col_types[ji.n_outer + c].notnull = 0;
  ji.left = left;
  ji.enc.assign(ji.col_types.size(), 0);
  for (int c = 0; c < outer.num_cols; ++c) if (outer.col_encoded_sizes) ji.enc[c] = outer.col_encoded_sizes[c];
  for (int c = 0; c < n_inner; ++c) if (inner.col_encoded_sizes) ji.enc[ji.n_outer + c] = inner.col_encoded_sizes[c];
  const B2QFragmentInfo* inf = inner.num_fragments ? &inner.fragments[0] : nullptr;
  ji.bufs.resize(outer.num_fragments);
  ji.stats.resize(outer.num_fragments);
  ji.frags.resize(outer.num_fragments);
  for (int f = 0; f < outer.num_fragments; ++f) {
    const B2QFragmentInfo& of = outer.fragments[f];
    if (of.col_buffers) ji.bufs[f].assign(of.col_buffers, of.col_buffers + outer.num_cols);
    else ji.bufs[f].assign(static_cast<size_t>(outer.num_cols), nullptr); /* a stats-only fragment: chunk stats, no data */
    ji.stats[f].assign(of.col_stats, of.col_stats + outer.num_cols);
    for (int c = 0; c < n_inner; ++c) {
      ji.bufs[f].push_back(inf ? inf->col_buffers[c] : nullptr);
      B2QChunkStats empty{};
      empty.int_min = INT64_MAX; empty.int_max = INT64_MIN; empty.fp_min = DBL_MAX; empty.fp_max = -DBL_MAX;
      ji.stats[f].push_back(inf ? inf->col_stats[c] : empty);
      if (left) ji.stats[f].back().has_nulls = 1; /* is_outer_join_proj: getLeafColumnRange starts from has_nulls = true (ExpressionRange.cpp:521-525, :642-652) */
    }
    ji.frags[f] = of;
    ji.frags[f].col_buffers = of.col_buffers ? ji.bufs[f].data() : nullptr;
    ji.frags[f].col_stats = ji.stats[f].data();
  }
  ji.t = outer;
  ji.t.num_cols = static_cast<int32_t>(ji.col_types.size());
  ji.t.col_types = ji.col_types.data();
  ji.t.col_encoded_sizes = ji.enc.data();
  ji.t.fragments = ji.frags.data();
}

/* PerfectJoinHashTable::getInstance (JoinHashTable/PerfectJoinHashTable.cpp:168-300): the table spans the INNER
 * column's range; too sparse a range switches the reference to a baseline join table, outside this path. */
Plan make_plan(const B2QExecUnit& u, const B2QTableInfo& tbl, const B2QExecutionOptions& eo,
               size_t max_groups_buffer_entry_guess, bool has_cardinality_estimation, JoinedInput* ji_out = nullptr) {
  if (!u.num_join_quals) return make_plan_single(u, tbl, eo, max_groups_buffer_entry_guess, has_cardinality_estimation);
  JoinedInput local;
  JoinedInput& ji = ji_out ? *ji_out : local;
  build_joined_input(u, tbl, ji);
  const Ti oti = ti_of(ji.t.col_types[ji.outer_col]), iti = ti_of(ji.t.col_types[ji.inner_vcol]);
  if (!is_integer(oti.type) || !is_integer(iti.type) || is_string(oti.type) || is_string(iti.type))
    fail(B2Q_ERR_UNSUPPORTED, "join keys must be integer columns (dictionary translation is outside this path)");
  if (is_decimal(oti.type) || is_decimal(iti.type)) fail(B2Q_ERR_UNSUPPORTED, "DECIMAL join keys are outside this path");
  if (is_date_in_days(ji.t, ji.outer_col) || is_date_in_days(ji.t, ji.inner_vcol)) fail(B2Q_ERR_UNSUPPORTED, "days-encoded DATE join keys are outside the product path");
  const B2QTableInfo& inner = *u.inner_table;
  uint64_t inner_tuples = 0;
  for (int f = 0; f < inner.num_fragments; ++f) inner_tuples += inner.fragments[f].num_tuples;
  Plan plan = make_plan_single(ji.u, ji.t, eo, max_groups_buffer_entry_guess, has_cardinality_estimation, inner_tuples);
  Range r; /* getExpressionRange(inner_col): over the inner table alone */
  {
    B2QTableInfo it = inner;
    r = leaf_column_range(it, ji.inner_vcol - ji.n_outer);
  }
  if (r.kind != Range::Integer) fail(B2Q_ERR_UNSUPPORTED, "could not compute the range of the join column (HashJoinFail)");
  int64_t entries = 0;
  if (r.imin <= r.imax && (__builtin_sub_overflow(r.imax, r.imin, &entries) || __builtin_add_overflow(entries, int64_t(1), &entries) || entries > INT32_MAX))
    fail(B2Q_ERR_UNSUPPORTED, "too many hash entries for a perfect join table (TooManyHashEntries)");
  const int64_t inner_rows = inner.num_fragments ? inner.fragments[0].num_tuples : 0;
  /* deploy_baseline_join (:235-246): g_ratio_num_hash_entry_to_num_tuple_switch_to_baseline = 100 (Execute.cpp:104) */
  if (inner_rows * 100 < entries) fail(B2Q_ERR_UNSUPPORTED, "join column range too wide for its row count: the reference switches to a baseline join table");
  plan.join = true;
  plan.join_outer_col = ji.outer_col;
  plan.join_inner_vcol = ji.inner_vcol;
  plan.join_outer_nullable = !oti.notnull;
  plan.join_left = ji.left;
  plan.p.join_min_key = r.imin;
  plan.p.join_max_key = r.imax;
  plan.p.join_entry_count = entries;
  plan.p.join_outer_col = ji.outer_col;
  plan.p.join_inner_col = ji.inner_vcol - ji.n_outer;
  return plan;
}

/* fill_hash_join_buff (JoinHashTable/Runtime/HashJoinRuntime.cpp:120-216, one-to-one): slot[key - min] = inner row,
 * NULL keys are skipped, a second row for a slot means the join is not one-to-one (NeedsOneToManyHash) */
void build_join_table(Plan& plan, const JoinedInput& ji, const B2QTableInfo& inner) {
  auto buff = std::make_shared<std::vector<int32_t>>(static_cast<size_t>(plan.p.join_entry_count), -1);
  if (inner.num_fragments && plan.p.join_entry_count > 0) {
    const B2QFragmentInfo& fr = inner.fragments[0];
    const int c = ji.inner_vcol - ji.n_outer;
    const int ctype = inner.col_types[c].type;
    const bool nullable = !inner.col_types[c].notnull;
    for (int64_t row = 0; row < fr.num_tuples; ++row) {
      const int64_t key = decode_int_column(inner, fr, c, row);
      if (nullable && key == inline_int_null_val(ctype)) continue;
      if (key < plan.p.join_min_key || key > plan.p.join_max_key) fail(B2Q_ERR_KEY_OUT_OF_RANGE, "inner join key outside its chunk-stats range");
      int32_t& slot = (*buff)[static_cast<size_t>(key - plan.p.join_min_key)];
      if (slot != -1) fail(B2Q_ERR_UNSUPPORTED, "join is not one-to-one (the reference rebuilds a one-to-many table)");
      slot = static_cast<int32_t>(row);
    }
  }
  plan.join_buff = buff;
}

/* ===================================================================================================
 * Filter: quals evaluated with the nullable compare semantics of RuntimeFunctions.cpp:73-107
 * (DEF_CMP_NULLABLE: lhs OP rhs if neither is the NULL sentinel else null_bool_val = INT8_MIN) and the
 * nullable logical_and / logical_or of RuntimeFunctions.cpp:320-357; a row passes iff the final value > 0
 * (CodeGenerator::toBool, LogicalIR.cpp:344-352).
 * ================================================================================================= */
constexpr int8_t kNullBool = INT8_MIN;

struct Frag {
  const B2QFragmentInfo* fi;
};

int8_t eval_bool(const B2QExecUnit& u, const B2QTableInfo& tbl, const B2QFragmentInfo& fr, int expr_idx, int64_t pos) {
  const B2QExpr& e = expr_at(u, expr_idx);
  if (e.kind == B2Q_EXPR_UOPER) {
    if (e.op == B2Q_kNOT) { /* logical_not (RuntimeFunctions.cpp:331-334) */
      const int8_t v = eval_bool(u, tbl, fr, e.left, pos);
      return v == kNullBool ? v : (v ? 0 : 1);
    }
    if (e.op == B2Q_kISNULL) { /* CodeGenerator::codegenIsNull / codegenIsNullNumber (LogicalIR.cpp:381-432) */
      const B2QExpr& o = expr_at(u, e.left);
      if (o.kind != B2Q_EXPR_COLUMN_VAR) fail(B2Q_ERR_UNSUPPORTED, "IS NULL operand must be a ColumnVar");
      const int ctype = tbl.col_types[o.col_id].type;
      if (tbl.col_types[o.col_id].notnull) return 0; /* inferred non-null: short-circuit to false */
      if (is_fp(ctype)) return decode_double_column(ctype, fr, o.col_id, pos) == fp_null_of(ctype);
      return decode_int_column(tbl, fr, o.col_id, pos) == inline_int_null_val(ctype);
    }
    fail(B2Q_ERR_UNSUPPORTED, "unary operator outside NOT / IS NULL");
  }
  if (e.kind != B2Q_EXPR_BIN_OPER) fail(B2Q_ERR_UNSUPPORTED, "qual must be a BinOper or NOT / IS NULL");
  if (e.op == B2Q_kAND || e.op == B2Q_kOR) {
    const int8_t lhs = eval_bool(u, tbl, fr, e.left, pos);
    const int8_t rhs = eval_bool(u, tbl, fr, e.right, pos);
    if (e.op == B2Q_kAND) { /* logical_and (:320-337) */
      if (lhs == kNullBool) return rhs == 0 ? rhs : kNullBool;
      if (rhs == kNullBool) return lhs == 0 ? lhs : kNullBool;
      return (lhs && rhs) ? 1 : 0;
    }
    /* logical_or (:339-357) */
    if (lhs == kNullBool) return rhs == 0 ? kNullBool : rhs;
    if (rhs == kNullBool) return lhs == 0 ? kNullBool : lhs;
    return (lhs || rhs) ? 1 : 0;
  }
  const B2QExpr& l = expr_at(u, e.left);
  const B2QExpr& r = expr_at(u, e.right);
  if (l.kind == B2Q_EXPR_COLUMN_VAR && r.kind == B2Q_EXPR_COLUMN_VAR) {
    /* ColumnVar OP ColumnVar: both sides cast to their common type by the analyzer (integers to the wider integer,
     * anything with a DOUBLE to DOUBLE), then the nullable compare: NULL on either side -> NULL */
    const int lt = tbl.col_types[l.col_id].type, rt = tbl.col_types[r.col_id].type;
    if (is_string(lt) != is_string(rt) || (is_string(lt) && e.op != B2Q_kEQ && e.op != B2Q_kNE))
      fail(B2Q_ERR_UNSUPPORTED, "dictionary-encoded strings compare by id: only = and <> between two string columns of one dictionary");
    if (is_date_in_days(tbl, l.col_id) != is_date_in_days(tbl, r.col_id)) fail(B2Q_ERR_UNSUPPORTED, "days-encoded DATE compared with a column of another encoding is outside the product path");
    const bool lnn = tbl.col_types[l.col_id].notnull != 0, rnn = tbl.col_types[r.col_id].notnull != 0;
    if (is_fp(lt) || is_fp(rt)) {
      double a, b;
      bool an, bn;
      if (is_fp(lt)) { a = decode_double_column(lt, fr, l.col_id, pos); an = !lnn && a == fp_null_of(lt); }
      else { const int64_t v = decode_int_column(tbl, fr, l.col_id, pos); an = !lnn && v == inline_int_null_val(lt); a = static_cast<double>(v); }
      if (is_fp(rt)) { b = decode_double_column(rt, fr, r.col_id, pos); bn = !rnn && b == fp_null_of(rt); }
      else { const int64_t v = decode_int_column(tbl, fr, r.col_id, pos); bn = !rnn && v == inline_int_null_val(rt); b = static_cast<double>(v); }
      if (an || bn) return kNullBool;
      switch (e.op) {
        case B2Q_kEQ: return a == b; case B2Q_kNE: return a != b; case B2Q_kLT: return a < b;
        case B2Q_kGT: return a > b; case B2Q_kLE: return a <= b; case B2Q_kGE: return a >= b;
        default: fail(B2Q_ERR_UNSUPPORTED, "comparison operator");
      }
    }
    const int64_t a = decode_int_column(tbl, fr, l.col_id, pos), b = decode_int_column(tbl, fr, r.col_id, pos);
    if ((!lnn && a == inline_int_null_val(lt)) || (!rnn && b == inline_int_null_val(rt))) return kNullBool;
    switch (e.op) {
      case B2Q_kEQ: return a == b; case B2Q_kNE: return a != b; case B2Q_kLT: return a < b;
      case B2Q_kGT: return a > b; case B2Q_kLE: return a <= b; case B2Q_kGE: return a >= b;
      default: fail(B2Q_ERR_UNSUPPORTED, "comparison operator");
    }
  }
  if (l.kind != B2Q_EXPR_COLUMN_VAR || r.kind != B2Q_EXPR_CONSTANT)
    fail(B2Q_ERR_UNSUPPORTED, "comparison must be ColumnVar OP Constant or ColumnVar OP ColumnVar");
  const int col = l.col_id;
  const int ctype = tbl.col_types[col].type;
  const bool col_notnull = tbl.col_types[col].notnull != 0;
  /* dictionary strings compare by id against a literal's id (CompareIR.cpp codegenStrCmp / translated literal):
   * only = and <> mean anything without the dictionary */
  if (is_string(ctype) && e.op != B2Q_kEQ && e.op != B2Q_kNE) fail(B2Q_ERR_UNSUPPORTED, "dictionary-encoded strings compare by id: only = and <> are on this path");
  if (is_string(ctype) && is_fp(r.ti.type)) fail(B2Q_ERR_INVALID_ARGUMENT, "string column compared with a floating-point constant");
  if (r.is_null) return kNullBool;
  if (is_fp(ctype) || is_fp(r.ti.type)) {
    /* fp compare: the integer side is cast to double (CompareIR.cpp codegenCmp after normalisation) */
    double lv;
    bool lnull;
    if (is_fp(ctype)) { lv = decode_double_column(ctype, fr, col, pos); lnull = !col_notnull && lv == fp_null_of(ctype); }
    else { const int64_t iv = decode_int_column(tbl, fr, col, pos); lnull = !col_notnull && iv == inline_int_null_val(ctype); lv = static_cast<double>(iv); }
    if (lnull) return kNullBool;
    const double rv = is_fp(r.ti.type) ? r.dval : static_cast<double>(r.ival);
    switch (e.op) {
      case B2Q_kEQ: return lv == rv; case B2Q_kNE: return lv != rv; case B2Q_kLT: return lv < rv;
      case B2Q_kGT: return lv > rv; case B2Q_kLE: return lv <= rv; case B2Q_kGE: return lv >= rv;
      default: fail(B2Q_ERR_UNSUPPORTED, "comparison operator");
    }
  }
  const int64_t lv = decode_int_column(tbl, fr, col, pos);
  if (!col_notnull && lv == inline_int_null_val(ctype)) return kNullBool;
  const int64_t rv = r.ival;
  switch (e.op) {
    case B2Q_kEQ: return lv == rv; case B2Q_kNE: return lv != rv; case B2Q_kLT: return lv < rv;
    case B2Q_kGT: return lv > rv; case B2Q_kLE: return lv <= rv; case B2Q_kGE: return lv >= rv;
    default: fail(B2Q_ERR_UNSUPPORTED, "comparison operator");
  }
}

bool g_filter_deleted = true; /* CompilationOptions::filter_on_deleted_column (set per oracle_execute call) */

bool row_passes(const B2QExecUnit& u, const B2QTableInfo& tbl, const B2QFragmentInfo& fr, int64_t pos) {
  /* codegenSkipDeletedOuterTableRow (NativeCodegen.cpp:3419-3451): toBool($deleted$) => the row function returns 0 */
  if (g_filter_deleted && tbl.deleted_column_plus1 > 0) {
    const int8_t d = static_cast<const int8_t*>(fr.col_buffers[tbl.deleted_column_plus1 - 1])[pos];
    if (d > 0) return false;
  }
  /* simple_quals and quals are AND-ed: each must be TRUE (`filter_lv = AND of toBool(qual)`, NativeCodegen.cpp:3455+) */
  for (int i = 0; i < u.num_simple_quals; ++i) if (!(eval_bool(u, tbl, fr, u.simple_quals[i], pos) > 0)) return false;
  for (int i = 0; i < u.num_quals; ++i) if (!(eval_bool(u, tbl, fr, u.quals[i], pos) > 0)) return false;
  return true;
}

/* ===================================================================================================
 * Per-target aggregate update, as emitted by TargetExprCodegen::codegenAggregate
 * (TargetExprBuilder.cpp:470-583): value conversion (convertNullIfAny, GroupByAndAggregate.cpp:1599-1660),
 * cast to the slot width, `_skip_val` variant when target_info.skip_null_val.
 * All slots are 8 bytes wide here except the COUNT(*)-only 4-byte layout, which uses the _int32 variants.
 * ================================================================================================= */
/* where entry `e` keeps slot `s` / key column `c`: row-wise rows (ResultSet.h:55-70) or columnar (:72-84) */
template <class B>
inline B* slot_ptr(const B2QPlan& p, B* buf, int64_t e, int s) {
  return p.output_columnar ? buf + p.slot_offset[s] + e * p.slot_padded_width[s] : buf + e * p.row_size + p.slot_offset[s];
}
template <class B>
inline B* key_ptr(const B2QPlan& p, B* buf, int64_t e, int c) {
  return p.output_columnar ? buf + c * align_to_int64(8 * p.entry_count) + e * 8 : buf + e * p.row_size + c * p.effective_key_width;
}

void update_target(const Plan& plan, const Target& t, int8_t* out, int64_t entry, const B2QTableInfo& tbl,
                   const B2QFragmentInfo& fr, int64_t pos) {
  const B2QPlan& p = plan.p;
  const int s = t.first_slot;
  const int w = p.slot_padded_width[s];
  if (w == 0) return; /* baseline: group-key targets are read from the key columns */
  int8_t* slot = slot_ptr(p, out, entry, s);
  if (w == 4) {
    /* only reachable for COUNT(*) / small-int key projections (pick_target_compact_width) */
    int32_t* a = reinterpret_cast<int32_t*>(slot);
    if (!t.is_agg) { *a = static_cast<int32_t>(decode_int_column(tbl, fr, t.arg_col, pos)); return; } /* agg_id_int32 */
    if (t.agg_kind == B2Q_kCOUNT && t.arg_col < 0) { *reinterpret_cast<uint32_t*>(a) += 1; return; } /* agg_count_int32 */
    fail(B2Q_ERR_UNSUPPORTED, "4-byte slot with an aggregate argument");
  }
  int64_t* a = reinterpret_cast<int64_t*>(slot);
  if (!t.is_agg) { /* agg_id on the projected group key, sign-extended to the slot */
    const int ctype = tbl.col_types[t.arg_col].type;
    if (is_fp(ctype)) agg_id(a, bits_of(decode_double_column(ctype, fr, t.arg_col, pos)));
    else agg_id(a, decode_int_column(tbl, fr, t.arg_col, pos));
    return;
  }
  if (t.agg_kind == B2Q_kCOUNT && t.arg_col < 0) { agg_count(a); return; }
  if (t.is_distinct) {
    /* agg_count_distinct_bitmap[_skip_val] (RuntimeFunctions.cpp:366-376, :1201-1210); *agg is the group's bitmap */
    const int64_t v = decode_int_column(tbl, fr, t.arg_col, pos);
    if (t.skip_null_val && v == inline_int_null_val(tbl.col_types[t.arg_col].type)) return;
    uint64_t bitmap_idx = static_cast<uint64_t>(v - t.cd_min);
    if (1 < t.cd_bucket) bitmap_idx /= static_cast<uint64_t>(t.cd_bucket);
    if (bitmap_idx >= static_cast<uint64_t>(t.cd_bits)) fail(B2Q_ERR_KEY_OUT_OF_RANGE, "COUNT(DISTINCT) value outside the chunk-stats range");
    int8_t* bitmap = out + t.cd_tail + entry * align_to_int64((t.cd_bits + 7) / 8);
    bitmap[bitmap_idx >> 3] |= static_cast<int8_t>(1 << (bitmap_idx & 7));
    return;
  }
  const int ctype = tbl.col_types[t.arg_col].type;
  const bool arg_notnull = t.arg_ti.notnull;
  const bool need_skip_null = t.skip_null_val;
  if (ctype == B2Q_kFLOAT && t.agg_kind != B2Q_kCOUNT) {
    /* takes_float_argument (TargetInfo.h:106-110): agg_{sum,min,max}_float[_skip_val] on the slot's low 4 bytes
     * (RuntimeFunctions.cpp:1496-1518, DEF_SKIP_AGG :1558-1596); AVG keeps its count in the 8-byte slot that follows */
    const float v = static_cast<float>(decode_double_column(ctype, fr, t.arg_col, pos));
    int32_t* a32 = reinterpret_cast<int32_t*>(slot);
    auto apply = [&](int kind) {
      float cur;
      memcpy(&cur, a32, 4);
      const float r = kind == B2Q_kMIN ? std::min(cur, v) : kind == B2Q_kMAX ? std::max(cur, v) : cur + v;
      memcpy(a32, &r, 4);
    };
    const int kind = t.agg_kind == B2Q_kAVG ? B2Q_kSUM : t.agg_kind;
    if (need_skip_null) {
      if (v != kNullFloat) { /* DEF_SKIP_AGG: the old value is compared bitwise with the skip pattern */
        if (*a32 != static_cast<int32_t>(float_bits(kNullFloat))) apply(kind); else memcpy(a32, &v, 4);
        if (t.agg_kind == B2Q_kAVG) agg_count(reinterpret_cast<int64_t*>(slot_ptr(p, out, entry, s + 1)));
      }
    } else {
      apply(kind);
      if (t.agg_kind == B2Q_kAVG) agg_count(reinterpret_cast<int64_t*>(slot_ptr(p, out, entry, s + 1)));
    }
    return;
  }
  if (is_fp(ctype)) {
    const double v = decode_double_column(ctype, fr, t.arg_col, pos);
    const double null_v = fp_null_of(ctype); /* arg null == agg null for DOUBLE; COUNT(float): value and NULL_FLOAT are fpext-ed (agg_count_double_skip_val) */
    switch (t.agg_kind) {
      case B2Q_kCOUNT: if (need_skip_null) agg_count_double_skip_val(a, v, null_v); else agg_count(a); break;
      case B2Q_kSUM: if (need_skip_null) agg_sum_double_skip_val(a, v, null_v); else agg_sum_double(a, v); break;
      case B2Q_kMIN: if (need_skip_null) agg_min_double_skip_val(a, v, null_v); else agg_min_double(a, v); break;
      case B2Q_kMAX: if (need_skip_null) agg_max_double_skip_val(a, v, null_v); else agg_max_double(a, v); break;
      case B2Q_kAVG: {
        int64_t* cnt = reinterpret_cast<int64_t*>(slot_ptr(p, out, entry, s + 1));
        if (need_skip_null) { agg_sum_double_skip_val(a, v, null_v); agg_count_double_skip_val(cnt, v, null_v); }
        else { agg_sum_double(a, v); agg_count(cnt); }
        break;
      }
      default: abort();
    }
    return;
  }
  /* integer argument */
  int64_t v = decode_int_column(tbl, fr, t.arg_col, pos);
  int64_t null_v;
  if (is_agg_domain_range_equivalent(t.agg_kind)) {
    null_v = inline_int_null_val(ctype); /* inlineIntNull(arg_ti) sign-extended to 64 bits (:548-556) */
  } else {
    const int agg_type = t.sql_type.type; /* BIGINT for SUM/AVG over ints; INT/BIGINT for COUNT */
    null_v = inline_int_null_val(agg_type);
    if (need_skip_null && !arg_notnull) { /* convertNullIfAny: arg NULL -> agg NULL, else cast to the agg type */
      if (v == inline_int_null_val(ctype)) v = null_v;
      else if (type_size(agg_type) == 4) v = static_cast<int32_t>(v); /* castToTypeIn(32) then sext to the slot */
    }
  }
  switch (t.agg_kind) {
    case B2Q_kCOUNT: if (need_skip_null) agg_count_skip_val(a, v, null_v); else agg_count(a); break;
    case B2Q_kSUM: if (need_skip_null) agg_sum_skip_val(a, v, null_v); else agg_sum(a, v); break;
    case B2Q_kMIN: if (need_skip_null) agg_min_skip_val(a, v, null_v); else agg_min(a, v); break;
    case B2Q_kMAX: if (need_skip_null) agg_max_skip_val(a, v, null_v); else agg_max(a, v); break;
    case B2Q_kAVG: {
      int64_t* cnt = reinterpret_cast<int64_t*>(slot_ptr(p, out, entry, s + 1));
      if (need_skip_null) { agg_sum_skip_val(a, v, null_v); agg_count_skip_val(cnt, v, null_v); }
      else { agg_sum(a, v); agg_count(cnt); }
      break;
    }
    default: abort();
  }
}

/* ---- buffer init: QueryMemoryInitializer::initRowGroups (QueryMemoryInitializer.cpp:620-700) ---- */
void init_buffer(const Plan& plan, std::vector<int8_t>& buf) {
  const B2QPlan& p = plan.p;
  buf.assign(static_cast<size_t>(p.buffer_size + plan.cd_total), 0); /* + zeroed COUNT(DISTINCT) bitmaps (allocateCountDistinctBuffers) */
  if (p.query_desc_type == B2Q_Estimator) return; /* the estimator buffer is a zeroed bitmap (QueryMemoryInitializer: allocateCountDistinct... / estimator_result_set_) */
  const bool has_key = p.query_desc_type != B2Q_NonGroupedAggregate && !p.keyless_hash;
  for (int64_t e = 0; e < p.entry_count; ++e) {
    if (has_key) {
      if (p.effective_key_width == 4) { int32_t k = kEmptyKey32; memcpy(key_ptr(p, buf.data(), e, 0), &k, 4); }
      else for (int kc = 0; kc < std::max(p.num_group_cols, 1); ++kc) { int64_t k = kEmptyKey64; memcpy(key_ptr(p, buf.data(), e, kc), &k, 8); } /* fill_empty_key / initColumnarGroups */
    }
    for (int s = 0; s < p.num_slots; ++s) {
      const int w = p.slot_padded_width[s];
      if (w == 8) memcpy(slot_ptr(p, buf.data(), e, s), &p.init_vals[s], 8);
      else if (w == 4) { int32_t v = static_cast<int32_t>(p.init_vals[s]); memcpy(slot_ptr(p, buf.data(), e, s), &v, 4); }
    }
  }
}

/* ---- the fragment row loop: multifrag_query_hoisted_literals -> query_group_by_template / query_template
 * (RuntimeFunctions.cpp:2434-2472, QueryTemplateGenerator.cpp:552-815): pos_start = 0, pos_step = 1 on CPU ---- */
int32_t run_rows(const Plan& plan, const B2QExecUnit& u, const B2QTableInfo& tbl, const B2QFragmentInfo& fr, std::vector<int8_t>& buf);

int32_t run_fragment(const Plan& plan, const B2QExecUnit& u, const B2QTableInfo& tbl, const B2QFragmentInfo& fr,
                     std::vector<int8_t>& buf) {
  init_buffer(plan, buf);
  return run_rows(plan, u, tbl, fr, buf);
}

/* the row function over one fragment into an ALREADY initialised buffer: what one iteration of the fragment loop of
 * multifrag_query_hoisted_literals does (RuntimeFunctions.cpp:2434-2472: every fragment of a kernel shares `out`) */
int32_t run_rows(const Plan& plan, const B2QExecUnit& u, const B2QTableInfo& tbl, const B2QFragmentInfo& fr, std::vector<int8_t>& buf) {
  const B2QPlan& p = plan.p;
  const int key_col = p.key_col_id;
  const int key_type = key_col >= 0 ? tbl.col_types[key_col].type : 0;
  const bool key_nullable = key_col >= 0 && !tbl.col_types[key_col].notnull;
  const uint32_t row_size_quad = static_cast<uint32_t>(p.row_size / 8);
  struct JoinScope { /* the inner-row iterator of this thread's row loop */
    explicit JoinScope(int n_outer) { g_join_row.n_outer = n_outer; }
    ~JoinScope() { g_join_row = JoinRowCtx{}; }
  } join_scope(plan.join ? plan.join_inner_vcol - p.join_inner_col : INT32_MAX);
  const int32_t* join_buff = plan.join && plan.join_buff ? plan.join_buff->data() : nullptr;
  const int64_t join_null = plan.join ? inline_int_null_val(tbl.col_types[plan.join_outer_col].type) : 0;
  for (int64_t pos = 0; pos < fr.num_tuples; ++pos) {
    if (plan.join) {
      /* deleted outer rows never reach the join loop (codegenSkipDeletedOuterTableRow precedes it) */
      if (g_filter_deleted && tbl.deleted_column_plus1 > 0 && static_cast<const int8_t*>(fr.col_buffers[tbl.deleted_column_plus1 - 1])[pos] > 0) continue;
      /* hash_join_idx[_nullable] (GroupByRuntime.cpp:283-311): NULL never matches, keys outside [min, max] miss */
      const int64_t key = decode_int_column(tbl, fr, plan.join_outer_col, pos);
      int64_t idx = -1;
      if (!(plan.join_outer_nullable && key == join_null) && key >= p.join_min_key && key <= p.join_max_key) idx = join_buff[key - p.join_min_key];
      if (idx < 0 && !plan.join_left) continue; /* INNER join: no match, no row */
      g_join_row.inner_pos = idx;        /* LEFT join: -1 => the inner columns read NULL */
    }
    if (!row_passes(u, tbl, fr, pos)) continue;
    if (p.query_desc_type == B2Q_Estimator) {
      /* codegenEstimator (GroupByAndAggregate.cpp:1825-1864): the tuple as int64 sub-keys (groupByColumnCodegen without
       * NULL translation: a NULL is its sentinel) -> linear_probabilistic_count (RuntimeFunctions.cpp:2399-2408) */
      int64_t key[B2Q_MAX_GROUP_COLS];
      const int n = static_cast<int>(plan.estimator_cols.size());
      for (int i = 0; i < n; ++i) key[i] = decode_int_column(tbl, fr, plan.estimator_cols[i], pos);
      const uint32_t bitmap_bytes = static_cast<uint32_t>(p.buffer_size);
      const uint32_t bit_pos = murmur3(key, n * 8, 0) % (bitmap_bytes * 8);
      reinterpret_cast<uint32_t*>(buf.data())[bit_pos / 32] |= 1u << (bit_pos % 32);
      continue;
    }
    int64_t entry = 0;
    if (p.query_desc_type != B2Q_NonGroupedAggregate) {
      if (plan.keys.size() > 1) {
        /* perfect_key_hash (codegenPerfectHashFunction, GroupByAndAggregate.cpp:1549-1597) over the NULL-translated
         * keys, then get_matching_group_value_perfect_hash[_keyless] (RuntimeFunctions.cpp:2077-2103) or, columnar,
         * set_matching_group_value_perfect_hash_columnar (:2109-2124) */
        int64_t keyv[B2Q_MAX_GROUP_COLS];
        int64_t hash = 0;
        bool oob = false;
        for (size_t i = 0; i < plan.keys.size(); ++i) {
          const KeyCol& kc = plan.keys[i];
          int64_t k = decode_int_column(tbl, fr, kc.col, pos);
          if (kc.has_nulls && !tbl.col_types[kc.col].notnull && k == inline_int_null_val(tbl.col_types[kc.col].type)) k = kc.max + (kc.bucket ? kc.bucket : 1);
          keyv[i] = k;
          int64_t d = k - kc.min;
          if (kc.bucket) d /= kc.bucket; /* codegenPerfectHashFunction :1583-1586 */
          oob |= d < 0 || d >= kc.card;
          hash += d * kc.mult;
        }
        if (oob) return B2Q_ERR_KEY_OUT_OF_RANGE;
        entry = hash;
        if (!p.keyless_hash) {
          int64_t first;
          memcpy(&first, key_ptr(p, buf.data(), entry, 0), 8);
          if (first == kEmptyKey64) for (size_t i = 0; i < plan.keys.size(); ++i) memcpy(key_ptr(p, buf.data(), entry, static_cast<int>(i)), &keyv[i], 8);
        }
      } else {
        if (is_fp(key_type)) fail(B2Q_ERR_UNSUPPORTED, "floating-point GROUP BY key");
        int64_t key = decode_int_column(tbl, fr, key_col, pos);
        if (p.query_desc_type == B2Q_GroupByPerfectHash) {
          /* NULL key -> max+1 bucket (GroupByAndAggregate.cpp:1337-1350, GroupByRuntime.cpp:414-425) */
          if (p.has_nulls && key_nullable && key == inline_int_null_val(key_type)) key = p.max_val + (p.bucket ? p.bucket : 1);
          /* get_group_value_fast[_keyless] (GroupByRuntime.cpp:194-209, RuntimeFunctions.cpp:2126-2133);
           * columnar: get_columnar_group_bin_offset (GroupByRuntime.cpp:228-241) */
          int64_t key_diff = key - p.min_val;
          if (p.bucket) key_diff /= p.bucket;
          if (key_diff < 0 || key_diff >= p.entry_count) return B2Q_ERR_KEY_OUT_OF_RANGE; /* stale stats: reference would corrupt memory */
          entry = key_diff;
          if (!p.keyless_hash) {
            int64_t cur;
            memcpy(&cur, key_ptr(p, buf.data(), entry, 0), 8);
            if (cur == kEmptyKey64) memcpy(key_ptr(p, buf.data(), entry, 0), &key, 8);
          }
        } else if (p.output_columnar) {
          /* get_group_value_columnar (GroupByRuntime.cpp:136-157): same hash and probe order over 8-byte keys, the
           * key lives in the key column at the slot index */
          entry = get_group_value_columnar_slot(reinterpret_cast<int64_t*>(buf.data()), static_cast<uint32_t>(p.entry_count), key);
          if (entry < 0) return -static_cast<int32_t>(std::min<int64_t>(pos + 1, INT32_MAX));
        } else {
          int64_t key_store = key;
          int64_t* slots;
          if (p.effective_key_width == 4) {
            int32_t k32 = static_cast<int32_t>(key);
            int64_t keybuf = 0;
            memcpy(&keybuf, &k32, 4);
            slots = get_group_value(reinterpret_cast<int64_t*>(buf.data()), static_cast<uint32_t>(p.entry_count), &keybuf, 1, 4, row_size_quad);
          } else {
            slots = get_group_value(reinterpret_cast<int64_t*>(buf.data()), static_cast<uint32_t>(p.entry_count), &key_store, 1, 8, row_size_quad);
          }
          if (!slots) return -static_cast<int32_t>(std::min<int64_t>(pos + 1, INT32_MAX)); /* out of slots: -pos (GroupByAndAggregate.cpp:1149-1154) */
          entry = (reinterpret_cast<int8_t*>(slots) - buf.data()) / p.row_size;
        }
      }
    }
    for (const auto& t : plan.targets) update_target(plan, t, buf.data(), entry, tbl, fr, pos);
  }
  return 0;
}

/* ---- is the entry empty?  ResultSetStorage::isEmptyEntry (ResultSetIteration.cpp:2457-2492) ---- */
bool is_empty_entry(const B2QPlan& p, const int8_t* buf, int64_t entry) {
  if (p.query_desc_type == B2Q_NonGroupedAggregate) return false;
  if (p.keyless_hash) { /* also isEmptyEntryColumnar (:2498-2526) */
    const int s = p.idx_target_as_key;
    const int w = p.slot_padded_width[s];
    int64_t v;
    if (w == 4) { int32_t x; memcpy(&x, slot_ptr(p, buf, entry, s), 4); v = x; } else memcpy(&v, slot_ptr(p, buf, entry, s), 8);
    return v == p.init_vals[s];
  }
  if (!p.output_columnar && p.effective_key_width == 4) { int32_t k; memcpy(&k, key_ptr(p, buf, entry, 0), 4); return k == kEmptyKey32; }
  int64_t k; /* columnar: first key column, stored as int64 (the plan refuses narrower first key columns) */
  memcpy(&k, key_ptr(p, buf, entry, 0), 8);
  return k == kEmptyKey64;
}

/* ---- ResultSetStorage::reduceOneSlot (ResultSetReduction.cpp:1496-1566) with the AGGREGATE_ONE_* macros
 * (:1290-1437): COUNT merges as SUM, AVG merges (sum, count) separately, nullable values use *_skip_val with the
 * slot's init value as the skip value. ---- */
void reduce_one_row(const Plan& plan, int8_t* this_buf, int64_t this_e, const int8_t* that_buf, int64_t that_e,
                    const B2QPlan* that_layout = nullptr) {
  const B2QPlan& p = plan.p;
  const B2QPlan& q = that_layout ? *that_layout : p; /* `that` may have another entry count (ResultSetManager::reduce grows the baseline destination) */
  for (const auto& t : plan.targets) {
    const int s = t.first_slot;
    const int w = p.slot_padded_width[s];
    if (w == 0) continue;
    int8_t* tp = slot_ptr(p, this_buf, this_e, s);
    const int8_t* op = slot_ptr(q, that_buf, that_e, s);
    const int64_t init_val = p.init_vals[s];
    if (w == 4) {
      int32_t a, b;
      memcpy(&a, tp, 4); memcpy(&b, op, 4);
      if (!t.is_agg) { if (b != static_cast<int32_t>(init_val)) a = b; }
      else a = static_cast<int32_t>(static_cast<uint32_t>(a) + static_cast<uint32_t>(b)); /* agg_sum_int32 */
      memcpy(tp, &a, 4);
      continue;
    }
    int64_t* a = reinterpret_cast<int64_t*>(tp);
    int64_t b;
    memcpy(&b, op, 8);
    if (!t.is_agg) { if (b != init_val) *a = b; continue; } /* projection: :1585-1640 case 8 */
    if (t.is_distinct) { /* count_distinct_set_union (CountDistinct.h:89-140): OR of the two bitmaps */
      const int64_t bytes = align_to_int64((t.cd_bits + 7) / 8);
      int8_t* x = this_buf + t.cd_tail + this_e * bytes;
      const int8_t* y = that_buf + t.cd_tail + that_e * bytes;
      for (int64_t k = 0; k < bytes; ++k) x[k] |= y[k];
      continue;
    }
    if (t.agg_arg_type.type == B2Q_kFLOAT && t.agg_kind != B2Q_kCOUNT) {
      /* float_argument_input in reduceOneSlot (ResultSetReduction.cpp:1514, AGGREGATE_ONE_NULLABLE_VALUE on 4 bytes) */
      int32_t* a32 = reinterpret_cast<int32_t*>(tp);
      int32_t b32;
      memcpy(&b32, op, 4);
      float bv, cur;
      memcpy(&bv, &b32, 4);
      memcpy(&cur, a32, 4);
      const int kind = t.agg_kind == B2Q_kAVG ? B2Q_kSUM : t.agg_kind;
      if (t.agg_kind == B2Q_kAVG) {
        int64_t bc;
        memcpy(&bc, slot_ptr(q, that_buf, that_e, s + 1), 8);
        agg_sum(reinterpret_cast<int64_t*>(slot_ptr(p, this_buf, this_e, s + 1)), bc);
      }
      const int32_t skip32 = static_cast<int32_t>(init_val);
      if (t.skip_null_val && b32 == skip32) continue;       /* `that` holds no value */
      float r;
      if (t.skip_null_val && *a32 == skip32) r = bv;        /* `this` holds none yet */
      else r = kind == B2Q_kMIN ? std::min(cur, bv) : kind == B2Q_kMAX ? std::max(cur, bv) : cur + bv;
      memcpy(a32, &r, 4);
      continue;
    }
    const bool fp = is_fp(get_compact_type(t).type);
    switch (t.agg_kind) {
      case B2Q_kCOUNT: agg_sum(a, b); break; /* AGGREGATE_ONE_COUNT */
      case B2Q_kAVG: {
        int64_t* ac = reinterpret_cast<int64_t*>(slot_ptr(p, this_buf, this_e, s + 1));
        int64_t bc;
        memcpy(&bc, slot_ptr(q, that_buf, that_e, s + 1), 8);
        agg_sum(ac, bc);
      } /* fall thru */
      case B2Q_kSUM:
        if (t.skip_null_val) { if (fp) agg_sum_double_skip_val(a, double_of(b), double_of(init_val)); else agg_sum_skip_val(a, b, init_val); }
        else { if (fp) agg_sum_double(a, double_of(b)); else agg_sum(a, b); }
        break;
      case B2Q_kMIN:
        if (t.skip_null_val) { if (fp) agg_min_double_skip_val(a, double_of(b), double_of(init_val)); else agg_min_skip_val(a, b, init_val); }
        else { if (fp) agg_min_double(a, double_of(b)); else agg_min(a, b); }
        break;
      case B2Q_kMAX:
        if (t.skip_null_val) { if (fp) agg_max_double_skip_val(a, double_of(b), double_of(init_val)); else agg_max_skip_val(a, b, init_val); }
        else { if (fp) agg_max_double(a, double_of(b)); else agg_max(a, b); }
        break;
      default: abort();
    }
  }
}

/* ResultSetStorage::reduce (ResultSetReduction.cpp:203-396): perfect hash => entry-wise
 * (reduceOneEntryNoCollisions :398-450: skip empty `that` entries, copy key); baseline => re-probe every
 * non-empty `that` entry into `this` (:698-828). */
int32_t reduce_buffers(const Plan& plan, std::vector<int8_t>& this_buf, const std::vector<int8_t>& that_buf, const B2QPlan* that_layout = nullptr) {
  const B2QPlan& p = plan.p;
  const B2QPlan& q = that_layout ? *that_layout : p;
  if (p.query_desc_type == B2Q_Estimator) { /* reduce_estimator_results (CardinalityEstimator.cpp:142-161) */
    for (size_t i = 0; i < this_buf.size(); ++i) this_buf[i] |= that_buf[i];
    return 0;
  }
  if (p.query_desc_type == B2Q_NonGroupedAggregate) {
    reduce_one_row(plan, this_buf.data(), 0, that_buf.data(), 0);
    return 0;
  }
  for (int64_t e = 0; e < q.entry_count; ++e) {
    if (is_empty_entry(q, that_buf.data(), e)) continue;
    if (p.query_desc_type == B2Q_GroupByPerfectHash) {
      if (!p.keyless_hash) /* key copy (copyKeyColWise :452-476 when columnar) */
        for (int c = 0; c < std::max(p.num_group_cols, 1); ++c)
          memcpy(key_ptr(p, this_buf.data(), e, c), key_ptr(q, that_buf.data(), e, c), p.output_columnar ? 8 : p.effective_key_width);
      reduce_one_row(plan, this_buf.data(), e, that_buf.data(), e);
    } else {
      int64_t keybuf = 0;
      memcpy(&keybuf, key_ptr(q, that_buf.data(), e, 0), p.effective_key_width);
      int64_t this_e;
      if (p.output_columnar) {
        this_e = get_group_value_columnar_slot(reinterpret_cast<int64_t*>(this_buf.data()), static_cast<uint32_t>(p.entry_count), keybuf);
        if (this_e < 0) return B2Q_ERR_OUT_OF_SLOTS;
      } else {
        int64_t* slots = get_group_value(reinterpret_cast<int64_t*>(this_buf.data()), static_cast<uint32_t>(p.entry_count), &keybuf, 1,
                                         static_cast<uint32_t>(p.effective_key_width), static_cast<uint32_t>(p.row_size / 8));
        if (!slots) return B2Q_ERR_OUT_OF_SLOTS;
        this_e = (reinterpret_cast<int8_t*>(slots) - this_buf.data()) / p.row_size;
      }
      reduce_one_row(plan, this_buf.data(), this_e, that_buf.data(), e, &q);
    }
  }
  return 0;
}

}  // namespace

/* ===================================================================================================
 * C API (ctypes-friendly)
 * ================================================================================================= */
struct OracleResult {
  Plan plan;
  std::vector<int8_t> buf;
  int64_t cursor{0};
  double exec_seconds{0};
  /* ResultSet::permutation_, drop_first_, keep_first_, fetched_so_far_ (ResultSet.h) */
  std::vector<uint32_t> perm;
  bool sorted{false};
  size_t drop_first{0}, keep_first{0}, fetched{0};
  bool empty_result{false}; /* LIMIT 0: RelSort::isEmptyResult() -> just_validate -> an empty result set (RelAlgDag.h:2557, RelAlgExecutor.cpp:1277,3559) */
};

namespace {

/* ResultSet::ResultSetComparator::operator() (ResultSet.cpp:1310-1478) for the numeric subset: per order entry
 * read the target like getColumnInternal (slot at its padded width; AVG as the (sum, count) pair; a baseline key
 * target from the key), NULLs by ResultSet::isNull (ResultSetIteration.cpp:2601-2618), then int / double / pair compare. */
struct ResultSetComparator {
  const OracleResult* r;
  std::vector<B2QOrderEntry> order_entries;
  struct Val { int64_t i1, i2; bool pair; };
  Val get(int64_t entry, const Target& t) const {
    const B2QPlan& p = r->plan.p;
    const int s = t.first_slot;
    int w = p.slot_padded_width[s];
    const int8_t* ptr = slot_ptr(p, r->buf.data(), entry, s);
    if (w == 0) { ptr = key_ptr(p, r->buf.data(), entry, 0); w = p.effective_key_width; }
    Val v{0, 0, false};
    if (w == 4) { int32_t x; memcpy(&x, ptr, 4); v.i1 = x; } else memcpy(&v.i1, ptr, 8);
    if (t.is_agg && t.agg_kind == B2Q_kAVG) { v.pair = true; memcpy(&v.i2, slot_ptr(p, r->buf.data(), entry, s + 1), 8); }
    return v;
  }
  static bool is_null(const Ti& ti, const Val& v) {
    if (ti.notnull) return false;
    if (v.pair) return !v.i2;
    return v.i1 == (is_fp(ti.type) ? bits_of(kNullDouble) : inline_int_null_val(ti.type)); /* null_val_bit_pattern */
  }
  static double pair_to_double(const Val& v, const Target& t) { /* ResultSetBufferAccessors.h:197-227 */
    if (!v.i2) return kNullDouble;
    const double dividend = is_fp(t.sql_type.type) ? double_of(v.i1) : static_cast<double>(v.i1);
    return is_decimal(t.sql_type.type) && t.sql_type.scale ? dividend / (static_cast<double>(v.i2) * exp_to_scale(t.sql_type.scale)) /* :222-225 */
                                                           : dividend / static_cast<double>(v.i2);
  }
  bool operator()(uint32_t lhs, uint32_t rhs) const {
    for (const B2QOrderEntry& oe : order_entries) {
      const Target& t = r->plan.targets[oe.tle_no - 1];
      const Ti ti = get_compact_type(t);
      const Val l = get(lhs, t), rv = get(rhs, t);
      const bool ln = is_null(ti, l), rn = is_null(ti, rv);
      if (ln && rn) continue;
      if (ln && !rn) return oe.nulls_first;
      if (rn && !ln) return !oe.nulls_first;
      if (!l.pair) {
        if (l.i1 == rv.i1) continue;
        if (is_fp(ti.type)) return (double_of(l.i1) < double_of(rv.i1)) != static_cast<bool>(oe.is_desc);
        return (l.i1 < rv.i1) != static_cast<bool>(oe.is_desc);
      }
      const double a = pair_to_double(l, t), b = pair_to_double(rv, t);
      if (a == b) continue;
      return (a < b) != static_cast<bool>(oe.is_desc);
    }
    return false;
  }
};

/* ResultSet::sort (ResultSet.cpp:781-849): initPermutationBuffer (:870-885) + topPermutation (:1501-1527).
 * The reference's std::partial_sort / std::sort leave ties in unspecified order; std::stable_sort over the
 * ascending permutation pins them (ascending entry index), which is also what the device sort produces. */
void result_sort(OracleResult* r, const B2QOrderEntry* oes, int n, size_t top_n) {
  const B2QPlan& p = r->plan.p;
  r->perm.clear();
  r->cursor = 0; r->fetched = 0;
  for (int64_t e = 0; e < p.entry_count; ++e) if (!is_empty_entry(p, r->buf.data(), e)) r->perm.push_back(static_cast<uint32_t>(e));
  ResultSetComparator cmp{r, std::vector<B2QOrderEntry>(oes, oes + n)};
  if (top_n == 0) top_n = r->perm.size();
  std::stable_sort(r->perm.begin(), r->perm.end(), cmp);
  if (top_n < r->perm.size()) r->perm.resize(top_n);
  r->sorted = true;
}

}  // namespace

static thread_local std::string g_last_error;

/* COUNT(DISTINCT): the reference leaves a pointer to the group's bitmap in the slot and counts its bits when the value is read
 * (count_distinct_set_size, CountDistinct.h:54-70; makeTargetValue, ResultSetIteration.cpp:2178-2181).  The boundary of the
 * product carries no pointers, so its result buffer holds the set size itself; the oracle's final buffer is put in the same
 * form here, after every reduce step has run on the bitmaps. */
static void finalize_count_distinct(OracleResult* res) {
  const B2QPlan& p = res->plan.p;
  if (!res->plan.cd_total) return;
  for (const auto& t : res->plan.targets) {
    if (!t.is_distinct) continue;
    const int64_t bytes = align_to_int64((t.cd_bits + 7) / 8);
    for (int64_t e = 0; e < std::max<int64_t>(p.entry_count, 1); ++e) {
      if (is_empty_entry(p, res->buf.data(), e)) continue;
      const uint8_t* bm = reinterpret_cast<const uint8_t*>(res->buf.data()) + t.cd_tail + e * bytes;
      int64_t n = 0;
      for (int64_t k = 0; k < bytes; ++k) n += __builtin_popcount(bm[k]);
      memcpy(slot_ptr(p, res->buf.data(), e, t.first_slot), &n, 8);
    }
  }
  res->buf.resize(static_cast<size_t>(p.buffer_size));
}

/* Worker placement for the timed CPU arm (bench.py): with pinning on, worker t of oracle_execute and of
 * oracle_gen_fragments runs on the t-th CPU of the process's affinity mask, so that the thread that scans fragment f is the
 * one that first touched its pages (NUMA-local memory).  Off by default: the tests do not care. */
static std::atomic<int> g_pin_threads{0};
ORACLE_EXPORT void oracle_set_thread_pinning(int32_t on) { g_pin_threads = on; }
static void pin_worker(int t) {
  if (!g_pin_threads) return;
  cpu_set_t mask;
  if (sched_getaffinity(0, sizeof(mask), &mask) != 0) return;
  const int n = CPU_COUNT(&mask);
  if (n <= 0) return;
  int want = t % n, seen = 0;
  for (int c = 0; c < CPU_SETSIZE; ++c) {
    if (!CPU_ISSET(c, &mask)) continue;
    if (seen++ == want) {
      cpu_set_t one;
      CPU_ZERO(&one);
      CPU_SET(c, &one);
      pthread_setaffinity_np(pthread_self(), sizeof(one), &one);
      return;
    }
  }
}
ORACLE_EXPORT void oracle_gen_column_strided(void* dst, int32_t sql_type, uint64_t seed, uint32_t col_tag, int64_t row0,
                                             int64_t count, int64_t lo, int64_t span, int64_t stride, int32_t num_threads);

ORACLE_EXPORT const char* oracle_last_error() { return g_last_error.c_str(); }
ORACLE_EXPORT void oracle_set_filter_on_deleted_column(int32_t on) { g_filter_deleted = on != 0; }

ORACLE_EXPORT uint32_t oracle_murmur3(const void* key, int len, uint32_t seed) { return murmur3(key, len, seed); }

/* get_group_value over a caller-provided row-wise buffer; returns the int64 offset of the slot pointer or -1 */
ORACLE_EXPORT int64_t oracle_get_group_value(int64_t* groups_buffer, uint32_t entry_count, const int64_t* key,
                                             uint32_t key_count, uint32_t key_width, uint32_t row_size_quad) {
  int64_t* r = get_group_value(groups_buffer, entry_count, key, key_count, key_width, row_size_quad);
  return r ? (r - groups_buffer) : -1;
}

ORACLE_EXPORT int32_t oracle_plan(const B2QExecUnit* u, const B2QTableInfo* tbl, const B2QExecutionOptions* eo,
                                  size_t entry_guess, int32_t has_cardinality_estimation, B2QPlan* out) {
  try {
    Plan plan = make_plan(*u, *tbl, *eo, entry_guess, has_cardinality_estimation != 0);
    *out = plan.p;
    return 0;
  } catch (const OracleError& e) {
    g_last_error = e.msg;
    return e.code;
  }
}

/* The CPU executor: one buffer per fragment (KernelPerFragment, Execute.cpp:3102-3153), `num_threads` worker
 * threads each taking fragments round-robin (the reference runs one thread per fragment, capped at
 * cpu_threads(), Shared/thread_count.h:25-28), then a host reduce in fragment order
 * (Execute.cpp:2833-2864 -> reduceMultiDeviceResultSets :1772). */
ORACLE_EXPORT int32_t oracle_execute(const B2QExecUnit* u, const B2QTableInfo* tbl, const B2QExecutionOptions* eo,
                                     size_t entry_guess, int32_t has_cardinality_estimation, int32_t num_threads,
                                     OracleResult** out) {
  try {
    std::unique_ptr<OracleResult> holder(new OracleResult());
    OracleResult* res = holder.get();
    JoinedInput ji;
    res->plan = make_plan(*u, *tbl, *eo, entry_guess, has_cardinality_estimation != 0, &ji);
    if (tbl->memory_level != B2Q_CPU_LEVEL) fail(B2Q_ERR_INVALID_ARGUMENT, "oracle needs host column buffers");
    if (ji.active) { /* from here on the unit / table are the combined ones */
      build_join_table(res->plan, ji, *u->inner_table);
      u = &ji.u;
      tbl = &ji.t;
    }
    const int nf = tbl->num_fragments;
    std::vector<std::vector<int8_t>> bufs(std::max(nf, 1));
    std::vector<int32_t> errs(std::max(nf, 1), 0);
    std::vector<std::string> msgs(std::max(nf, 1));
    if (nf == 0) init_buffer(res->plan, bufs[0]);
    const int nt = std::max(1, std::min(num_threads, nf));
    auto work = [&](int tid) {
      pin_worker(tid);
      for (int f = tid; f < nf; f += nt) {
        try {
          errs[f] = run_fragment(res->plan, *u, *tbl, tbl->fragments[f], bufs[f]);
        } catch (const OracleError& e) {
          errs[f] = e.code;
          msgs[f] = e.msg;
        }
      }
    };
    if (nt == 1 && !g_pin_threads) work(0);
    else {
      std::vector<std::thread> ths;
      for (int t = 0; t < nt; ++t) ths.emplace_back(work, t);
      for (auto& t : ths) t.join();
    }
    for (int f = 0; f < nf; ++f) if (errs[f]) { g_last_error = msgs[f]; return errs[f]; }
    for (int f = 1; f < nf; ++f) {
      int32_t rc = reduce_buffers(res->plan, bufs[0], bufs[f]);
      if (rc) return rc;
      std::vector<int8_t>().swap(bufs[f]);
    }
    res->buf = std::move(bufs[0]);
    finalize_count_distinct(res);
    /* the tail of RelAlgExecutor::executeSort (RelAlgExecutor.cpp:3586-3610) when the unit carries sort_info */
    if (u->num_order_entries) result_sort(res, u->order_entries, u->num_order_entries, static_cast<size_t>((u->has_limit ? u->limit : 0) + u->offset));
    if (u->has_limit || u->offset) {
      res->drop_first = static_cast<size_t>(u->offset);
      if (u->has_limit) res->keep_first = static_cast<size_t>(u->limit);
    }
    if (u->has_limit && u->limit == 0) { res->empty_result = true; res->perm.clear(); res->sorted = true; }
    *out = holder.release();
    return 0;
  } catch (const OracleError& e) {
    g_last_error = e.msg;
    return e.code;
  }
}

/* ---- full-size check of the benchmark configurations -----------------------------------------------------------
 * The same executor over a table that is never materialised: column c of global row r is the counter-based generator's
 * value (oracle_gen.h), produced slab by slab into thread-local buffers right before the row function reads it.  Work is
 * cut into slabs of 64 Ki rows; each worker thread owns ONE output buffer for all its slabs — the multi-fragment kernel
 * of the reference (multifrag_query_hoisted_literals, RuntimeFunctions.cpp:2434-2472: one `out` per kernel, the row loop
 * run fragment after fragment; ExecutionOptions::allow_multifrag) — and the per-thread buffers are reduced with
 * ResultSetStorage::reduce: perfect hash entry range by entry range in thread order (the order a sequential reduce
 * visits each entry), baseline hash pairwise (the re-probe reduce is associative on the set of rows).
 * Fragments of `tbl` need no column buffers (num_tuples, fragment_id and chunk stats only); global row of tuple i of
 * fragment f = fragment_id * rows_per_fragment_id + i. */
struct OracleGenCol { int32_t sql_type; uint32_t col_tag; int64_t lo, span, stride; };

ORACLE_EXPORT int32_t oracle_execute_generated(const B2QExecUnit* u, const B2QTableInfo* tbl, const B2QExecutionOptions* eo,
                                               size_t entry_guess, int32_t has_cardinality_estimation, int32_t num_threads,
                                               uint64_t seed, const OracleGenCol* gen, int64_t rows_per_fragment_id,
                                               OracleResult** out) {
  try {
    std::unique_ptr<OracleResult> holder(new OracleResult());
    OracleResult* res = holder.get();
    res->plan = make_plan(*u, *tbl, *eo, entry_guess, has_cardinality_estimation != 0, nullptr);
    if (res->plan.join) fail(B2Q_ERR_UNSUPPORTED, "generated tables have no join level");
    const int nc = tbl->num_cols;
    const int64_t slab = int64_t(1) << 16;
    struct Item { int frag; int64_t row0, rows; };
    std::vector<Item> items;
    for (int f = 0; f < tbl->num_fragments; ++f)
      for (int64_t r = 0; r < tbl->fragments[f].num_tuples; r += slab) items.push_back({f, r, std::min(slab, tbl->fragments[f].num_tuples - r)});
    const int nt = std::max<int>(1, std::min<int64_t>(num_threads, std::max<size_t>(items.size(), 1)));
    std::vector<std::vector<int8_t>> bufs(nt);
    std::vector<int32_t> errs(nt, 0);
    std::vector<std::string> msgs(nt);
    std::atomic<size_t> next{0};
    auto width_of = [](int t) { return t == B2Q_kTINYINT ? 1 : t == B2Q_kSMALLINT ? 2 : t == B2Q_kINT ? 4 : 8; };
    auto work = [&](int tid) {
      try {
        init_buffer(res->plan, bufs[tid]);
        std::vector<std::vector<int8_t>> cols(nc);
        std::vector<const void*> ptrs(nc, nullptr);
        for (int c = 0; c < nc; ++c) { cols[c].resize(static_cast<size_t>(slab) * width_of(gen[c].sql_type)); ptrs[c] = cols[c].data(); }
        for (;;) {
          const size_t i = next.fetch_add(1);
          if (i >= items.size() || errs[tid]) break;
          const Item& it = items[i];
          const B2QFragmentInfo& src = tbl->fragments[it.frag];
          const int64_t g0 = static_cast<int64_t>(src.fragment_id) * rows_per_fragment_id + it.row0;
          for (int c = 0; c < nc; ++c) oracle_gen_column_strided(cols[c].data(), gen[c].sql_type, seed, gen[c].col_tag, g0, it.rows, gen[c].lo, gen[c].span, gen[c].stride, 1);
          B2QFragmentInfo fr = src;
          fr.num_tuples = it.rows;
          fr.col_buffers = ptrs.data();
          errs[tid] = run_rows(res->plan, *u, *tbl, fr, bufs[tid]);
        }
      } catch (const OracleError& e) {
        errs[tid] = e.code;
        msgs[tid] = e.msg;
      }
    };
    {
      std::vector<std::thread> ths;
      for (int t = 0; t < nt; ++t) ths.emplace_back(work, t);
      for (auto& t : ths) t.join();
    }
    for (int t = 0; t < nt; ++t) if (errs[t]) { g_last_error = msgs[t]; return errs[t]; }
    const B2QPlan& p = res->plan.p;
    if (p.query_desc_type == B2Q_GroupByPerfectHash && nt > 1) {
      /* reduceOneEntryNoCollisions is entry-local: thread j folds its entry range of buffers 1..nt-1 into buffer 0, in order */
      auto fold = [&](int j) {
        const int64_t e0 = p.entry_count * j / nt, e1 = p.entry_count * (j + 1) / nt;
        for (int t = 1; t < nt; ++t)
          for (int64_t e = e0; e < e1; ++e) {
            if (is_empty_entry(p, bufs[t].data(), e)) continue;
            if (!p.keyless_hash)
              for (int c = 0; c < std::max(p.num_group_cols, 1); ++c)
                memcpy(key_ptr(p, bufs[0].data(), e, c), key_ptr(p, bufs[t].data(), e, c), p.output_columnar ? 8 : p.effective_key_width);
            reduce_one_row(res->plan, bufs[0].data(), e, bufs[t].data(), e);
          }
      };
      std::vector<std::thread> ths;
      for (int j = 0; j < nt; ++j) ths.emplace_back(fold, j);
      for (auto& t : ths) t.join();
    } else {
      std::atomic<int32_t> rerr{0};
      for (int step = 1; step < nt; step *= 2) { /* pairwise: (0,1)(2,3).. then (0,2)(4,6).. */
        std::vector<std::thread> ths;
        for (int a = 0; a + step < nt; a += 2 * step)
          ths.emplace_back([&, a, step]() {
            const int32_t rc = reduce_buffers(res->plan, bufs[a], bufs[a + step]);
            if (rc) rerr = rc;
            std::vector<int8_t>().swap(bufs[a + step]);
          });
        for (auto& t : ths) t.join();
        if (rerr) return rerr.load();
      }
    }
    res->buf = std::move(bufs[0]);
    finalize_count_distinct(res);
    *out = holder.release();
    return 0;
  } catch (const OracleError& e) {
    g_last_error = e.msg;
    return e.code;
  }
}

/* A result set over a storage buffer the caller filled — ResultSet(targets, device_type, query_mem_desc, ...) +
 * allocateStorage() as Tests/ResultSetTest.cpp:879-894 / :1026-1046 use it: the descriptor is the planned query's. */
ORACLE_EXPORT int32_t oracle_result_from_storage(const B2QExecUnit* u, const B2QTableInfo* tbl, const B2QExecutionOptions* eo,
                                                 size_t entry_guess, int32_t has_cardinality_estimation, const int8_t* storage,
                                                 size_t size_bytes, OracleResult** out) {
  try {
    std::unique_ptr<OracleResult> res(new OracleResult());
    JoinedInput ji;
    res->plan = make_plan(*u, *tbl, *eo, entry_guess, has_cardinality_estimation != 0, &ji);
    if (res->plan.cd_total) fail(B2Q_ERR_UNSUPPORTED, "storage of a COUNT(DISTINCT) query carries bitmap pointers");
    if (size_bytes != static_cast<size_t>(res->plan.p.buffer_size)) fail(B2Q_ERR_INVALID_ARGUMENT, "storage size differs from the descriptor's buffer size");
    res->buf.assign(storage, storage + size_bytes);
    *out = res.release();
    return 0;
  } catch (const OracleError& e) {
    g_last_error = e.msg;
    return e.code;
  }
}

/* ResultSetManager::reduce (ResultSetReduction.cpp:1055-1140): the first set's storage is the destination.  For baseline
 * hash a storage with the SUM of the sets' entry counts is initialised first and the first set's entries are moved into it
 * (moveEntriesToBuffer / moveOneEntryToBuffer :941-1050: every non-empty entry is re-probed into the bigger table and its
 * slots copied); then every other set is reduced into the destination with ResultSetStorage::reduce. */
ORACLE_EXPORT int32_t oracle_result_sets_reduce(OracleResult* const* sets, int32_t n, OracleResult** out) {
  try {
    if (!sets || n < 1 || !out) fail(B2Q_ERR_INVALID_ARGUMENT, "result sets");
    std::unique_ptr<OracleResult> res(new OracleResult());
    res->plan = sets[0]->plan;
    B2QPlan& p = res->plan.p;
    if (p.query_desc_type == B2Q_GroupByBaselineHash) {
      if (res->plan.cd_total) fail(B2Q_ERR_UNSUPPORTED, "baseline growth with COUNT(DISTINCT) bitmaps");
      int64_t total = 0;
      for (int i = 0; i < n; ++i) total += sets[i]->plan.p.entry_count;
      const B2QPlan first = p;
      p.entry_count = total;
      if (p.output_columnar) { /* the offsets of the columnar layout follow the entry count (getColOffInBytes :918-955) */
        int64_t off = align_to_int64(8 * p.entry_count);
        for (int s = 0; s < p.num_slots; ++s) { p.slot_offset[s] = off; off += align_to_int64(static_cast<int64_t>(p.slot_padded_width[s]) * p.entry_count); }
        p.buffer_size = off;
      } else p.buffer_size = p.row_size * p.entry_count;
      init_buffer(res->plan, res->buf);
      for (int64_t e = 0; e < first.entry_count; ++e) { /* moveOneEntryToBuffer: claim the key's slot in the new table, copy the value slots */
        if (is_empty_entry(first, sets[0]->buf.data(), e)) continue;
        int64_t key = 0;
        memcpy(&key, key_ptr(first, sets[0]->buf.data(), e, 0), first.effective_key_width);
        int64_t dst;
        if (p.output_columnar) dst = get_group_value_columnar_slot(reinterpret_cast<int64_t*>(res->buf.data()), static_cast<uint32_t>(p.entry_count), key);
        else {
          int64_t* slots = get_group_value(reinterpret_cast<int64_t*>(res->buf.data()), static_cast<uint32_t>(p.entry_count), &key, 1,
                                           static_cast<uint32_t>(p.effective_key_width), static_cast<uint32_t>(p.row_size / 8));
          dst = slots ? (reinterpret_cast<int8_t*>(slots) - res->buf.data()) / p.row_size : -1;
        }
        if (dst < 0) fail(B2Q_ERR_OUT_OF_SLOTS, "moveEntriesToBuffer: no slot");
        for (int s = 0; s < p.num_slots; ++s)
          if (p.slot_padded_width[s]) memcpy(slot_ptr(p, res->buf.data(), dst, s), slot_ptr(first, sets[0]->buf.data(), e, s), p.slot_padded_width[s]);
      }
    } else {
      res->buf = sets[0]->buf;
    }
    for (int i = 1; i < n; ++i) {
      const int32_t rc = reduce_buffers(res->plan, res->buf, sets[i]->buf, &sets[i]->plan.p);
      if (rc) fail(rc, "ResultSetStorage::reduce");
    }
    *out = res.release();
    return 0;
  } catch (const OracleError& e) {
    g_last_error = e.msg;
    return e.code;
  }
}

ORACLE_EXPORT const B2QPlan* oracle_result_plan(const OracleResult* r) { return &r->plan.p; }
ORACLE_EXPORT const int8_t* oracle_result_buffer(const OracleResult* r, size_t* size) {
  if (size) *size = r->buf.size();
  return r->buf.data();
}
ORACLE_EXPORT size_t oracle_result_entry_count(const OracleResult* r) { /* ResultSet::entryCount() */
  return r->sorted ? r->perm.size() : static_cast<size_t>(r->plan.p.entry_count);
}
ORACLE_EXPORT int32_t oracle_result_sort(OracleResult* r, const B2QOrderEntry* oes, int32_t n, size_t top_n) {
  for (int i = 0; i < n; ++i) if (oes[i].tle_no < 1 || oes[i].tle_no > static_cast<int>(r->plan.targets.size())) return B2Q_ERR_INVALID_ARGUMENT;
  result_sort(r, oes, n, top_n);
  return 0;
}
ORACLE_EXPORT void oracle_result_drop_first_n(OracleResult* r, size_t n) { r->drop_first = n; r->cursor = 0; r->fetched = 0; }
ORACLE_EXPORT void oracle_result_keep_first_n(OracleResult* r, size_t n) { r->keep_first = n; r->cursor = 0; r->fetched = 0; }
/* the i-th entry index in iteration order (tests compare the device permutation with this one) */
ORACLE_EXPORT int64_t oracle_result_permutation_at(const OracleResult* r, size_t i) { return r->sorted && i < r->perm.size() ? r->perm[i] : -1; }
ORACLE_EXPORT int32_t oracle_result_is_row_at_empty(const OracleResult* r, size_t e) { return is_empty_entry(r->plan.p, r->buf.data(), static_cast<int64_t>(e)); }
ORACLE_EXPORT size_t oracle_result_row_count(const OracleResult* r) { /* ResultSet::rowCountImpl (ResultSet.cpp:565-600) */
  if (r->plan.p.query_desc_type == B2Q_Estimator) return 0; /* an estimator result set has no storage, only the bitmap */
  if (r->empty_result) return 0;
  size_t n = 0;
  if (r->sorted) n = r->perm.size();
  else for (int64_t e = 0; e < r->plan.p.entry_count; ++e) n += !is_empty_entry(r->plan.p, r->buf.data(), e);
  if (n <= r->drop_first) return 0; /* get_truncated_row_count */
  n -= r->drop_first;
  return r->keep_first ? std::min(n, r->keep_first) : n;
}
ORACLE_EXPORT size_t oracle_result_col_count(const OracleResult* r) { return r->plan.targets.size(); }
/* ResultSet::getNDVEstimator (CardinalityEstimator.cpp:33-52) */
ORACLE_EXPORT size_t oracle_result_ndv_estimator(const OracleResult* r) {
  if (r->plan.p.query_desc_type != B2Q_Estimator) return 0;
  size_t bits_set = 0;
  for (int8_t b : r->buf) bits_set += static_cast<size_t>(__builtin_popcount(static_cast<uint8_t>(b)));
  if (bits_set == 0) return 1;
  const size_t total_bits = r->buf.size() * 8;
  const size_t unset_bits = total_bits - bits_set;
  const double ratio = static_cast<double>(unset_bits) / static_cast<double>(total_bits);
  if (ratio == 0.) return 0;
  return static_cast<size_t>(-static_cast<double>(total_bits) * log(ratio));
}
ORACLE_EXPORT void oracle_result_move_to_begin(OracleResult* r) { r->cursor = 0; r->fetched = 0; }
ORACLE_EXPORT void oracle_result_free(OracleResult* r) { delete r; }

/* ResultSet::getColType: AVG targets read out as DOUBLE (ResultSet.cpp getColType) */
ORACLE_EXPORT B2QTypeInfo oracle_result_col_type(const OracleResult* r, size_t col) {
  const Target& t = r->plan.targets[col];
  if (t.is_agg && t.agg_kind == B2Q_kAVG) return B2QTypeInfo{B2Q_kDOUBLE, 0, 0};
  return B2QTypeInfo{t.sql_type.type, t.sql_type.notnull, t.sql_type.scale};
}

/* ResultSet::getNextRow -> getTargetValueFromBufferRowwise -> makeTargetValue (ResultSetIteration.cpp:2086-2220),
 * AVG via make_avg_target_value (:43-82) + pair_to_double (ResultSetBufferAccessors.h:197-227). */
ORACLE_EXPORT int32_t oracle_result_get_next_row(OracleResult* r, B2QTargetValue* row, int32_t decimal_to_double) {
  const B2QPlan& p = r->plan.p;
  if (p.query_desc_type == B2Q_Estimator || r->empty_result) return 0;
  /* getNextRowImpl + advanceCursorToNextEntry (ResultSetIteration.cpp:320-340, :731-750) */
  const int64_t n_entries = r->sorted ? static_cast<int64_t>(r->perm.size()) : p.entry_count;
  int64_t entry = 0;
  do {
    if (r->keep_first && r->fetched >= r->drop_first + r->keep_first) return 0;
    while (r->cursor < n_entries && is_empty_entry(p, r->buf.data(), r->sorted ? r->perm[r->cursor] : r->cursor)) ++r->cursor;
    if (r->cursor >= n_entries) return 0;
    entry = r->sorted ? r->perm[r->cursor] : r->cursor;
    ++r->cursor;
    ++r->fetched;
  } while (r->drop_first && r->fetched <= r->drop_first);
  for (size_t i = 0; i < r->plan.targets.size(); ++i) {
    Target t = r->plan.targets[i];
    /* ResultSet's targets_: non-grouped MIN/MAX/SUM/AVG are nullable (target_exprs_to_infos, set_notnull false) */
    if (t.is_agg && t.arg_col >= 0 && p.query_desc_type == B2Q_NonGroupedAggregate && t.agg_kind != B2Q_kCOUNT) {
      t.sql_type.notnull = false; t.agg_arg_type.notnull = false;
    }
    const int s = t.first_slot;
    int w = p.slot_padded_width[s];
    const int8_t* ptr = slot_ptr(p, r->buf.data(), entry, s);
    if (w == 0) { /* baseline: key column (getTargetValueFromBufferRowwise :2425-2452 / ...Colwise :2267-2340) */
      ptr = key_ptr(p, r->buf.data(), entry, 0);
      w = p.effective_key_width;
    }
    int64_t ival;
    if (w == 4) { int32_t x; memcpy(&x, ptr, 4); ival = x; } else memcpy(&ival, ptr, 8);
    B2QTargetValue& o = row[i];
    o.is_fp = 0; o.is_null = 0; o.ival = 0; o.dval = 0;
    const Ti chosen = get_compact_type(t);
    if (t.is_agg && t.agg_kind == B2Q_kAVG) {
      int64_t cnt;
      memcpy(&cnt, slot_ptr(p, r->buf.data(), entry, s + 1), 8);
      o.is_fp = 1;
      if (cnt == 0) { o.dval = kNullDouble; o.is_null = 1; }
      else {
        double dividend = is_fp(t.sql_type.type) ? double_of(ival) : static_cast<double>(ival);
        if (t.sql_type.type == B2Q_kFLOAT) { float f; memcpy(&f, ptr, 4); dividend = f; } /* float_argument_input: pair_to_double (ResultSetBufferAccessors.h:205-214) */
        o.dval = is_decimal(t.sql_type.type) && t.sql_type.scale ? dividend / (static_cast<double>(cnt) * exp_to_scale(t.sql_type.scale))
                                                                 : dividend / static_cast<double>(cnt);
        o.is_null = o.dval == kNullDouble;
      }
      continue;
    }
    if (chosen.type == B2Q_kFLOAT) { /* make_target_value: a float out of the slot's low 4 bytes */
      float f;
      memcpy(&f, ptr, 4);
      o.is_fp = 1;
      o.dval = f;
      o.is_null = f == kNullFloat;
      continue;
    }
    if (is_fp(chosen.type)) {
      o.is_fp = 1;
      o.dval = double_of(ival);
      o.is_null = o.dval == kNullDouble;
      continue;
    }
    if (is_decimal(chosen.type)) { /* makeTargetValue :2193-2210: the agg kinds test against the BIGINT sentinel whatever notnull says */
      const bool agg_null = t.is_agg && (t.agg_kind == B2Q_kSUM || t.agg_kind == B2Q_kMIN || t.agg_kind == B2Q_kMAX);
      o.is_null = ival == kNullBigint && (agg_null || !chosen.notnull);
      if (decimal_to_double) { o.is_fp = 1; o.dval = o.is_null ? kNullDouble : static_cast<double>(ival) / exp_to_scale(chosen.scale); }
      else o.ival = ival;
      continue;
    }
    /* :2184-2188: NULL iff the value, resized to the compact type's logical size, equals that type's sentinel;
     * the returned value is then the TARGET type's sentinel */
    int64_t resized;
    switch (type_size(chosen.type)) {
      case 1: resized = static_cast<int8_t>(ival); break;
      case 2: resized = static_cast<int16_t>(ival); break;
      case 4: resized = static_cast<int32_t>(ival); break;
      default: resized = ival;
    }
    if (inline_int_null_val(chosen.type) == resized) { o.ival = inline_int_null_val(t.sql_type.type); o.is_null = 1; }
    else o.ival = ival;
  }
  return 1;
}

/* ---- synthetic columns (bench / tests) ---- */
/* whole fragments, fragment f by worker f % num_threads — the worker that oracle_execute gives the fragment to */
ORACLE_EXPORT void oracle_gen_fragments(void* const* dst /* [nf * nc] */, const OracleGenCol* gen, int32_t nc, const int64_t* rows,
                                        const int64_t* row0, int32_t nf, uint64_t seed, int32_t num_threads);

ORACLE_EXPORT void oracle_gen_column_strided(void* dst, int32_t sql_type, uint64_t seed, uint32_t col_tag, int64_t row0,
                                             int64_t count, int64_t lo, int64_t span, int64_t stride, int32_t num_threads);
ORACLE_EXPORT void oracle_gen_column(void* dst, int32_t sql_type, uint64_t seed, uint32_t col_tag, int64_t row0,
                                     int64_t count, int64_t lo, int64_t span, int32_t num_threads) {
  oracle_gen_column_strided(dst, sql_type, seed, col_tag, row0, count, lo, span, 1, num_threads);
}
ORACLE_EXPORT void oracle_gen_column_strided(void* dst, int32_t sql_type, uint64_t seed, uint32_t col_tag, int64_t row0,
                                             int64_t count, int64_t lo, int64_t span, int64_t stride, int32_t num_threads) {
  auto work = [&](int64_t b, int64_t e) {
    for (int64_t i = b; i < e; ++i) {
      const int64_t row = row0 + i;
      switch (sql_type) {
        case B2Q_kDOUBLE: static_cast<double*>(dst)[i] = oracle_gen_double(seed, col_tag, row); break;
        case B2Q_kBIGINT: static_cast<int64_t*>(dst)[i] = lo + (oracle_gen_int(seed, col_tag, row, 0, span)) * stride; break;
        case B2Q_kINT: static_cast<int32_t*>(dst)[i] = static_cast<int32_t>(oracle_gen_int(seed, col_tag, row, lo, span)); break;
        case B2Q_kSMALLINT: static_cast<int16_t*>(dst)[i] = static_cast<int16_t>(oracle_gen_int(seed, col_tag, row, lo, span)); break;
        case B2Q_kTINYINT: static_cast<int8_t*>(dst)[i] = static_cast<int8_t>(oracle_gen_int(seed, col_tag, row, lo, span)); break;
        default: abort();
      }
    }
  };
  const int nt = std::max(1, num_threads);
  if (nt == 1 || count < (1 << 16)) { work(0, count); return; }
  std::vector<std::thread> ths;
  const int64_t per = (count + nt - 1) / nt;
  for (int t = 0; t < nt; ++t) {
    const int64_t b = t * per, e = std::min(count, b + per);
    if (b < e) ths.emplace_back(work, b, e);
  }
  for (auto& t : ths) t.join();
}

ORACLE_EXPORT void oracle_gen_fragments(void* const* dst, const OracleGenCol* gen, int32_t nc, const int64_t* rows,
                                        const int64_t* row0, int32_t nf, uint64_t seed, int32_t num_threads) {
  const int nt = std::max(1, std::min(num_threads, nf));
  auto work = [&](int tid) {
    pin_worker(tid);
    for (int f = tid; f < nf; f += nt)
      for (int c = 0; c < nc; ++c)
        oracle_gen_column_strided(dst[static_cast<size_t>(f) * nc + c], gen[c].sql_type, seed, gen[c].col_tag, row0[f], rows[f], gen[c].lo, gen[c].span, gen[c].stride, 1);
  };
  std::vector<std::thread> ths;
  for (int t = 0; t < nt; ++t) ths.emplace_back(work, t);
  for (auto& t : ths) t.join();
}
