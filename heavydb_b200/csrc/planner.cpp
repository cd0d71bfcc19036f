/*
 * planner.cpp — host-side planning for the B200 path: what GroupByAndAggregate + QueryMemoryDescriptor decide in
 * the reference, then lowering of quals / targets to the device program the static kernels interpret.
 *
 * Reference behaviour restated (paths relative to the reference tree):
 *   hash type          GroupByAndAggregate::getColRangeInfo        QueryEngine/GroupByAndAggregate.cpp:232-365
 *   key range          getLeafColumnRange / apply_simple_quals     QueryEngine/ExpressionRange.cpp:521-632, :144-200
 *   keyless decision   get_keyless_info                            QueryEngine/GroupByAndAggregate.cpp:489-648
 *   entry count/layout QueryMemoryDescriptor::init, getRowSize     QueryEngine/Descriptors/QueryMemoryDescriptor.cpp:240-444,848-955
 *   slot widths        pick_target_compact_width, ColSlotContext   QueryMemoryDescriptor.cpp:748-842, ColSlotContext.cpp:35-101
 *   init values        init_agg_val_vec / get_agg_initial_val      QueryEngine/OutputBufferInitialization.cpp:26-262
 *   target info        get_target_info_impl, get_compact_type      Shared/TargetInfo.cpp:25-78, Shared/SqlTypesLayout.h:37-63
 *   null skipping      TargetExprCodegen::codegenAggregate         QueryEngine/TargetExprBuilder.cpp:470-583,
 *                      convertNullIfAny                            QueryEngine/GroupByAndAggregate.cpp:1599-1660
 */
#include <algorithm>
#include <cfloat>
#include <climits>
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <limits>
#include <string>
#include <map>
#include <vector>

#include "b2q_internal.h"

namespace b2q {

struct PlanError {
  int32_t code;
  std::string msg;
};

namespace {

[[noreturn]] void reject(int32_t code, const std::string& m) { throw PlanError{code, m}; }

struct SqlType {
  int32_t type = 0;
  bool notnull = false;
  int32_t scale = 0; /* SQLTypeInfo::get_scale() of a DECIMAL / NUMERIC */
  bool is_string() const { return type == B2Q_kTEXT || type == B2Q_kVARCHAR || type == B2Q_kCHAR; } /* dictionary ids */
  bool is_time() const { return type == B2Q_kTIME || type == B2Q_kTIMESTAMP || type == B2Q_kDATE; }
  /* everything the path handles as an integer: dictionary ids are int32 (is_int_and_no_bigger_than(ti, 4) ||
   * dict string, QueryMemoryDescriptor.cpp:803-804), time types int64 (sqltypes.h is_time()) */
  /* DECIMAL / NUMERIC: value x 10^scale as int64; every decision that is not is_fp() treats it like BIGINT, the scale only
   * matters at read-out (makeTargetValue, pair_to_double) */
  bool is_decimal() const { return type == B2Q_kDECIMAL || type == B2Q_kNUMERIC; }
  bool is_int() const { return type == B2Q_kTINYINT || type == B2Q_kSMALLINT || type == B2Q_kINT || type == B2Q_kBIGINT || is_string() || is_time() || is_decimal(); }
  bool is_number() const { return is_int() && !is_string() && !is_time(); }
  bool is_fp() const { return type == B2Q_kDOUBLE || type == B2Q_kFLOAT; }
  bool is_float() const { return type == B2Q_kFLOAT; } /* 4-byte chunks and slots; widened (exactly) to double on every load */
  int size() const { /* logical size */
    switch (type) {
      case B2Q_kTINYINT: return 1;
      case B2Q_kSMALLINT: return 2;
      case B2Q_kINT: case B2Q_kFLOAT: case B2Q_kTEXT: case B2Q_kVARCHAR: case B2Q_kCHAR: return 4;
      case B2Q_kBIGINT: case B2Q_kDOUBLE: case B2Q_kTIME: case B2Q_kTIMESTAMP: case B2Q_kDATE: case B2Q_kDECIMAL: case B2Q_kNUMERIC: return 8;
      default: return -1;
    }
  }
  int64_t int_null() const { /* Shared/InlineNullValues.h:30-36, :100-150 */
    switch (type) {
      case B2Q_kTINYINT: return INT8_MIN;
      case B2Q_kSMALLINT: return INT16_MIN;
      case B2Q_kINT: case B2Q_kTEXT: case B2Q_kVARCHAR: case B2Q_kCHAR: return INT32_MIN;
      default: return INT64_MIN;
    }
  }
};
SqlType from_abi(const B2QTypeInfo& t) { return SqlType{t.type, t.notnull != 0, t.scale}; }
B2QTypeInfo to_abi(const SqlType& t) { return B2QTypeInfo{t.type, t.notnull ? 1 : 0, t.scale}; }

int64_t dbl_bits(double d) { int64_t b; memcpy(&b, &d, 8); return b; }
double bits_dbl(int64_t b) { double d; memcpy(&d, &b, 8); return d; }
int64_t align8(int64_t v) { return (v + 7) & ~int64_t(7); }
constexpr double kNullDouble = DBL_MIN;
constexpr double kNullFloat = FLT_MIN; /* NULL_FLOAT (Shared/InlineNullValues.h), as the double it widens to */
static bool fp_type(int t) { return t == B2Q_kDOUBLE || t == B2Q_kFLOAT; }

struct ColRange {
  bool valid = false, fp = false, has_nulls = false;
  int64_t imin = 0, imax = -1;
  double fmin = 0, fmax = -1;
  int64_t bucket = 0; /* 86400 for DATE columns (getLeafColumnRange, ExpressionRange.cpp:622-624) */
};

struct TargetDesc {
  bool is_agg = false;
  int agg = B2Q_kMIN;
  SqlType sql_type, arg_type; /* arg_type.type == 0: no argument */
  bool skip_null = false;
  bool constrained = false; /* the quals hold a top-level `arg IS NOT NULL` (constrained_not_null, OutputBufferInitialization.cpp:301-324) */
  bool distinct = false;    /* COUNT(DISTINCT arg): CountDistinctDescriptor{Bitmap, cd_min, cd_bucket, cd_bits} */
  int64_t cd_min = 0, cd_bits = 0, cd_bucket = 0;
  int arg_col = -1;
  int first_slot = 0;
  SqlType compact() const { /* get_compact_type */
    if (!is_agg || arg_type.type == 0) return sql_type;
    if (agg == B2Q_kMIN || agg == B2Q_kMAX) return arg_type;
    SqlType t = sql_type;
    t.notnull = arg_type.notnull;
    return t;
  }
};

class Planner {
 public:
  Planner(const B2QExecUnit& u, const B2QTableInfo& t, const B2QExecutionOptions& eo, size_t guess, bool has_card,
          bool filter_deleted)
      : u_(u), t_(t), eo_(eo), guess_(guess), has_card_(has_card), filter_deleted_(filter_deleted) {}

  /* join level of the unit this planner was given in its combined form (make_query) */
  void set_join(int n_outer, int outer_col, int inner_col, const B2QTableInfo& inner, bool left) {
    join_ = true;
    join_left_ = left;
    n_outer_ = n_outer;
    join_outer_col_ = outer_col;
    join_inner_col_ = inner_col;
    inner_ = &inner;
  }

  void run(B2QQuery& q) {
    memset(&q, 0, sizeof(q));
    q.prog.join.fk_col = -1;
    q.plan.join_outer_col = q.plan.join_inner_col = -1;
    validate();
    if (u_.has_estimator) { /* createNdvExecutionUnit: quals (+ join level) and the estimator's tuple, nothing else */
      plan_join(q.plan);
      plan_estimator(q.plan);
      lower(q);
      choose_kernel(q);
      return;
    }
    build_targets();
    for (int i = 0; i < u_.num_order_entries; ++i) { /* the device sort orders 8-byte images; float slots would need their own */
      const TargetDesc& d = targets_[u_.order_entries[i].tle_no - 1];
      if (d.compact().is_float()) reject(B2Q_ERR_UNSUPPORTED, "ORDER BY a FLOAT target is outside this path");
    }
    plan_join(q.plan);
    choose_hash_type(q.plan);
    count_distinct_descriptors(q.plan);
    layout_slots(q.plan);
    init_values(q.plan);
    publish_targets(q.plan);
    lower(q);
    choose_kernel(q);
    q.n_order = u_.num_order_entries;
    for (int i = 0; i < u_.num_order_entries; ++i) q.order[i] = u_.order_entries[i];
    q.has_limit = u_.has_limit ? 1 : 0;
    q.limit = u_.limit;
    q.offset = u_.offset;
    q.total_tuples = 0;
    for (int f = 0; f < t_.num_fragments; ++f) q.total_tuples += t_.fragments[f].num_tuples;
  }

 private:
  const B2QExecUnit& u_;
  const B2QTableInfo& t_;
  const B2QExecutionOptions& eo_;
  size_t guess_;
  bool has_card_;
  bool filter_deleted_;
  std::vector<TargetDesc> targets_;
  bool grouped_ = false;
  struct KeyComp { int col; int64_t min, max, card, mult; bool has_nulls; int64_t bucket = 0; };
  std::vector<KeyComp> keycomps_; /* multi-column perfect hash */
  int key_col_ = -1;
  bool keyless_ = false;
  int keyless_idx_ = -1;
  std::vector<bool> slot_key_ref_;
  bool join_ = false, join_left_ = false;
  int n_outer_ = 0, join_outer_col_ = -1, join_inner_col_ = -1;
  const B2QTableInfo* inner_ = nullptr;

  /* PerfectJoinHashTable::getInstance (JoinHashTable/PerfectJoinHashTable.cpp:168-300): the table spans the inner
   * key's range (getExpressionRange(inner_col)), one int32 slot per value; a range much wider than the row count
   * makes the reference switch to a baseline join table (deploy_baseline_join, :235-246) — outside this path */
  void plan_join(B2QPlan& p) {
    if (!join_) return;
    const SqlType ot = col_type(join_outer_col_), it = col_type(n_outer_ + join_inner_col_);
    if (!ot.is_int() || !it.is_int() || ot.is_string() || it.is_string())
      reject(B2Q_ERR_UNSUPPORTED, "join keys must be integer columns (dictionary translation is outside this path)");
    if (ot.is_decimal() || it.is_decimal()) reject(B2Q_ERR_UNSUPPORTED, "DECIMAL join keys are outside this path");
    if (is_days(join_outer_col_) || is_days(n_outer_ + join_inner_col_)) reject(B2Q_ERR_UNSUPPORTED, "days-encoded DATE join keys are outside this path");
    /* getExpressionRange(inner_col): over the inner table alone (getLeafColumnRange, ExpressionRange.cpp:521-632) */
    ColRange r;
    r.valid = true;
    const int64_t inner_tuples = inner_->num_fragments ? inner_->fragments[0].num_tuples : 0;
    if (inner_tuples > 0) {
      const B2QChunkStats& st = inner_->fragments[0].col_stats[join_inner_col_];
      r.imin = st.int_min; r.imax = st.int_max; r.has_nulls = st.has_nulls != 0;
      if (r.imax < r.imin) { r.imin = 0; r.imax = -1; }
    }
    int64_t entries = 0;
    if (r.imin <= r.imax && (__builtin_sub_overflow(r.imax, r.imin, &entries) || __builtin_add_overflow(entries, int64_t(1), &entries) || entries > INT32_MAX))
      reject(B2Q_ERR_UNSUPPORTED, "too many hash entries for a perfect join table (TooManyHashEntries)");
    const int64_t inner_rows = inner_->num_fragments ? inner_->fragments[0].num_tuples : 0;
    if (inner_rows * 100 < entries) /* g_ratio_num_hash_entry_to_num_tuple_switch_to_baseline, Execute.cpp:104 */
      reject(B2Q_ERR_UNSUPPORTED, "join column range too wide for its row count: the reference switches to a baseline join table");
    p.join_min_key = r.imin;
    p.join_max_key = r.imax;
    p.join_entry_count = entries;
    p.join_outer_col = join_outer_col_;
    p.join_inner_col = join_inner_col_;
  }

  /* QueryDescriptionType::Estimator (QueryMemoryDescriptor::init :270-300): entry_count 1, the output is the
   * estimator's bitmap of Estimator::getBufferSize() bytes (CardinalityEstimator.h:89-116, .cpp:27-29) */
  std::vector<int> estimator_cols_;
  void plan_estimator(B2QPlan& p) {
    if (u_.has_estimator != 1 && u_.has_estimator != 2) reject(B2Q_ERR_INVALID_ARGUMENT, "estimator kind");
    if (u_.num_groupby_exprs || u_.num_target_exprs || u_.num_order_entries || u_.has_limit || u_.offset)
      reject(B2Q_ERR_INVALID_ARGUMENT, "an estimator unit has no groupby_exprs, targets or sort_info");
    if (u_.num_estimator_args <= 0 || u_.num_estimator_args > B2Q_MAX_GROUP_COLS || !u_.estimator_args)
      reject(B2Q_ERR_UNSUPPORTED, "estimator argument count");
    p.query_desc_type = B2Q_Estimator;
    p.entry_count = 1;
    p.key_col_id = -1;
    p.idx_target_as_key = -1;
    p.effective_key_width = 8;
    p.buffer_size = (u_.has_estimator == 2 ? int64_t(256) : int64_t(1)) * 1024 * 1024;
    for (int i = 0; i < u_.num_estimator_args; ++i) {
      const B2QExpr& e = ex(u_.estimator_args[i]);
      if (e.kind != B2Q_EXPR_COLUMN_VAR) reject(B2Q_ERR_UNSUPPORTED, "estimator argument must be a ColumnVar");
      if (!col_type(e.col_id).is_int()) reject(B2Q_ERR_UNSUPPORTED, "estimator over a floating-point key");
      if (is_days(e.col_id)) reject(B2Q_ERR_UNSUPPORTED, "estimator over a days-encoded DATE is outside this path");
      estimator_cols_.push_back(e.col_id);
      p.group_col_ids[i] = e.col_id;
      p.group_col_widths[i] = static_cast<int8_t>(col_type(e.col_id).size());
    }
    p.num_group_cols = u_.num_estimator_args;
  }

  const B2QExpr& ex(int i) const {
    if (i < 0 || i >= u_.num_exprs) reject(B2Q_ERR_INVALID_ARGUMENT, "expression index out of range");
    return u_.exprs[i];
  }
  SqlType col_type(int c) const {
    if (c < 0 || c >= t_.num_cols) reject(B2Q_ERR_INVALID_ARGUMENT, "column id out of range");
    return from_abi(t_.col_types[c]);
  }
  /* physical element width / NULL sentinel of the chunk: narrower than the logical type under ENCODING FIXED
   * (FixedWidthInt decode + codgenAdjustFixedEncNull, ColumnIR.cpp:456-500) */
  int phys_size(int c) const {
    if (t_.col_encoded_sizes && t_.col_encoded_sizes[c] > 0) return t_.col_encoded_sizes[c];
    if (t_.col_encoded_sizes && t_.col_encoded_sizes[c] < 0) return -t_.col_encoded_sizes[c];
    return col_type(c).size();
  }
  /* kENCODING_DATE_IN_DAYS (the default for DATE columns): the chunk holds int32 / int16 days, NULL = the physical
   * minimum, decoded as days * 86400 (FixedWidthSmallDate, ColumnIR.cpp:73-81; DecodersImpl.h:138-146).  The scan never
   * multiplies: constants and key ranges are divided on the host and materialise scales keys and MIN / MAX back. */
  bool is_days(int c) const { return t_.col_encoded_sizes && t_.col_encoded_sizes[c] < 0; }
  static int64_t floor_div(int64_t a, int64_t b) { int64_t q = a / b; return (a % b != 0 && ((a < 0) != (b < 0))) ? q - 1 : q; }
  static int64_t ceil_div(int64_t a, int64_t b) { int64_t q = a / b; return (a % b != 0 && ((a < 0) == (b < 0))) ? q + 1 : q; }
  /* dictionary ids stored on 1 or 2 bytes are UNSIGNED (FixedWidthUnsigned, ColumnIR.cpp:59-67) */
  bool phys_unsigned(int c) const { return col_type(c).is_string() && phys_size(c) < 4; }
  /* width as the kernels take it: bytes, negative for an unsigned (zero-extending) load */
  int phys_width_code(int c) const { return phys_unsigned(c) ? -phys_size(c) : phys_size(c); }
  int64_t phys_int_null(int c) const {
    if (phys_unsigned(c)) return phys_size(c) == 1 ? 255 : 65535; /* inline_fixed_encoding_null_val, InlineNullValues.h:173-182 */
    switch (phys_size(c)) { case 1: return INT8_MIN; case 2: return INT16_MIN; case 4: return INT32_MIN; default: return INT64_MIN; }
  }

  void validate() {
    if (u_.num_join_quals || u_.has_union_all || u_.has_window_function)
      reject(B2Q_ERR_UNSUPPORTED, "join_quals / union_all / window functions are outside this path");
    if (u_.num_order_entries < 0 || u_.num_order_entries > B2Q_MAX_ORDER_ENTRIES) reject(B2Q_ERR_UNSUPPORTED, "more ORDER BY entries than the path carries");
    if (u_.num_order_entries && !u_.order_entries) reject(B2Q_ERR_INVALID_ARGUMENT, "order_entries is null");
    for (int i = 0; i < u_.num_order_entries; ++i)
      if (u_.order_entries[i].tle_no < 1 || u_.order_entries[i].tle_no > u_.num_target_exprs)
        reject(B2Q_ERR_INVALID_ARGUMENT, "order entry refers to a target that does not exist (tle_no is 1-based)");
    if (u_.offset < 0 || (u_.has_limit && u_.limit < 0)) reject(B2Q_ERR_INVALID_ARGUMENT, "negative LIMIT / OFFSET");
    if (u_.num_exprs < 0 || (u_.num_exprs && !u_.exprs)) reject(B2Q_ERR_INVALID_ARGUMENT, "exprs");
    /* the node array is in construction order: operands precede the node that uses them (no cycles, bounded recursion) */
    for (int i = 0; i < u_.num_exprs; ++i) {
      const B2QExpr& e = u_.exprs[i];
      if (e.left < -1 || e.left >= i || e.right < -1 || e.right >= i)
        reject(B2Q_ERR_INVALID_ARGUMENT, "expression operands must be earlier nodes of the array (or -1)");
      /* a DECIMAL compares as its scaled integer, so both sides must be DECIMALs of one scale — what the analyzer leaves
       * when the common type is the column's (constants are folded to it); otherwise it wraps the column in a CAST */
      if (e.kind == B2Q_EXPR_BIN_OPER && e.op != B2Q_kAND && e.op != B2Q_kOR && e.left >= 0 && e.right >= 0) {
        const SqlType a = from_abi(u_.exprs[e.left].ti), b = from_abi(u_.exprs[e.right].ti);
        if ((a.is_decimal() || b.is_decimal()) && !(a.is_decimal() && b.is_decimal() && a.scale == b.scale))
          reject(B2Q_ERR_UNSUPPORTED, "DECIMAL compared with a value of another type / scale needs the analyzer's cast");
      }
    }
    if (u_.num_groupby_exprs > B2Q_MAX_GROUP_COLS) reject(B2Q_ERR_UNSUPPORTED, "more GROUP BY columns than the path carries");
    if (u_.num_groupby_exprs < 0 || (u_.num_target_exprs <= 0 && !u_.has_estimator) || u_.num_target_exprs > B2Q_MAX_TARGETS)
      reject(B2Q_ERR_INVALID_ARGUMENT, "bad groupby/target counts");
    for (int c = 0; c < t_.num_cols; ++c) {
      const bool is_deleted_col = t_.deleted_column_plus1 == c + 1;
      if (t_.col_types[c].type == B2Q_kBOOLEAN) {
        if (!is_deleted_col) reject(B2Q_ERR_UNSUPPORTED, "BOOLEAN is only supported as the deleted-rows column");
        continue;
      }
      if (col_type(c).size() < 0) reject(B2Q_ERR_UNSUPPORTED, "column type outside TINYINT/SMALLINT/INT/BIGINT/DOUBLE/TIME/TIMESTAMP/DATE/dictionary-encoded strings");
      if (t_.col_encoded_sizes && t_.col_encoded_sizes[c]) {
        const int e = t_.col_encoded_sizes[c];
        if (e < 0) {
          if (t_.col_types[c].type != B2Q_kDATE || (e != -4 && e != -2)) reject(B2Q_ERR_UNSUPPORTED, "ENCODING DAYS needs a DATE column and 32 or 16 bits");
        } else if (!col_type(c).is_int() || (e != 1 && e != 2 && e != 4) || e >= col_type(c).size())
          reject(B2Q_ERR_UNSUPPORTED, "ENCODING FIXED needs an integer column and a physical width below the logical one");
      }
    }
    if (t_.deleted_column_plus1 < 0 || t_.deleted_column_plus1 > t_.num_cols) reject(B2Q_ERR_INVALID_ARGUMENT, "deleted column id out of range");
    if (t_.num_fragments < 0 || (t_.num_fragments && !t_.fragments)) reject(B2Q_ERR_INVALID_ARGUMENT, "fragments");
    for (int f = 0; f < t_.num_fragments; ++f) {
      if (t_.fragments[f].num_tuples < 0) reject(B2Q_ERR_INVALID_ARGUMENT, "negative fragment row count");
      if (t_.num_cols && !t_.fragments[f].col_stats) reject(B2Q_ERR_INVALID_ARGUMENT, "fragment without chunk stats");
    }
  }

  /* constrained_not_null (OutputBufferInitialization.cpp:301-324): one of ra_exe_unit.quals — the simple_quals are not
   * consulted — is NOT(ISNULL(col)) at its top level, for the very ColumnVar the aggregate reads */
  bool quals_constrain_not_null(const B2QExpr& col) const {
    for (int i = 0; i < u_.num_quals; ++i) {
      const B2QExpr& n = ex(u_.quals[i]);
      if (n.kind != B2Q_EXPR_UOPER || n.op != B2Q_kNOT) continue;
      const B2QExpr& isn = ex(n.left);
      if (isn.kind != B2Q_EXPR_UOPER || isn.op != B2Q_kISNULL) continue;
      const B2QExpr& c = ex(isn.left);
      if (c.kind == B2Q_EXPR_COLUMN_VAR && c.col_id == col.col_id && c.rte_idx == col.rte_idx) return true;
    }
    return false;
  }

  void build_targets() {
    const bool bigint_count = eo_.bigint_count != 0;
    bool any_agg = false;
    for (int i = 0; i < u_.num_target_exprs; ++i) {
      const B2QExpr& e = ex(u_.target_exprs[i]);
      TargetDesc d;
      if (e.kind == B2Q_EXPR_COLUMN_VAR) {
        d.is_agg = false;
        d.sql_type = from_abi(e.ti);
        d.arg_col = e.col_id;
        col_type(e.col_id);
      } else if (e.kind == B2Q_EXPR_AGG) {
        d.is_agg = true;
        d.agg = e.op;
        any_agg = true;
        if (e.op != B2Q_kCOUNT && e.op != B2Q_kSUM && e.op != B2Q_kMIN && e.op != B2Q_kMAX && e.op != B2Q_kAVG)
          reject(B2Q_ERR_UNSUPPORTED, "aggregate kind outside COUNT/SUM/MIN/MAX/AVG");
        if (e.ival != 0 && (e.op != B2Q_kCOUNT || e.left < 0)) reject(B2Q_ERR_UNSUPPORTED, "DISTINCT is on this path for COUNT(DISTINCT column) only");
        d.distinct = e.ival != 0;
        if (e.left < 0) {
          if (e.op != B2Q_kCOUNT) reject(B2Q_ERR_INVALID_ARGUMENT, "aggregate without argument must be COUNT");
          d.sql_type = SqlType{bigint_count ? B2Q_kBIGINT : B2Q_kINT, e.ti.notnull != 0};
        } else {
          const B2QExpr& a = ex(e.left);
          if (a.kind != B2Q_EXPR_COLUMN_VAR) reject(B2Q_ERR_UNSUPPORTED, "aggregate argument must be a ColumnVar");
          d.arg_col = a.col_id;
          d.arg_type = from_abi(a.ti);
          if (d.arg_type.size() != col_type(a.col_id).size()) reject(B2Q_ERR_INVALID_ARGUMENT, "ColumnVar type does not match the table");
          d.skip_null = !d.arg_type.notnull;
          d.constrained = quals_constrain_not_null(a);
          /* what the analyzer lets through (Analyzer.cpp / RelAlgTranslator): no SUM / AVG of strings or time types,
           * MIN / MAX of a dictionary string would need dictionary order */
          if (d.arg_type.is_string() && e.op != B2Q_kCOUNT) reject(B2Q_ERR_UNSUPPORTED, "only COUNT of a dictionary-encoded string is on this path");
          if (d.arg_type.is_time() && (e.op == B2Q_kSUM || e.op == B2Q_kAVG)) reject(B2Q_ERR_UNSUPPORTED, "SUM / AVG of a TIME / TIMESTAMP / DATE");
          /* SQLTypeInfo::is_integer() is false for a DECIMAL: its AVG keeps type and scale (TargetInfo.cpp:57-67) for pair_to_double */
          if (e.op == B2Q_kAVG) d.sql_type = (d.arg_type.is_int() && !d.arg_type.is_decimal()) ? SqlType{B2Q_kBIGINT, d.arg_type.notnull} : d.arg_type;
          else if (e.op == B2Q_kCOUNT) d.sql_type = SqlType{bigint_count ? B2Q_kBIGINT : B2Q_kINT, e.ti.notnull != 0};
          else d.sql_type = from_abi(e.ti);
        }
      } else {
        reject(B2Q_ERR_UNSUPPORTED, "target must be a ColumnVar or an AggExpr");
      }
      targets_.push_back(d);
    }
    if (!any_agg) reject(B2Q_ERR_UNSUPPORTED, "projection-only queries are outside this path");
    for (int i = 0; i < u_.num_order_entries; ++i) /* ResultSet::sort orders dictionary strings through the dictionary (ResultSet.cpp:1431-1446) */
      if (targets_[u_.order_entries[i].tle_no - 1].sql_type.is_string()) reject(B2Q_ERR_UNSUPPORTED, "ORDER BY a dictionary-encoded string needs the dictionary");
  }

  ColRange leaf_range(int col) const {
    ColRange r;
    const SqlType ct = col_type(col);
    r.valid = true;
    r.fp = ct.is_fp();
    int64_t total = 0;
    for (int f = 0; f < t_.num_fragments; ++f) total += t_.fragments[f].num_tuples;
    if (total == 0) return r; /* [0,-1], no nulls */
    bool first = true;
    for (int f = 0; f < t_.num_fragments; ++f) {
      const B2QFragmentInfo& fr = t_.fragments[f];
      if (fr.col_stats[col].has_nulls) r.has_nulls = true;
      if (fr.num_tuples == 0) continue;
      const B2QChunkStats& s = fr.col_stats[col];
      if (first) { r.imin = s.int_min; r.imax = s.int_max; r.fmin = s.fp_min; r.fmax = s.fp_max; first = false; }
      else {
        r.imin = std::min(r.imin, s.int_min); r.imax = std::max(r.imax, s.int_max);
        r.fmin = std::min(r.fmin, s.fp_min); r.fmax = std::max(r.fmax, s.fp_max);
      }
    }
    if (!r.fp && r.imax < r.imin) { r.imin = 0; r.imax = -1; }
    r.bucket = t_.col_types[col].type == B2Q_kDATE ? 86400 : 0;
    return r;
  }

  void narrow_by_simple_quals(int col, ColRange& r) const {
    for (int i = 0; i < u_.num_simple_quals; ++i) {
      const B2QExpr& q = ex(u_.simple_quals[i]);
      if (q.kind != B2Q_EXPR_BIN_OPER) continue;
      const B2QExpr& l = ex(q.left);
      const B2QExpr& c = ex(q.right);
      if (l.kind != B2Q_EXPR_COLUMN_VAR || l.col_id != col || c.kind != B2Q_EXPR_CONSTANT) continue;
      const bool cfp = fp_type(c.ti.type);
      if (cfp != r.fp) continue; /* mixed int/fp comparisons are never simple quals in the reference (see sqlmini.py) */
      if (r.fp) {
        const double v = cfp ? c.dval : static_cast<double>(c.ival);
        if (q.op == B2Q_kGT || q.op == B2Q_kGE || q.op == B2Q_kEQ) r.fmin = std::max(r.fmin, v);
        if (q.op == B2Q_kLT || q.op == B2Q_kLE || q.op == B2Q_kEQ) r.fmax = std::min(r.fmax, v);
      } else {
        const int64_t v = cfp ? static_cast<int64_t>(c.dval) : c.ival;
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

  static double fp_null(const SqlType& t) { return t.is_float() ? kNullFloat : kNullDouble; }
  static int64_t flt_bits(float f) { int32_t b; memcpy(&b, &f, 4); return b; } /* a float pattern in a 64-bit slot: its int32 image, sign-extended (get_agg_initial_val, OutputBufferInitialization.cpp:141-247) */

  static int64_t agg_init(int agg, const SqlType& ti, bool compaction, unsigned min_width) {
    if (ti.is_float()) { /* float_argument_input: byte_width 4 whatever the padded slot width (init_agg_val_vec :66-76) */
      switch (agg) {
        case B2Q_kSUM: return ti.notnull ? flt_bits(0.f) : flt_bits(FLT_MIN);
        case B2Q_kAVG: case B2Q_kCOUNT: return 0;
        case B2Q_kMIN: return ti.notnull ? flt_bits(FLT_MAX) : flt_bits(FLT_MIN);
        case B2Q_kMAX: return ti.notnull ? flt_bits(-FLT_MAX) : flt_bits(FLT_MIN);
        default: reject(B2Q_ERR_UNSUPPORTED, "aggregate kind");
      }
    }
    const unsigned bw = compaction ? std::max<unsigned>(ti.size(), min_width) : 8u;
    const bool fp = ti.is_fp();
    switch (agg) {
      case B2Q_kSUM:
        if (!ti.notnull) return fp ? dbl_bits(kNullDouble) : ti.int_null();
        return 0; /* +0.0 has all-zero bits */
      case B2Q_kAVG: case B2Q_kCOUNT: return 0;
      case B2Q_kMIN:
        if (fp) return dbl_bits(ti.notnull ? DBL_MAX : kNullDouble);
        if (!ti.notnull) return ti.int_null();
        return bw == 1 ? INT8_MAX : bw == 2 ? INT16_MAX : bw == 4 ? INT32_MAX : INT64_MAX;
      case B2Q_kMAX:
        if (fp) return dbl_bits(ti.notnull ? -DBL_MAX : kNullDouble);
        if (!ti.notnull) return ti.int_null();
        return bw == 1 ? INT8_MIN : bw == 2 ? INT16_MIN : bw == 4 ? INT32_MIN : INT64_MIN;
      default: reject(B2Q_ERR_UNSUPPORTED, "aggregate kind");
    }
  }

  bool any_distinct() const { for (const TargetDesc& d : targets_) if (d.distinct) return true; return false; }
  /* GroupByAndAggregate::getBaselineThreshold (:222-230): on the GPU a query with COUNT(DISTINCT) targets switches to
   * baseline hash four times earlier (g_baseline_groupby_threshold = 1e6, Execute.cpp:111) */
  int64_t baseline_threshold() const { return any_distinct() ? 1000000 / 4 : 1000000; }

  /* init_count_distinct_descriptors (GroupByAndAggregate.cpp:650-855) for COUNT(DISTINCT column): the argument's range
   * (get_expr_range_info: chunk stats narrowed by the simple quals) decides.  An integer range gives the Bitmap implementation
   * with get_bucketed_cardinality_without_nulls bits (:379-395); fp arguments, ranges of g_bitmap_memory_limit (8e9) bits and
   * more, and bitmaps that would total 8e9 bytes over the group range fall to the std::set implementation or an error in the
   * reference — neither runs on its GPU (QueryMustRunOnCpu) and both are refused here.  check_total_bitmap_memory
   * (QueryMemoryInitializer.cpp:40-66) is applied to the planned entry count as well. */
  void count_distinct_descriptors(const B2QPlan& p) {
    const int64_t limit = 8000000000ll; /* g_bitmap_memory_limit, QueryMemoryInitializer.cpp:28 */
    int64_t bytes_per_group = 0;
    for (TargetDesc& d : targets_) {
      if (!d.distinct) continue;
      if (d.arg_type.is_fp()) reject(B2Q_ERR_UNSUPPORTED, "COUNT(DISTINCT) of a floating-point column needs the set implementation (CPU only in the reference)");
      if (is_days(d.arg_col)) reject(B2Q_ERR_UNSUPPORTED, "COUNT(DISTINCT) of a days-encoded DATE is outside this path");
      ColRange r = leaf_range(d.arg_col);
      narrow_by_simple_quals(d.arg_col, r);
      if (r.imin > r.imax) { d.cd_min = 0; d.cd_bucket = r.bucket; d.cd_bits = 64; bytes_per_group += 8; continue; } /* isEmpty(): :735-744 */
      uint64_t size = static_cast<uint64_t>(r.imax) - static_cast<uint64_t>(r.imin);
      if (r.bucket) size /= static_cast<uint64_t>(r.bucket);
      const int64_t bits = size >= static_cast<uint64_t>(INT64_MAX) ? 0 : static_cast<int64_t>(size + 1);
      if (bits <= 0 || limit <= bits) reject(B2Q_ERR_UNSUPPORTED, "COUNT(DISTINCT): argument range too wide for a bitmap (set implementation, CPU only in the reference)");
      const int64_t padded = align8((bits + 7) / 8); /* compute_bytes_per_group / bitmapPaddedSizeBytes on the GPU */
      int64_t groups = 1;
      if (grouped_) { /* maximum_num_groups over the GROUP BY range (:762-764); our composite ranges carry min 0 / max = product */
        const int64_t bucket = std::max<int64_t>(p.bucket, 1);
        groups = p.max_val >= p.min_val ? (p.max_val - p.min_val + 1) / bucket : 0;
      }
      if (groups > 0 && padded >= (limit + groups - 1) / groups) reject(B2Q_ERR_UNSUPPORTED, "COUNT(DISTINCT): bitmaps over the group range exceed g_bitmap_memory_limit (set implementation or an error in the reference)");
      d.cd_min = r.imin; d.cd_bucket = r.bucket; d.cd_bits = bits;
      bytes_per_group += padded;
    }
    if (bytes_per_group && p.entry_count > 0 && bytes_per_group >= (limit + p.entry_count - 1) / p.entry_count)
      reject(B2Q_ERR_OUT_OF_GPU_MEM, "COUNT(DISTINCT) bitmaps exceed g_bitmap_memory_limit (OutOfHostMemory in the reference)");
  }

  void keyless_info() {
    bool keyless = true, found = false;
    int index = 0;
    for (const TargetDesc& d : targets_) {
      if (!found && d.is_agg && !d.distinct) { /* `!is_distinct_target(agg_info)`, GroupByAndAggregate.cpp:503 */
        const bool has_arg = d.arg_col >= 0;
        const ColRange r = has_arg ? leaf_range(d.arg_col) : ColRange{};
        switch (d.agg) {
          case B2Q_kAVG:
            ++index; /* AVG's COUNT slot is the marker */
            if (!(has_arg && !d.arg_type.notnull && (!r.valid || r.has_nulls))) found = true;
            break;
          case B2Q_kCOUNT:
            if (!(has_arg && !d.arg_type.notnull && (!r.valid || r.has_nulls))) found = true;
            break;
          case B2Q_kSUM: /* the one aggregate whose keyless test honours `arg IS NOT NULL` (GroupByAndAggregate.cpp:531-533) */
            if (!d.arg_type.notnull && !d.constrained) { if (r.valid && !r.has_nulls) found = true; }
            else if (r.fp ? (r.fmax < 0 || r.fmin > 0) : (r.imax < 0 || r.imin > 0)) found = true;
            break;
          case B2Q_kMIN: { /* note: no has_nulls test in the reference (kMAX has one) */
            const int64_t init_max = agg_init(d.agg, d.compact(), true, 8);
            if (r.fp ? (r.fmax < bits_dbl(init_max)) : (r.imax < init_max)) found = true;
            break;
          }
          case B2Q_kMAX: {
            if (!r.valid || r.has_nulls) break;
            const int64_t init_min = agg_init(d.agg, d.compact(), true, 8);
            if (r.fp ? (r.fmin > bits_dbl(init_min)) : (r.imin > init_min)) found = true;
            break;
          }
          default: keyless = false;
        }
      }
      if (!keyless) break;
      if (!found) ++index;
    }
    keyless_ = keyless && found;
    keyless_idx_ = index;
  }

  void choose_hash_type(B2QPlan& p) {
    grouped_ = u_.num_groupby_exprs >= 1;
    p.key_col_id = -1;
    p.effective_key_width = 8;
    p.idx_target_as_key = -1;
    p.num_group_cols = u_.num_groupby_exprs;
    if (!grouped_) {
      p.query_desc_type = B2Q_NonGroupedAggregate;
      p.entry_count = 1;
      return;
    }
    if (u_.num_groupby_exprs > 1) {
      /* getColRangeInfo for several GROUP BY columns (GroupByAndAggregate.cpp:240-280): perfect hash over the product
       * of the per-column cardinalities when every column has a valid integer range and the product is within
       * g_baseline_groupby_threshold (1e6); otherwise baseline hash, which for composite keys is outside this path */
      int64_t cardinality = 1;
      bool has_nulls = false;
      for (int i = 0; i < u_.num_groupby_exprs; ++i) {
        const B2QExpr& g = ex(u_.groupby_exprs[i]);
        if (g.kind != B2Q_EXPR_COLUMN_VAR) reject(B2Q_ERR_UNSUPPORTED, "GROUP BY expression must be a ColumnVar");
        if (col_type(g.col_id).is_fp()) reject(B2Q_ERR_UNSUPPORTED, "multi-column baseline hash (fp key) is outside this path");
        ColRange r = leaf_range(g.col_id);
        narrow_by_simple_quals(g.col_id, r);
        if (r.imin > r.imax) reject(B2Q_ERR_UNSUPPORTED, "multi-column baseline hash is outside this path");
        KeyComp k{g.col_id, r.imin, r.imax, 0, cardinality, r.has_nulls, r.bucket};
        int64_t span;
        const bool span_ovf = __builtin_sub_overflow(r.imax, r.imin, &span);
        if (!span_ovf && r.bucket) span /= r.bucket; /* getBucketedCardinality (:367-375) */
        if (span_ovf || __builtin_add_overflow(span, int64_t(1 + (r.has_nulls ? 1 : 0)), &k.card) ||
            __builtin_mul_overflow(cardinality, k.card, &cardinality))
          reject(B2Q_ERR_UNSUPPORTED, "multi-column baseline hash is outside this path");
        has_nulls |= r.has_nulls;
        keycomps_.push_back(k);
        p.group_col_ids[i] = g.col_id;
        p.group_col_widths[i] = static_cast<int8_t>(col_type(g.col_id).size());
      }
      if (!cardinality || cardinality > baseline_threshold()) reject(B2Q_ERR_UNSUPPORTED, "multi-column baseline hash is outside this path");
      key_col_ = keycomps_[0].col;
      p.key_col_id = key_col_;
      p.group_col_width = p.group_col_widths[0];
      p.query_desc_type = B2Q_GroupByPerfectHash;
      p.min_val = 0; p.max_val = cardinality; p.bucket = 0; p.has_nulls = has_nulls;
      keyless_info();
      p.keyless_hash = keyless_ ? 1 : 0;
      p.idx_target_as_key = keyless_idx_;
      p.entry_count = cardinality;
      return;
    }
    const B2QExpr& g = ex(u_.groupby_exprs[0]);
    if (g.kind != B2Q_EXPR_COLUMN_VAR) reject(B2Q_ERR_UNSUPPORTED, "GROUP BY expression must be a ColumnVar");
    key_col_ = g.col_id;
    const SqlType kt = col_type(key_col_);
    if (kt.is_fp()) reject(B2Q_ERR_UNSUPPORTED, "floating-point GROUP BY key (baseline double keys) is outside this path");
    p.key_col_id = key_col_;
    p.group_col_width = kt.size();
    p.group_col_ids[0] = key_col_;
    p.group_col_widths[0] = static_cast<int8_t>(kt.size());
    ColRange r = leaf_range(key_col_);
    narrow_by_simple_quals(key_col_, r);
    bool perfect = r.imin <= r.imax;
    p.has_nulls = r.has_nulls;
    if (perfect) {
      p.min_val = r.imin; p.max_val = r.imax; p.bucket = r.bucket;
      const int64_t col_count = u_.num_groupby_exprs + u_.num_target_exprs;
      int64_t max_entries = (int64_t(1) << 30) / (col_count * 8); /* kMaxBufferSize, GroupByAndAggregate.cpp:57 */
      if (any_distinct()) max_entries = std::min(max_entries, baseline_threshold()); /* :307-309 */
      int64_t span;
      const bool too_big = __builtin_sub_overflow(r.imax, r.imin, &span) || span >= max_entries;
      if (kt.is_string() && !r.bucket) {
        /* :311-356 dictionary ids are dense: a too-big range stays perfect hash unless a filter can be expected to
         * thin it out — with filters and no sort, baseline when there is no estimate yet or 2 * estimate < range */
        const bool has_filters = u_.num_quals > 0 || u_.num_simple_quals > 0;
        if (has_filters && too_big && u_.num_order_entries != 0) {
          if (any_distinct()) perfect = false; /* :329-341: with a sort the range is kept, except under COUNT(DISTINCT) */
        } else if (has_filters && too_big) {
          int64_t twice;
          const bool less = has_card_ && !__builtin_mul_overflow(static_cast<int64_t>(guess_), int64_t(2), &twice) && twice < span;
          if (!has_card_ || less) perfect = false;
        }
      } else if (too_big && !r.bucket) perfect = false; /* :357-363, keeps min/max */
      if (!perfect) p.bucket = 0;
    } else {
      p.min_val = 0; p.max_val = -1;
    }
    if (perfect) {
      p.query_desc_type = B2Q_GroupByPerfectHash;
      keyless_info();
      p.keyless_hash = (!p.bucket && keyless_) ? 1 : 0; /* QueryMemoryDescriptor.cpp:327-333; no sort hint, no baseline sort on this path */
      p.idx_target_as_key = keyless_idx_;
      int64_t card;
      if (__builtin_sub_overflow(p.max_val, p.min_val, &card)) /* only a bucketed (DATE) range gets here with an overflowing span: getBucketedCardinality (:367-375) is undefined there */
        reject(B2Q_ERR_UNSUPPORTED, "DATE key range wider than int64");
      if (p.bucket) card /= p.bucket; /* getBucketedCardinality (:367-375) */
      p.entry_count = std::max<int64_t>(card + 1 + (p.has_nulls ? 1 : 0), 1);
    } else {
      p.query_desc_type = B2Q_GroupByBaselineHash;
      if (is_days(key_col_)) reject(B2Q_ERR_UNSUPPORTED, "baseline hash over a days-encoded DATE key is outside this path");
      if (!has_card_) reject(B2Q_ERR_CARDINALITY_ESTIMATION_REQUIRED, "baseline hash group-by needs a cardinality estimate (CardinalityEstimationRequired)");
      if (guess_ == 0 || guess_ > 0xFFFFFFFFull) reject(B2Q_ERR_INVALID_ARGUMENT, "max_groups_buffer_entry_guess must be in [1, 2^32)");
      p.entry_count = static_cast<int64_t>(guess_);
      /* pick_baseline_key_width (QueryMemoryDescriptor.cpp:112-147) on the un-narrowed column range */
      const ColRange kr = leaf_range(key_col_);
      int w = 8;
      if (!(p.group_col_width == 8 && kr.has_nulls) && kr.imin > INT32_MIN && kr.imax < int64_t(INT32_MAX) - 1) w = 4;
      /* group_col_compact_width = output_columnar ? 8 : pick_baseline_key_width (QueryMemoryDescriptor.cpp:391-393) */
      p.effective_key_width = eo_.output_columnar_hint ? 8 : std::max(4, w);
      p.min_val = p.max_val = p.bucket = 0;
      p.has_nulls = 0;
    }
  }

  void layout_slots(B2QPlan& p) {
    std::vector<int8_t> logical;
    for (TargetDesc& d : targets_) {
      d.first_slot = static_cast<int>(logical.size());
      logical.push_back(static_cast<int8_t>(d.compact().size()));
      if (d.is_agg && d.agg == B2Q_kAVG) logical.push_back(8);
    }
    if (logical.size() > B2Q_MAX_SLOTS) reject(B2Q_ERR_UNSUPPORTED, "too many output slots");
    slot_key_ref_.assign(logical.size(), false);
    if (p.query_desc_type == B2Q_GroupByBaselineHash)
      for (const TargetDesc& d : targets_)
        if (!d.is_agg && d.arg_col == key_col_) slot_key_ref_[d.first_slot] = true; /* target_groupby_indices */

    /* pick_target_compact_width with crt_min_byte_width = 8 */
    int8_t width = 0;
    if (eo_.bigint_count) width = 8;
    else {
      /* QueryMemoryDescriptor.cpp:775-778: `groupby_exprs.size() != 1 || !groupby_exprs.front()` — non-grouped units and every
       * multi-column GROUP BY keep 8-byte slots; only a single-column GROUP BY can compact to 4 */
      int8_t compact = (grouped_ && u_.num_groupby_exprs == 1) ? 0 : 8;
      if (!compact) {
        for (int i = 0; i < u_.num_target_exprs && !compact; ++i) {
          const B2QExpr& e = ex(u_.target_exprs[i]);
          if (e.kind == B2Q_EXPR_AGG) { if (e.left >= 0) compact = 8; continue; }
          const SqlType ti = from_abi(e.ti);
          if (!(ti.is_int() && ti.size() <= 4)) compact = 8;
        }
      }
      if (!compact) {
        /* QueryMemoryDescriptor.cpp:826-833 sums the tuples of every input table (query_infos): with a join level, the
         * inner table's rows count too, although the combined input carries only the outer table's row counts */
        uint64_t tuples = 0;
        for (int f = 0; f < t_.num_fragments; ++f) tuples += static_cast<uint64_t>(t_.fragments[f].num_tuples);
        if (join_)
          for (int f = 0; f < inner_->num_fragments; ++f) tuples += static_cast<uint64_t>(inner_->fragments[f].num_tuples);
        width = tuples <= UINT32_MAX ? 4 : 8;
      } else {
        for (int i = 0; i < u_.num_target_exprs; ++i) compact = std::max<int8_t>(compact, static_cast<int8_t>(from_abi(ex(u_.target_exprs[i]).ti).size()));
        width = compact;
      }
    }
    p.num_targets = static_cast<int32_t>(targets_.size());
    p.num_slots = static_cast<int32_t>(logical.size());
    /* QueryMemoryDescriptor ctor (:510-536): without GPU sort the columnar decision is the hint itself */
    p.output_columnar = eo_.output_columnar_hint ? 1 : 0;
    if (p.output_columnar) {
      /* ResultSet.h:72-84: [key columns, int64 each, absent if keyless][slot columns], every column 8-byte aligned
       * (getPrependedGroupBufferSizeInBytes :987-997, getColOffInBytes :920-944) */
      if (grouped_ && !p.keyless_hash && p.group_col_widths[0] != 8)
        /* isEmptyEntryColumnar (ResultSetIteration.cpp:2533-2543) reads the first key column at the COLUMN's width
         * although initColumnarGroups stores int64 keys: the reference's own reader/reduce misjudge emptiness, so
         * there is no defined result to reproduce */
        reject(B2Q_ERR_UNSUPPORTED, "columnar output with a stored GROUP BY key narrower than 8 bytes (reference reader reads it at the column's width)");
      int64_t off = (grouped_ && !p.keyless_hash) ? static_cast<int64_t>(u_.num_groupby_exprs) * align8(8 * p.entry_count) : 0;
      int64_t cols_size = 0;
      for (size_t s = 0; s < logical.size(); ++s) {
        p.slot_offset[s] = off;
        if (slot_key_ref_[s]) { p.slot_logical_width[s] = p.slot_padded_width[s] = 0; continue; }
        if (logical[s] > width) reject(B2Q_ERR_UNSUPPORTED, "slot wider than the compact width");
        p.slot_logical_width[s] = logical[s];
        p.slot_padded_width[s] = width;
        off += align8(static_cast<int64_t>(width) * p.entry_count);
        cols_size += width;
      }
      p.row_size = align8(cols_size);
      p.buffer_size = off;
      return;
    }
    const int64_t key_bytes = (grouped_ && !p.keyless_hash) ? align8(static_cast<int64_t>(u_.num_groupby_exprs) * p.effective_key_width) : 0;
    int64_t cols = 0;
    for (size_t s = 0; s < logical.size(); ++s) {
      if (slot_key_ref_[s]) { p.slot_logical_width[s] = p.slot_padded_width[s] = 0; p.slot_offset[s] = key_bytes + cols; continue; }
      if (logical[s] > width) reject(B2Q_ERR_UNSUPPORTED, "slot wider than the compact width");
      p.slot_logical_width[s] = logical[s];
      p.slot_padded_width[s] = width;
      if (width == 8) cols = align8(cols);
      p.slot_offset[s] = key_bytes + cols;
      cols += width;
    }
    p.row_size = align8(key_bytes + cols);
    p.buffer_size = p.row_size * p.entry_count;
  }

  void init_values(B2QPlan& p) {
    int8_t compact_width = 8;
    for (int s = 0; s < p.num_slots; ++s) if (p.slot_padded_width[s]) { compact_width = p.slot_padded_width[s]; break; }
    int s = 0;
    for (const TargetDesc& d : targets_) {
      if (!d.is_agg) { p.init_vals[s++] = 0; continue; }
      SqlType ti = d.compact();
      if (d.constrained && d.arg_col >= 0) ti.notnull = true; /* set_notnull(target, true), OutputBufferInitialization.cpp:287-289 */
      if (!grouped_) ti.notnull = false; /* non-grouped aggregates are nullable (OutputBufferInitialization.cpp:66-68,283-288) */
      p.init_vals[s++] = agg_init(d.agg, ti, grouped_, compact_width);
      if (d.agg == B2Q_kAVG) p.init_vals[s++] = 0;
    }
  }

  void publish_targets(B2QPlan& p) {
    for (size_t i = 0; i < targets_.size(); ++i) {
      TargetDesc& d = targets_[i];
      if (d.is_agg && d.arg_col >= 0 && !grouped_) d.skip_null = true; /* TargetExprBuilder.cpp:653-657 */
      else if (d.is_agg && d.arg_col >= 0 && d.constrained) d.skip_null = false; /* :690-692 */
      B2QTargetInfo& o = p.targets[i];
      o.is_agg = d.is_agg; o.agg_kind = d.agg;
      o.sql_type = to_abi(d.sql_type); o.agg_arg_type = to_abi(d.arg_type);
      o.skip_null_val = d.skip_null; o.is_distinct = d.distinct ? 1 : 0; o.arg_col_id = d.arg_col; o.first_slot = d.first_slot;
      p.count_distinct_min[i] = d.distinct ? d.cd_min : 0;
      p.count_distinct_bits[i] = d.distinct ? d.cd_bits : 0;
    }
  }

  /* ---------------- lowering to the device program ---------------- */
  int launch_col(B2QQuery& q, int table_col) {
    for (int i = 0; i < q.prog.n_cols; ++i) if (q.col_ids[i] == table_col) return i;
    if (q.prog.n_cols >= B2Q_MAX_COLS) reject(B2Q_ERR_UNSUPPORTED, "too many referenced columns");
    q.col_ids[q.prog.n_cols] = table_col;
    q.prog.col_inner[q.prog.n_cols] = (join_ && table_col >= n_outer_) ? 1 : 0;
    /* what an unmatched LEFT-join row reads: the column's own NULL as STORED (a FLOAT is widened after the load) */
    q.prog.col_null[q.prog.n_cols] = col_type(table_col).is_float() ? flt_bits(FLT_MIN) : col_type(table_col).is_fp() ? dbl_bits(kNullDouble) : (t_.col_types[table_col].type == B2Q_kBOOLEAN ? 0 : phys_int_null(table_col));
    q.prog.col_width[q.prog.n_cols] = static_cast<int8_t>(t_.col_types[table_col].type == B2Q_kBOOLEAN ? 1 : phys_size(table_col));
    return q.prog.n_cols++;
  }

  std::vector<double> term_sel_; /* estimated selectivity per filter term (uniformity assumption over chunk stats) */

  /* `range`: the comparison is `=` ("in") / `<>` ("not in") against the closed interval [range[0], range[1]] that a
   * chain of leaves on this column folded into (lower_chain_items); its own constant only supplies the type */
  void lower_cmp(B2QQuery& q, const B2QExpr& e, const int64_t* range = nullptr, const double* frange = nullptr) {
    DevFilter& f = q.prog.filter;
    const B2QExpr& l = ex(e.left);
    const B2QExpr& c = ex(e.right);
    if (l.kind == B2Q_EXPR_COLUMN_VAR && c.kind == B2Q_EXPR_COLUMN_VAR) { lower_cmp_cols(q, e, l, c); return; }
    if (l.kind != B2Q_EXPR_COLUMN_VAR || c.kind != B2Q_EXPR_CONSTANT) reject(B2Q_ERR_UNSUPPORTED, "comparison must be ColumnVar OP Constant or ColumnVar OP ColumnVar");
    if (f.n_terms >= B2Q_MAX_TERMS || f.n_ops >= B2Q_MAX_FILTER_OPS) reject(B2Q_ERR_UNSUPPORTED, "filter too large");
    const SqlType ct = col_type(l.col_id);
    const ColRange cr = leaf_range(l.col_id);
    DevTerm t;
    memset(&t, 0, sizeof(t));
    t.col2 = -1;
    t.col = launch_col(q, l.col_id);
    t.width = static_cast<int8_t>(phys_width_code(l.col_id));
    t.col_is_fp = ct.is_fp();
    if (ct.is_string() && e.op != B2Q_kEQ && e.op != B2Q_kNE) reject(B2Q_ERR_UNSUPPORTED, "dictionary-encoded strings compare by id: only = and <> are on this path");
    if (ct.is_string() && fp_type(c.ti.type)) reject(B2Q_ERR_INVALID_ARGUMENT, "string column compared with a floating-point constant");
    const bool nullable = !ct.notnull;
    t.null_bits = ct.is_fp() ? dbl_bits(fp_null(ct)) : phys_int_null(l.col_id);
    const bool cfp = fp_type(c.ti.type);
    if (cfp && is_days(l.col_id)) reject(B2Q_ERR_UNSUPPORTED, "days-encoded DATE compared with a floating-point constant");
    t.cmp_fp = ct.is_fp() || cfp;
    bool negate = e.op == B2Q_kNE;
    const double inf = std::numeric_limits<double>::infinity();
    double sel = 0.5;
    if (t.cmp_fp) {
      /* closed fp range; default empty (never TRUE; under negate always TRUE except NULL) */
      t.flo = inf; t.fhi = -inf;
      if (c.is_null) negate = false; /* comparison with a NULL literal is never TRUE */
      else {
        const double k = cfp ? c.dval : static_cast<double>(c.ival);
        if (!std::isnan(k)) {
          switch (e.op) {
            case B2Q_kEQ: case B2Q_kNE: t.flo = frange ? frange[0] : k; t.fhi = frange ? frange[1] : k; break;
            case B2Q_kLT: if (k != -inf) { t.flo = -inf; t.fhi = std::nextafter(k, -inf); } break;
            case B2Q_kLE: t.flo = -inf; t.fhi = k; break;
            case B2Q_kGT: if (k != inf) { t.flo = std::nextafter(k, inf); t.fhi = inf; } break;
            case B2Q_kGE: t.flo = k; t.fhi = inf; break;
            default: reject(B2Q_ERR_UNSUPPORTED, "comparison operator");
          }
        }
      }
      t.negate = negate;
      t.null_check = nullable; /* NULL_DOUBLE sits inside the value range: always test explicitly */
      const double cmin = cr.fp ? cr.fmin : static_cast<double>(cr.imin), cmax = cr.fp ? cr.fmax : static_cast<double>(cr.imax);
      if (cmax > cmin && t.flo <= t.fhi) sel = std::max(0.0, std::min(t.fhi, cmax) - std::max(t.flo, cmin)) / (cmax - cmin);
      else if (t.flo > t.fhi) sel = 0.0;
      if (negate) sel = 1.0 - sel;
    } else {
      int64_t lo = 1, hi = 0; /* empty */
      if (c.is_null) negate = false;
      else {
        const int64_t k = c.ival;
        switch (e.op) {
          case B2Q_kEQ: case B2Q_kNE: lo = range ? range[0] : k; hi = range ? range[1] : k; break;
          case B2Q_kLT: if (k != INT64_MIN) { lo = INT64_MIN; hi = k - 1; } break;
          case B2Q_kLE: lo = INT64_MIN; hi = k; break;
          case B2Q_kGT: if (k != INT64_MAX) { lo = k + 1; hi = INT64_MAX; } break;
          case B2Q_kGE: lo = k; hi = INT64_MAX; break;
          default: reject(B2Q_ERR_UNSUPPORTED, "comparison operator");
        }
      }
      /* selectivity estimate on the un-clamped range */
      if (cr.imax >= cr.imin && lo <= hi) {
        const double ov = static_cast<double>(std::min(hi, cr.imax)) - static_cast<double>(std::max(lo, cr.imin)) + 1.0;
        sel = std::max(0.0, ov) / (static_cast<double>(cr.imax) - static_cast<double>(cr.imin) + 1.0);
      } else if (lo > hi) sel = 0.0;
      if (negate) sel = 1.0 - sel;
      if (is_days(l.col_id) && lo <= hi) {
        /* days * 86400 in [lo, hi]  <=>  days in [ceil(lo / 86400), floor(hi / 86400)]: a constant off the day grid
         * leaves `=` with an empty range, exactly as the decoded comparison would */
        if (lo != INT64_MIN) lo = ceil_div(lo, 86400);
        if (hi != INT64_MAX) hi = floor_div(hi, 86400);
      }
      /* clamp to the column's register class: 32-bit compares for 1/2/4-byte columns */
      const int64_t dmin = t.width <= 4 ? INT32_MIN : INT64_MIN, dmax = t.width <= 4 ? INT32_MAX : INT64_MAX;
      lo = std::max(lo, dmin);
      hi = std::min(hi, dmax);
      const int64_t nullv = phys_int_null(l.col_id);
      bool null_check = false;
      if (nullable) {
        if (negate) null_check = true;                      /* v != k must still fail for NULL */
        else if (lo <= hi && lo <= nullv && nullv <= hi) lo = nullv + 1; /* NULL is the type's minimum: cut it off the range */
      }
      if (lo > hi) { /* never in range: encode as "always in range" with the negation flipped */
        t.lo = 0;
        t.span = t.width <= 4 ? 0xFFFFFFFFull : ~0ull;
        negate = !negate;
      } else {
        t.lo = lo;
        t.span = static_cast<uint64_t>(hi) - static_cast<uint64_t>(lo);
      }
      t.negate = negate;
      t.null_check = null_check;
    }
    term_sel_.push_back(std::min(1.0, std::max(0.0, sel)));
    f.ops[f.n_ops++] = static_cast<uint8_t>((FOP_TERM << 4) | f.n_terms);
    f.terms[f.n_terms++] = t;
  }

  /* ColumnVar OP ColumnVar: the analyzer casts both sides to their common type (integers to the wider one, anything
   * with a DOUBLE to DOUBLE) and DEF_CMP_NULLABLE yields TRUE only when neither side is NULL */
  void lower_cmp_cols(B2QQuery& q, const B2QExpr& e, const B2QExpr& l, const B2QExpr& r) {
    DevFilter& f = q.prog.filter;
    if (f.n_terms >= B2Q_MAX_TERMS || f.n_ops >= B2Q_MAX_FILTER_OPS) reject(B2Q_ERR_UNSUPPORTED, "filter too large");
    if (e.op != B2Q_kEQ && e.op != B2Q_kNE && e.op != B2Q_kLT && e.op != B2Q_kGT && e.op != B2Q_kLE && e.op != B2Q_kGE) reject(B2Q_ERR_UNSUPPORTED, "comparison operator");
    const SqlType lt = col_type(l.col_id), rt = col_type(r.col_id);
    if (is_days(l.col_id) != is_days(r.col_id)) reject(B2Q_ERR_UNSUPPORTED, "days-encoded DATE compared with a column of another encoding");
    if (lt.is_string() != rt.is_string() || (lt.is_string() && e.op != B2Q_kEQ && e.op != B2Q_kNE))
      reject(B2Q_ERR_UNSUPPORTED, "dictionary-encoded strings compare by id: only = and <> between two string columns of one dictionary");
    DevTerm t;
    memset(&t, 0, sizeof(t));
    t.col = launch_col(q, l.col_id);
    t.width = static_cast<int8_t>(phys_width_code(l.col_id));
    t.col_is_fp = lt.is_fp();
    t.null_bits = lt.is_fp() ? dbl_bits(fp_null(lt)) : phys_int_null(l.col_id);
    t.nullable1 = !lt.notnull;
    t.col2 = launch_col(q, r.col_id);
    t.width2 = static_cast<int8_t>(phys_width_code(r.col_id));
    t.col2_is_fp = rt.is_fp();
    t.null_bits2 = rt.is_fp() ? dbl_bits(fp_null(rt)) : phys_int_null(r.col_id);
    t.nullable2 = !rt.notnull;
    t.cmp_fp = lt.is_fp() || rt.is_fp();
    t.op2 = static_cast<int8_t>(e.op);
    term_sel_.push_back(e.op == B2Q_kEQ ? 0.05 : e.op == B2Q_kNE ? 0.95 : 0.5);
    f.ops[f.n_ops++] = static_cast<uint8_t>((FOP_TERM << 4) | f.n_terms);
    f.terms[f.n_terms++] = t;
  }

  double estimate_selectivity(const DevFilter& f) const {
    if (f.n_ops == 0) return 1.0;
    double st[8];
    int sp = 0;
    for (int i = 0; i < f.n_ops; ++i) {
      const int kind = f.ops[i] >> 4;
      if (kind == FOP_TERM) st[sp++] = term_sel_[f.ops[i] & 15];
      else {
        const double b = st[--sp], a = st[--sp];
        st[sp++] = kind == FOP_AND ? a * b : 1.0 - (1.0 - a) * (1.0 - b);
      }
      if (sp >= 7) break;
    }
    return sp > 0 ? st[sp - 1] : 1.0;
  }

  /* Quals are lowered to postfix AND / OR over "is TRUE" bits.  NOT never reaches the device: in Kleene logic
   * (logical_and / logical_or / logical_not, RuntimeFunctions.cpp:331-357) NOT distributes over AND / OR by De Morgan,
   * NOT(col OP k) is the inverse comparison (still NULL -> not TRUE), and NOT(col IS NULL) is two-valued, so the
   * host pushes the negation down to the leaves. */
  static int inverse_cmp(int op) {
    switch (op) {
      case B2Q_kEQ: return B2Q_kNE; case B2Q_kNE: return B2Q_kEQ;
      case B2Q_kLT: return B2Q_kGE; case B2Q_kGE: return B2Q_kLT;
      case B2Q_kGT: return B2Q_kLE; case B2Q_kLE: return B2Q_kGT;
      default: return -1;
    }
  }
  int stack_need(int idx) const { /* mask-stack slots the postfix evaluation of this subtree needs */
    const B2QExpr& e = ex(idx);
    if (e.kind == B2Q_EXPR_UOPER) return e.op == B2Q_kNOT ? stack_need(e.left) : 1;
    if (e.kind == B2Q_EXPR_BIN_OPER && (e.op == B2Q_kAND || e.op == B2Q_kOR)) {
      const int l = stack_need(e.left), r = stack_need(e.right);
      return l == r ? l + 1 : std::max(l, r);
    }
    return 1;
  }

  /* ---- IN lists: `c = v1 OR c = v2 OR ...` (what the analyzer expands a short IN list to) and its negation
   * `c <> v1 AND c <> v2 AND ...`.  Values that are consecutive in the column's domain (step 1; one day for a
   * days-encoded DATE) fold into ONE range term — fewer loads and compares per row, and long dense lists fit the
   * 16-leaf program. ---- */
  struct ChainItem { int idx; bool negated; };
  void flatten_chain(int idx, bool negated, bool want_and, std::vector<ChainItem>& out) const {
    const B2QExpr& e = ex(idx);
    if (e.kind == B2Q_EXPR_UOPER && e.op == B2Q_kNOT) { flatten_chain(e.left, !negated, want_and, out); return; }
    if (e.kind == B2Q_EXPR_BIN_OPER && (e.op == B2Q_kAND || e.op == B2Q_kOR) && ((e.op == B2Q_kAND) != negated) == want_and) {
      flatten_chain(e.left, negated, want_and, out);
      flatten_chain(e.right, negated, want_and, out);
      return;
    }
    out.push_back({idx, negated});
  }
  /* a leaf `int column OP k` (k a non-NULL integer constant) as the closed interval of values that satisfy it, after the
   * pending negation is applied; `<>` is not an interval (is_ne) */
  bool interval_leaf(const ChainItem& it, int* col, int64_t* lo, int64_t* hi, bool* is_ne) const {
    const B2QExpr& e = ex(it.idx);
    if (e.kind != B2Q_EXPR_BIN_OPER || e.op == B2Q_kAND || e.op == B2Q_kOR) return false;
    const int op = it.negated ? inverse_cmp(e.op) : e.op;
    const B2QExpr& l = ex(e.left);
    const B2QExpr& c = ex(e.right);
    if (l.kind != B2Q_EXPR_COLUMN_VAR || c.kind != B2Q_EXPR_CONSTANT || c.is_null || fp_type(c.ti.type)) return false;
    if (col_type(l.col_id).is_fp()) return false;
    const int64_t k = c.ival;
    *col = l.col_id;
    *is_ne = false;
    switch (op) {
      case B2Q_kEQ: *lo = k; *hi = k; return true;
      case B2Q_kNE: *lo = k; *hi = k; *is_ne = true; return true;
      case B2Q_kLT: if (k == INT64_MIN) { *lo = 1; *hi = 0; } else { *lo = INT64_MIN; *hi = k - 1; } return true;
      case B2Q_kLE: *lo = INT64_MIN; *hi = k; return true;
      case B2Q_kGT: if (k == INT64_MAX) { *lo = 1; *hi = 0; } else { *lo = k + 1; *hi = INT64_MAX; } return true;
      case B2Q_kGE: *lo = k; *hi = INT64_MAX; return true;
      default: return false;
    }
  }

  /* the same for a DOUBLE column: closed interval of doubles (`<` / `>` step to the neighbouring double) */
  bool interval_leaf_fp(const ChainItem& it, int* col, double* lo, double* hi, bool* is_ne) const {
    const B2QExpr& e = ex(it.idx);
    if (e.kind != B2Q_EXPR_BIN_OPER || e.op == B2Q_kAND || e.op == B2Q_kOR) return false;
    const int op = it.negated ? inverse_cmp(e.op) : e.op;
    const B2QExpr& l = ex(e.left);
    const B2QExpr& c = ex(e.right);
    if (l.kind != B2Q_EXPR_COLUMN_VAR || c.kind != B2Q_EXPR_CONSTANT || c.is_null || !col_type(l.col_id).is_fp()) return false;
    const double k = fp_type(c.ti.type) ? c.dval : static_cast<double>(c.ival);
    if (std::isnan(k)) return false;
    const double inf = std::numeric_limits<double>::infinity();
    *col = l.col_id;
    *is_ne = false;
    switch (op) {
      case B2Q_kEQ: *lo = k; *hi = k; return true;
      case B2Q_kNE: *lo = k; *hi = k; *is_ne = true; return true;
      case B2Q_kLT: if (k == -inf) { *lo = inf; *hi = -inf; } else { *lo = -inf; *hi = std::nextafter(k, -inf); } return true;
      case B2Q_kLE: *lo = -inf; *hi = k; return true;
      case B2Q_kGT: if (k == inf) { *lo = inf; *hi = -inf; } else { *lo = std::nextafter(k, inf); *hi = inf; } return true;
      case B2Q_kGE: *lo = k; *hi = inf; return true;
      default: return false;
    }
  }

  /* Lowers the items of one AND / OR chain.  Leaves on the SAME integer column fold:
   *  - AND: every `=`, `<`, `<=`, `>`, `>=` leaf into the intersection of their intervals (BETWEEN is one range test);
   *         runs of consecutive values of `<>` leaves (NOT IN) into one negated range each;
   *  - OR:  runs of consecutive values of `=` leaves (IN) into one range each; `c < a OR c > b` (NOT BETWEEN) into the
   *         negated range [a, b].
   * NULL behaves as in the unfolded chain: every leaf on a NULL value is NULL, so the chain's contribution is "not
   * TRUE" — exactly what one range term yields (lower_cmp keeps NULL out of the range / adds the NULL check).
   * Returns -1 when nothing folds (the caller lowers the binary tree as it is). */
  struct ChainEmit { int need; bool is_range; size_t item; int64_t lo, hi; bool negate; bool is_fp = false; double flo = 0, fhi = 0; };
  int lower_chain_items(B2QQuery& q, const std::vector<ChainItem>& items, int depth, bool want_and) {
    struct Leaf { size_t item; int64_t lo, hi; bool is_ne; };
    std::map<int, std::vector<Leaf>> by_col;
    for (size_t i = 0; i < items.size(); ++i) {
      int col;
      Leaf lf{i, 0, 0, false};
      if (interval_leaf(items[i], &col, &lf.lo, &lf.hi, &lf.is_ne)) by_col[col].push_back(lf);
    }
    std::vector<ChainEmit> emits;
    std::vector<bool> consumed(items.size(), false);
    bool folded = false;
    for (auto& g : by_col) {
      const int64_t step = is_days(g.first) ? 86400 : 1;
      /* points to fold into runs: `<>` leaves of an AND chain, `=` leaves of an OR chain */
      std::vector<std::pair<int64_t, size_t>> pts;
      std::vector<Leaf> ranges; /* AND: every non-`<>` leaf; OR: the one-sided leaves */
      for (const Leaf& lf : g.second) {
        const bool point = lf.lo == lf.hi;
        if (want_and ? lf.is_ne : (point && !lf.is_ne)) pts.push_back({lf.lo, lf.item});
        else if (!lf.is_ne) ranges.push_back(lf);
      }
      bool on_grid = true;
      for (const auto& v : pts) on_grid &= v.first % step == 0;
      if (pts.size() >= 2 && on_grid) { /* a DATE constant off the day grid matches nothing: those stay single leaves */
        std::sort(pts.begin(), pts.end());
        size_t run_begin = 0;
        for (size_t i = 1; i <= pts.size(); ++i) {
          int64_t gap = 0;
          if (i < pts.size() && !__builtin_sub_overflow(pts[i].first, pts[i - 1].first, &gap) && (gap == step || gap == 0)) continue;
          if (i - run_begin > 1) {
            emits.push_back({1, true, pts[run_begin].second, pts[run_begin].first, pts[i - 1].first, want_and});
            for (size_t k = run_begin; k < i; ++k) consumed[pts[k].second] = true;
            folded = true;
          }
          run_begin = i;
        }
      }
      if (want_and && ranges.size() >= 2) {
        int64_t lo = INT64_MIN, hi = INT64_MAX;
        bool empty = false;
        for (const Leaf& lf : ranges) {
          if (lf.lo > lf.hi) empty = true;
          lo = std::max(lo, lf.lo);
          hi = std::min(hi, lf.hi);
        }
        if (empty || lo > hi) { lo = 1; hi = 0; }
        emits.push_back({1, true, ranges[0].item, lo, hi, false});
        for (const Leaf& lf : ranges) consumed[lf.item] = true;
        folded = true;
      } else if (!want_and && ranges.size() == 2) {
        const Leaf& a = ranges[0].lo == INT64_MIN ? ranges[0] : ranges[1]; /* upper-bounded: c <= a.hi */
        const Leaf& b = ranges[0].lo == INT64_MIN ? ranges[1] : ranges[0]; /* lower-bounded: c >= b.lo */
        if (a.lo == INT64_MIN && a.lo <= a.hi && a.hi != INT64_MAX && b.hi == INT64_MAX && b.lo <= b.hi && b.lo != INT64_MIN && a.hi < b.lo) {
          emits.push_back({1, true, a.item, a.hi + 1, b.lo - 1, true}); /* NOT in (a.hi, b.lo) */
          consumed[a.item] = consumed[b.item] = true;
          folded = true;
        }
      }
    }
    /* DOUBLE columns: bounds intersect (AND), `d < a OR d > b` is the negated range (OR); no runs of points */
    {
      struct FLeaf { size_t item; double lo, hi; };
      std::map<int, std::vector<FLeaf>> fby_col;
      for (size_t i = 0; i < items.size(); ++i) {
        int col;
        double lo, hi;
        bool is_ne;
        if (!consumed[i] && interval_leaf_fp(items[i], &col, &lo, &hi, &is_ne) && !is_ne) fby_col[col].push_back({i, lo, hi});
      }
      const double inf = std::numeric_limits<double>::infinity();
      for (auto& g : fby_col) {
        std::vector<FLeaf>& ranges = g.second;
        if (want_and && ranges.size() >= 2) {
          double lo = -inf, hi = inf;
          for (const FLeaf& lf : ranges) { lo = std::max(lo, lf.lo); hi = std::min(hi, lf.hi); }
          if (lo > hi) { lo = inf; hi = -inf; }
          ChainEmit em{1, true, ranges[0].item, 0, 0, false};
          em.is_fp = true; em.flo = lo; em.fhi = hi;
          emits.push_back(em);
          for (const FLeaf& lf : ranges) consumed[lf.item] = true;
          folded = true;
        } else if (!want_and && ranges.size() == 2) {
          const FLeaf& a = ranges[0].lo == -inf ? ranges[0] : ranges[1]; /* d <= a.hi */
          const FLeaf& b = ranges[0].lo == -inf ? ranges[1] : ranges[0]; /* d >= b.lo */
          if (a.lo == -inf && a.hi != inf && a.hi != -inf && b.hi == inf && b.lo != -inf && b.lo != inf && a.hi < b.lo) {
            ChainEmit em{1, true, a.item, 0, 0, true};
            em.is_fp = true; em.flo = std::nextafter(a.hi, inf); em.fhi = std::nextafter(b.lo, -inf); /* NOT in the open gap */
            emits.push_back(em);
            consumed[a.item] = consumed[b.item] = true;
            folded = true;
          }
        }
      }
    }
    if (want_and) {
      /* `c IS NOT NULL` next to a comparison on c in the same AND chain adds nothing: a comparison is never TRUE on NULL */
      std::vector<bool> compared(static_cast<size_t>(t_.num_cols), false);
      for (size_t i = 0; i < items.size(); ++i) {
        int col;
        int64_t lo, hi;
        double flo, fhi;
        bool ne;
        if (interval_leaf(items[i], &col, &lo, &hi, &ne) || interval_leaf_fp(items[i], &col, &flo, &fhi, &ne)) compared[col] = true;
      }
      for (size_t i = 0; i < items.size(); ++i) {
        const B2QExpr& e = ex(items[i].idx);
        if (consumed[i] || e.kind != B2Q_EXPR_UOPER || e.op != B2Q_kISNULL || !items[i].negated) continue;
        const B2QExpr& l = ex(e.left);
        if (l.kind == B2Q_EXPR_COLUMN_VAR && l.col_id >= 0 && l.col_id < t_.num_cols && compared[l.col_id]) {
          consumed[i] = true;
          folded = true;
        }
      }
    }
    if (!folded) return -1;
    for (size_t i = 0; i < items.size(); ++i)
      if (!consumed[i]) emits.push_back({stack_need(items[i].idx), false, i, 0, 0, false});
    std::stable_sort(emits.begin(), emits.end(), [](const ChainEmit& a, const ChainEmit& b) { return a.need > b.need; });
    DevFilter& f = q.prog.filter;
    int max_depth = depth;
    for (size_t i = 0; i < emits.size(); ++i) {
      const ChainEmit& em = emits[i];
      const int at = depth + (i ? 1 : 0);
      if (em.is_range) {
        B2QExpr leaf = ex(items[em.item].idx);
        leaf.op = em.negate ? B2Q_kNE : B2Q_kEQ; /* the pending negation is already applied */
        const int64_t range[2] = {em.lo, em.hi};
        const double frange[2] = {em.flo, em.fhi};
        if (em.is_fp) lower_cmp(q, leaf, nullptr, frange);
        else lower_cmp(q, leaf, range);
        max_depth = std::max(max_depth, at + 1);
      } else {
        max_depth = std::max(max_depth, lower_bool(q, items[em.item].idx, at, items[em.item].negated));
      }
      if (i) {
        if (f.n_ops >= B2Q_MAX_FILTER_OPS) reject(B2Q_ERR_UNSUPPORTED, "filter too large");
        f.ops[f.n_ops++] = static_cast<uint8_t>((want_and ? FOP_AND : FOP_OR) << 4);
      }
    }
    return max_depth;
  }
  int lower_in_list_chain(B2QQuery& q, int idx, int depth, bool negated, bool want_and) {
    std::vector<ChainItem> items;
    flatten_chain(idx, negated, want_and, items);
    return lower_chain_items(q, items, depth, want_and);
  }

  int lower_bool(B2QQuery& q, int idx, int depth, bool negated = false) { /* returns max stack depth used */
    const B2QExpr& e = ex(idx);
    if (e.kind == B2Q_EXPR_UOPER) {
      if (e.op == B2Q_kNOT) return lower_bool(q, e.left, depth, !negated);
      if (e.op == B2Q_kISNULL) { lower_is_null(q, e, negated); return depth + 1; }
      reject(B2Q_ERR_UNSUPPORTED, "unary operator outside NOT / IS NULL");
    }
    if (e.kind != B2Q_EXPR_BIN_OPER) reject(B2Q_ERR_UNSUPPORTED, "qual must be a BinOper or NOT / IS NULL");
    if (e.op == B2Q_kAND || e.op == B2Q_kOR) {
      /* the device evaluates the postfix program on a 4-deep stack of row masks: lowering the operand that needs the
       * deeper stack FIRST (Sethi-Ullman; AND / OR are symmetric in the reference's three-valued logic too,
       * RuntimeFunctions.cpp:331-357) lets any tree of up to 16 terms fit */
      {
        const int folded = lower_in_list_chain(q, idx, depth, negated, (e.op == B2Q_kAND) != negated);
        if (folded >= 0) return folded;
      }
      const bool right_first = stack_need(e.right) > stack_need(e.left);
      const int d1 = lower_bool(q, right_first ? e.right : e.left, depth, negated);
      const int d2 = lower_bool(q, right_first ? e.left : e.right, depth + 1, negated);
      DevFilter& f = q.prog.filter;
      if (f.n_ops >= B2Q_MAX_FILTER_OPS) reject(B2Q_ERR_UNSUPPORTED, "filter too large");
      const bool is_and = (e.op == B2Q_kAND) != negated; /* De Morgan */
      f.ops[f.n_ops++] = static_cast<uint8_t>((is_and ? FOP_AND : FOP_OR) << 4);
      return std::max(d1, d2);
    }
    if (negated) {
      B2QExpr inv = e;
      inv.op = inverse_cmp(e.op);
      if (inv.op < 0) reject(B2Q_ERR_UNSUPPORTED, "comparison operator");
      lower_cmp(q, inv);
    } else {
      lower_cmp(q, e);
    }
    return depth + 1;
  }

  /* <ColumnVar> IS [NOT] NULL (CodeGenerator::codegenIsNull, LogicalIR.cpp:381-432): constant false for a NOT NULL
   * column, else value == NULL sentinel — a closed range [null, null] without the usual NULL exclusion */
  void lower_is_null(B2QQuery& q, const B2QExpr& e, bool negated) {
    DevFilter& f = q.prog.filter;
    const B2QExpr& l = ex(e.left);
    if (l.kind != B2Q_EXPR_COLUMN_VAR) reject(B2Q_ERR_UNSUPPORTED, "IS NULL operand must be a ColumnVar");
    if (f.n_terms >= B2Q_MAX_TERMS || f.n_ops >= B2Q_MAX_FILTER_OPS) reject(B2Q_ERR_UNSUPPORTED, "filter too large");
    const SqlType ct = col_type(l.col_id);
    DevTerm t;
    memset(&t, 0, sizeof(t));
    t.col2 = -1;
    t.col = launch_col(q, l.col_id);
    t.width = static_cast<int8_t>(phys_width_code(l.col_id));
    t.col_is_fp = ct.is_fp();
    t.cmp_fp = ct.is_fp();
    t.null_bits = ct.is_fp() ? dbl_bits(fp_null(ct)) : phys_int_null(l.col_id);
    t.null_check = 0;
    double sel;
    if (ct.notnull) { /* never NULL: "always in range" + negate encodes the constant FALSE */
      t.lo = 0;
      t.span = t.width == 8 ? ~0ull : 0xFFFFFFFFull;
      t.flo = -std::numeric_limits<double>::infinity(); t.fhi = std::numeric_limits<double>::infinity();
      t.negate = !negated;
      sel = negated ? 1.0 : 0.0;
    } else {
      const int64_t nullv = phys_int_null(l.col_id);
      t.lo = nullv; t.span = 0;
      t.flo = t.fhi = fp_null(ct);
      t.negate = negated;
      const ColRange cr = leaf_range(l.col_id);
      sel = cr.has_nulls ? 0.1 : 0.0;
      if (negated) sel = 1.0 - sel;
    }
    term_sel_.push_back(sel);
    f.ops[f.n_ops++] = static_cast<uint8_t>((FOP_TERM << 4) | f.n_terms);
    f.terms[f.n_terms++] = t;
  }

  /* scan-side parameters of a DATE key with the day bucket.  Days-encoded chunk: idx = days - first_day (no division
   * on the device).  8-byte chunk: idx = (seconds - min) / 86400, the kernel divides and checks the day grid.
   * A DATE under ENCODING FIXED(32) (legacy seconds-in-int32) would need the division on the 32-bit key path. */
  void day_key(int col, int64_t min_secs, int64_t* min_out, int8_t* div_day) const {
    if (is_days(col)) { *min_out = ceil_div(min_secs, 86400); *div_day = 0; return; }
    if (phys_size(col) != 8) reject(B2Q_ERR_UNSUPPORTED, "DATE ENCODING FIXED(32) as a GROUP BY key is outside this path");
    *min_out = min_secs;
    *div_day = 1;
  }

  int find_or_add_acc(B2QQuery& q, const DevAcc& a) {
    for (int i = 0; i < q.prog.n_accs; ++i) if (!memcmp(&q.prog.accs[i], &a, sizeof(DevAcc))) return i;
    if (q.prog.n_accs >= B2Q_MAX_ACCS) reject(B2Q_ERR_UNSUPPORTED, "too many aggregates");
    q.prog.accs[q.prog.n_accs] = a;
    return q.prog.n_accs++;
  }

  DevAcc make_acc(B2QQuery& q, int op, const TargetDesc* d) {
    DevAcc a;
    memset(&a, 0, sizeof(a));
    a.op = static_cast<int8_t>(op);
    a.col = -1;
    if (!d || d->arg_col < 0) return a;
    const SqlType at = d->arg_type;
    a.col = launch_col(q, d->arg_col);
    a.width = static_cast<int8_t>(phys_width_code(d->arg_col));
    const int64_t arg_null = phys_int_null(d->arg_col); /* the sentinel as stored in the chunk */
    a.is_fp = at.is_fp();
    if (!d->skip_null) return a;
    if (at.is_fp()) { /* agg_*_double_skip_val: fp compare against NULL_DOUBLE */
      a.skip1_en = 1;
      a.skip1_val = dbl_bits(fp_null(at));
      return a;
    }
    if (d->agg == B2Q_kMIN || d->agg == B2Q_kMAX) { /* null = inlineIntNull(arg_ti) sign-extended */
      a.skip1_en = 1;
      a.skip1_val = arg_null;
      return a;
    }
    /* SUM / AVG / COUNT: convertNullIfAny + cast to the aggregate type + compare with ITS sentinel */
    const SqlType agg_t = d->sql_type;
    if (!at.notnull) { a.skip1_en = 1; a.skip1_val = arg_null; }
    a.skip2_en = 1;
    a.skip2_val = agg_t.int_null();
    a.skip2_trunc32 = (!at.notnull && agg_t.size() == 4) ? 1 : 0;
    return a;
  }

  void lower(B2QQuery& q) {
    B2QPlan& p = q.plan;
    DevProgram& g = q.prog;
    q.bigint_count = eo_.bigint_count;
    if (join_) { /* probe parameters: hash_join_idx[_nullable](buff, key, min, max[, null]) (GroupByRuntime.cpp:283-311) */
      g.join.fk_col = launch_col(q, join_outer_col_);
      g.join.fk_width = static_cast<int8_t>(phys_width_code(join_outer_col_));
      g.join.min_key = p.join_min_key;
      g.join.entry_count = p.join_entry_count;
      g.join.nullable = !col_type(join_outer_col_).notnull;
      g.join.null_val = phys_int_null(join_outer_col_);
      g.join.left = join_left_ ? 1 : 0;
    }
    /* filter: all simple_quals and quals AND-ed */
    int n_quals = 0, max_depth = 0;
    auto add_qual = [&](int idx) {
      max_depth = std::max(max_depth, lower_bool(q, idx, n_quals ? 1 : 0));
      if (n_quals) {
        if (g.filter.n_ops >= B2Q_MAX_FILTER_OPS) reject(B2Q_ERR_UNSUPPORTED, "filter too large");
        g.filter.ops[g.filter.n_ops++] = static_cast<uint8_t>(FOP_AND << 4);
      }
      ++n_quals;
    };
    if (filter_deleted_ && t_.deleted_column_plus1 > 0) {
      /* codegenSkipDeletedOuterTableRow (NativeCodegen.cpp:3419-3451): toBool($deleted$) => row skipped, before any
       * qual.  As a filter term: pass iff the int8 flag is <= 0 (NULL_BOOLEAN = INT8_MIN is "not deleted"). */
      DevFilter& f = g.filter;
      DevTerm t;
      memset(&t, 0, sizeof(t));
      t.col2 = -1;
      t.col = launch_col(q, t_.deleted_column_plus1 - 1);
      t.width = 1;
      t.lo = INT32_MIN;
      t.span = static_cast<uint64_t>(0) - static_cast<uint64_t>(static_cast<int64_t>(INT32_MIN));
      f.ops[f.n_ops++] = static_cast<uint8_t>((FOP_TERM << 4) | f.n_terms);
      f.terms[f.n_terms++] = t;
      term_sel_.push_back(1.0);
      ++n_quals;
      max_depth = std::max(max_depth, 1);
    }
    {
      /* simple_quals and quals are the conjuncts of ONE AND chain (the analyzer split the WHERE clause at its top-level
       * ANDs): leaves on the same column fold across them — `c >= a` and `c <= b` arrive as two quals */
      std::vector<ChainItem> conjuncts;
      for (int i = 0; i < u_.num_simple_quals; ++i) flatten_chain(u_.simple_quals[i], false, true, conjuncts);
      for (int i = 0; i < u_.num_quals; ++i) flatten_chain(u_.quals[i], false, true, conjuncts);
      const int d = conjuncts.size() >= 2 ? lower_chain_items(q, conjuncts, n_quals ? 1 : 0, true) : -1;
      if (d >= 0) {
        max_depth = std::max(max_depth, d);
        if (n_quals) {
          if (g.filter.n_ops >= B2Q_MAX_FILTER_OPS) reject(B2Q_ERR_UNSUPPORTED, "filter too large");
          g.filter.ops[g.filter.n_ops++] = static_cast<uint8_t>(FOP_AND << 4);
        }
        ++n_quals;
      } else {
        for (int i = 0; i < u_.num_simple_quals; ++i) add_qual(u_.simple_quals[i]);
        for (int i = 0; i < u_.num_quals; ++i) add_qual(u_.quals[i]);
      }
    }
    if (max_depth > 4) reject(B2Q_ERR_UNSUPPORTED, "filter expression nests deeper than 4");
    /* load scheduling hints: a 32-byte sector holds 4-8 rows, so predicating a column load on the filter only saves
     * HBM traffic when almost every row fails; otherwise loading eagerly puts all column loads in flight at once */
    g.est_selectivity = static_cast<float>(estimate_selectivity(g.filter));
    g.eager_key = g.est_selectivity >= 0.10f;
    g.eager_args = g.est_selectivity >= 0.25f;

    if (u_.has_estimator) { /* the tuple rides in keys[]; ONE accumulator: the bitmap (see ACC_NDV) */
      g.n_keys = static_cast<int32_t>(estimator_cols_.size());
      for (size_t i = 0; i < estimator_cols_.size(); ++i) {
        const int c = estimator_cols_[i];
        const SqlType kt = col_type(c);
        DevKeyComp& d = g.keys[i];
        d.col = launch_col(q, c);
        d.width = static_cast<int8_t>(phys_width_code(c));
        /* groupByColumnCodegen without NULL translation: a NULL contributes the LOGICAL sentinel, so the chunk's
         * physical sentinel (ENCODING FIXED / DICT(8|16)) is mapped back */
        d.translate_null = !kt.notnull && phys_int_null(c) != kt.int_null();
        d.null_val = phys_int_null(c);
        d.null_logical = kt.int_null();
        g.col_prefetch[d.col] = 1;
      }
      g.key.col = -1;
      g.key.entry_count = 1;
      DevAcc a;
      memset(&a, 0, sizeof(a));
      a.op = ACC_NDV;
      a.col = -1;
      g.accs[0] = a;
      g.n_accs = 1;
      g.fused = 0; g.fused_cnt = -1; g.fused_sum = -1; g.touch_acc = -1; g.touch_piggyback = -1;
      DevLayout& EL = q.layout;
      EL.entry_count = 1;
      EL.n_slots = 0;
      EL.touched_acc = -1;
      EL.touch_via_acc = -1;
      EL.keyless_marker = -1;
      for (int t = 0; t < g.filter.n_terms; ++t) { g.col_prefetch[g.filter.terms[t].col] = 1; if (g.filter.terms[t].col2 >= 0) g.col_prefetch[g.filter.terms[t].col2] = 1; }
      if (join_) g.col_prefetch[g.join.fk_col] = 1;
      g.join.packed_col = -1;
      for (int c = 0; c < g.n_cols; ++c) if (g.col_inner[c]) g.col_prefetch[c] = 0;
      return;
    }

    /* key */
    g.n_keys = static_cast<int32_t>(keycomps_.size());
    for (size_t i = 0; i < keycomps_.size(); ++i) {
      const KeyComp& kc = keycomps_[i];
      const SqlType kt = col_type(kc.col);
      DevKeyComp& d = g.keys[i];
      d.col = launch_col(q, kc.col);
      d.width = static_cast<int8_t>(phys_width_code(kc.col));
      d.min_val = kc.min;
      d.card = static_cast<uint32_t>(kc.card);
      d.mult = static_cast<uint32_t>(kc.mult);
      d.translate_null = kc.has_nulls && !kt.notnull;
      d.null_val = kt.notnull ? kt.int_null() : phys_int_null(kc.col);
      d.null_logical = kt.int_null();
      d.step = kc.bucket ? kc.bucket : 1;
      d.null_stored = kc.max + d.step;
      if (kc.bucket) day_key(kc.col, kc.min, &d.min_val, &d.div_day);
    }
    DevKey& k = g.key;
    k.col = -1;
    k.entry_count = p.entry_count;
    k.hash_magic = p.entry_count > 0 ? ~0ull / static_cast<uint64_t>(p.entry_count) + 1 : 0;
    k.null_idx = -1;
    if (grouped_ && keycomps_.size() <= 1) {
      const SqlType kt = col_type(key_col_);
      k.col = launch_col(q, key_col_);
      k.width = static_cast<int8_t>(phys_width_code(key_col_));
      k.min_val = p.min_val;
      k.null_val = kt.notnull ? kt.int_null() : phys_int_null(key_col_);
      k.null_logical = kt.int_null();
      k.hash_key_width = static_cast<int8_t>(p.effective_key_width);
      if (p.query_desc_type == B2Q_GroupByPerfectHash && p.bucket) day_key(key_col_, p.min_val, &k.min_val, &k.div_day);
      if (p.query_desc_type == B2Q_GroupByPerfectHash && p.has_nulls && !kt.notnull) {
        k.translate_null = 1;
        k.null_idx = (p.max_val - p.min_val) / (p.bucket ? p.bucket : 1) + 1;
      }
    }

    /* accumulators + slot recipes */
    DevLayout& L = q.layout;
    L.row_size = p.row_size;
    L.columnar = p.output_columnar;
    L.key_col_stride = align8(8 * p.entry_count);
    L.entry_count = p.entry_count;
    L.n_slots = p.num_slots;
    /* with a day bucket entry i holds the i-th day on or after min: (key - min) / 86400 == i  <=>  key = first + i * 86400 */
    L.key_step = p.bucket ? p.bucket : 1;
    L.key_min = p.bucket ? ceil_div(p.min_val, p.bucket) * p.bucket : p.min_val;
    L.key_null_stored = p.max_val + L.key_step;
    L.null_idx = k.null_idx;
    L.key_null_val = grouped_ ? col_type(key_col_).int_null() : 0;
    L.has_key_col = grouped_ && !p.keyless_hash;
    L.key_width = static_cast<int8_t>(p.effective_key_width);
    L.baseline = p.query_desc_type == B2Q_GroupByBaselineHash;
    L.touched_acc = -1;
    L.touch_via_acc = -1;
    L.n_keys = g.n_keys;
    for (int i = 0; i < g.n_keys; ++i) {
      L.keys[i] = g.keys[i];
      if (keycomps_[i].bucket) L.keys[i].min_val = ceil_div(keycomps_[i].min, keycomps_[i].bucket) * keycomps_[i].bucket;
    }
    L.keyless_marker = (grouped_ && p.keyless_hash) ? p.idx_target_as_key : -1;
    for (const TargetDesc& d : targets_) {
      const int s = d.first_slot;
      DevSlot& sl = L.slots[s];
      sl.init_val = p.init_vals[s];
      sl.offset = p.slot_offset[s];
      sl.width = p.slot_padded_width[s];
      sl.acc = -1; sl.nn = -1;
      if (sl.width == 0) { sl.kind = SLOT_NONE; continue; }
      if (!d.is_agg) {
        sl.kind = SLOT_KEY;
        sl.key_comp = 0;
        if (keycomps_.size() > 1) {
          int comp = -1;
          for (size_t c = 0; c < keycomps_.size(); ++c) if (keycomps_[c].col == d.arg_col) comp = static_cast<int>(c);
          if (comp < 0) reject(B2Q_ERR_UNSUPPORTED, "non-aggregate target must be a GROUP BY column");
          sl.key_comp = static_cast<int8_t>(comp);
        } else if (d.arg_col != key_col_) {
          reject(B2Q_ERR_UNSUPPORTED, "non-aggregate target must be the GROUP BY column");
        }
        continue;
      }
      if (sl.width == 4 && !(d.agg == B2Q_kCOUNT && d.arg_col < 0)) reject(B2Q_ERR_UNSUPPORTED, "4-byte slot with an aggregate argument");
      const bool fp = d.arg_col >= 0 && d.arg_type.is_fp();
      /* the count of values that survive the skip test: decides NULL for SUM, is AVG's count, is COUNT(c) */
      auto non_null_count = [&]() -> int {
        if (!(d.arg_col >= 0 && d.skip_null)) return -1;
        DevAcc c = make_acc(q, ACC_COUNT, &d);
        if (!c.skip1_en && !c.skip2_en) { c.col = -1; c.width = 0; c.is_fp = 0; } /* nothing to skip: COUNT(*) */
        return find_or_add_acc(q, c);
      };
      switch (d.agg) {
        case B2Q_kCOUNT: {
          if (d.distinct) { /* codegenCountDistinct (GroupByAndAggregate.cpp:1889-1963): agg_count_distinct_bitmap[_skip_val] */
            DevAcc a;
            memset(&a, 0, sizeof(a));
            a.op = ACC_BITMAP;
            a.col = launch_col(q, d.arg_col);
            a.width = static_cast<int8_t>(phys_width_code(d.arg_col));
            if (d.skip_null) { a.skip1_en = 1; a.skip1_val = phys_int_null(d.arg_col); } /* inlineIntNull(arg_ti), as stored */
            a.bm_min = d.cd_min;
            a.bm_bits = d.cd_bits;
            a.bm_words = static_cast<int32_t>(align8((d.cd_bits + 7) / 8) / 4);
            a.bm_bucket = static_cast<int32_t>(d.cd_bucket);
            sl.kind = SLOT_BITCOUNT;
            sl.acc = find_or_add_acc(q, a);
            sl.bm_words = a.bm_words;
            break;
          }
          sl.kind = SLOT_COUNT;
          const int nn = non_null_count();
          sl.acc = nn >= 0 ? nn : find_or_add_acc(q, make_acc(q, ACC_COUNT, nullptr));
          break;
        }
        case B2Q_kSUM:
        case B2Q_kAVG: {
          sl.kind = SLOT_VALUE;
          sl.as_float = d.arg_type.is_float() ? 1 : 0; /* takes_float_argument: a 4-byte float in the slot's low word */
          sl.acc = find_or_add_acc(q, make_acc(q, fp ? ACC_SUM_F64 : ACC_SUM_I64, &d));
          const int nn = non_null_count();
          sl.nn = nn;
          if (d.agg == B2Q_kAVG) {
            DevSlot& cs = L.slots[s + 1];
            cs.init_val = 0; cs.offset = p.slot_offset[s + 1]; cs.width = p.slot_padded_width[s + 1];
            cs.kind = SLOT_COUNT; cs.nn = -1;
            cs.acc = nn >= 0 ? nn : find_or_add_acc(q, make_acc(q, ACC_COUNT, nullptr));
          }
          break;
        }
        case B2Q_kMIN:
        case B2Q_kMAX: {
          const int op = d.agg == B2Q_kMIN ? (fp ? ACC_MIN_F64 : ACC_MIN_I64) : (fp ? ACC_MAX_F64 : ACC_MAX_I64);
          sl.kind = fp ? SLOT_VALUE_ORD : SLOT_VALUE;
          sl.as_float = d.arg_type.is_float() ? 1 : 0;
          sl.acc = find_or_add_acc(q, make_acc(q, op, &d));
          sl.identity = b2q_acc_identity(op);
          sl.scale_day = is_days(d.arg_col) ? 1 : 0;
          /* "no value seen" <=> the accumulator still holds its identity.  Exact except for a nullable BIGINT MIN
           * whose only non-NULL values are INT64_MAX (the identity is a legal value there): that case counts. */
          if (d.skip_null && !fp && d.arg_type.size() == 8 && d.agg == B2Q_kMIN) sl.nn = non_null_count();
          else sl.nn = -2;
          break;
        }
        default: reject(B2Q_ERR_UNSUPPORTED, "aggregate kind");
      }
    }
    if (grouped_ && !p.keyless_hash && !L.baseline) L.touched_acc = find_or_add_acc(q, make_acc(q, ACC_TOUCH, nullptr));
    /* columns worth prefetching: filter columns always; key / arguments when they are loaded eagerly */
    for (int t = 0; t < g.filter.n_terms; ++t) { g.col_prefetch[g.filter.terms[t].col] = 1; if (g.filter.terms[t].col2 >= 0) g.col_prefetch[g.filter.terms[t].col2] = 1; }
    if (grouped_ && g.eager_key) { if (g.n_keys > 1) { for (int i = 0; i < g.n_keys; ++i) g.col_prefetch[g.keys[i].col] = 1; } else g.col_prefetch[g.key.col] = 1; }
    if (g.eager_args)
      for (int a = 0; a < g.n_accs; ++a) if (g.accs[a].col >= 0) g.col_prefetch[g.accs[a].col] = 1;
    if (join_) g.col_prefetch[g.join.fk_col] = 1;
    g.join.packed_col = -1;
    g.join.probe_cg = []() { const char* e = getenv("B2Q_JOIN_CG"); return e && atoi(e) != 0; }() ? 1 : 0;
    if (join_) { /* the first 1/2/4-byte inner column the program reads rides in the join table itself */
      static const bool pack = []() { const char* e = getenv("B2Q_JOIN_PACK"); return !e || atoi(e) != 0; }();
      for (int c = 0; c < g.n_cols && pack; ++c)
        if (g.col_inner[c] && g.col_width[c] <= 4 && !col_type(q.col_ids[c]).is_fp()) {
          g.join.packed_col = static_cast<int8_t>(c);
          g.join.packed_width = static_cast<int8_t>(phys_width_code(q.col_ids[c]));
          break;
        }
    }
    /* value-only 16-bit slots: when the packed column is the ONLY inner column read and its values span < 65534 */
    g.join.slot16 = 0;
    if (join_ && g.join.packed_col >= 0) {
      static const bool s16 = []() { const char* e = getenv("B2Q_JOIN_SLOT16"); return !e || atoi(e) != 0; }();
      int n_inner = 0;
      for (int c = 0; c < g.n_cols; ++c) n_inner += g.col_inner[c] ? 1 : 0;
      ColRange vr = leaf_range(q.col_ids[g.join.packed_col]);
      if (is_days(q.col_ids[g.join.packed_col]) && vr.imin <= vr.imax) { /* the slot holds the chunk's raw days, the stats are seconds */
        vr.imin = floor_div(vr.imin, 86400);
        vr.imax = floor_div(vr.imax, 86400);
      }
      int64_t span = 0;
      if (s16 && n_inner == 1 && vr.valid && !vr.fp && vr.imin <= vr.imax && !__builtin_sub_overflow(vr.imax, vr.imin, &span) && span < 65534) {
        g.join.slot16 = 1;
        g.join.slot16_min = vr.imin;
      }
    }
    for (int c = 0; c < g.n_cols; ++c) if (g.col_inner[c]) g.col_prefetch[c] = 0; /* gathered by join index, not streamed */
    /* fused fast path of the shared-memory-table kernel (the reference's JIT specialises per query; this is the
     * static-kernel equivalent for the most common shape: GROUP BY k with COUNT(*) and/or one integer SUM) */
    g.fused = 0; g.fused_cnt = -1; g.fused_sum = -1;
    {
      bool ok = g.n_accs >= 1 && g.n_accs <= 2;
      for (int a = 0; a < g.n_accs && ok; ++a) {
        const DevAcc& c = g.accs[a];
        if (c.op == ACC_COUNT && c.col < 0 && g.fused_cnt < 0) g.fused_cnt = static_cast<int8_t>(a);
        else if ((c.op == ACC_SUM_I64 || (c.op == ACC_SUM_F64 && c.width == 8)) && !c.skip1_en && !c.skip2_en && g.fused_sum < 0) g.fused_sum = static_cast<int8_t>(a);
        else ok = false;
      }
      g.fused = ok ? 1 : 0;
    }
    g.touch_acc = static_cast<int8_t>(L.touched_acc);
    g.touch_piggyback = -1;
    if (L.touched_acc >= 0)
      for (int want : {ACC_COUNT, ACC_SUM_I64}) { /* a COUNT first: it is non-zero for every touched group whatever the values */
        for (int a = 0; a < g.n_accs && g.touch_piggyback < 0; ++a) {
          const DevAcc& c = g.accs[a];
          if (c.op == want && !c.skip1_en && !c.skip2_en) g.touch_piggyback = static_cast<int8_t>(a);
        }
      }
    /* materialise: an entry is touched when its flag is set OR this accumulator is non-zero (the HBM-table kernels with plain
     * 8-byte words only flag the rows whose value could leave the sum at zero: see global_split_add_touch) */
    L.touch_via_acc = g.touch_piggyback;
  }

  void choose_kernel(B2QQuery& q) {
    B2QPlan& p = q.plan;
    SmemPlan& sm = q.smem;
    memset(&sm, 0, sizeof(sm));
    sm.replicas = 1;
    /* shared-memory footprint per entry: COUNT 4 B, SUM_I64 4 B (low word; carries go to HBM), others 8 B;
     * 8-byte arrays first so they stay 8-byte aligned */
    int off = 0;
    for (int pass = 0; pass < 2; ++pass)
      for (int a = 0; a < q.prog.n_accs; ++a) {
        const int op = q.prog.accs[a].op;
        const int bytes = op == ACC_BITMAP ? 0 /* bitmaps stay in HBM */ : op == ACC_TOUCH ? 1 : (op == ACC_COUNT || op == ACC_SUM_I64) ? 4 : 8;
        if ((pass == 0) != (bytes == 8)) continue;
        sm.acc_bytes[a] = bytes;
        sm.acc_off[a] = off;
        const int64_t arr = ((p.entry_count * bytes + 15) / 16) * 16;
        off = static_cast<int>(std::min<int64_t>(int64_t(off) + arr, int64_t(1) << 30));
      }
    const int64_t per_replica = off;
    const int64_t budget = 200 * 1024; /* of the 227 KB a CTA may opt in to */
    auto use_smem_table = [&]() {
      sm.use_smem = 1;
      sm.replica_bytes = static_cast<int32_t>(per_replica);
      int rep = 1;
      /* the join kernels gather from the join table through L1/L2: shared memory left to the group-table replicas is L1
       * taken from those gathers (B2Q_JOIN_SMEM_KB: experiment knob, default = the plain kernels' 96 KB) */
      static const int64_t join_cap_kb = []() { const char* e = getenv("B2Q_JOIN_SMEM_KB"); return e ? atoll(e) : int64_t(96); }();
      const int64_t cap = (join_ ? join_cap_kb : 96) * 1024;
      while (rep < 32 && int64_t(rep) * 2 * per_replica <= cap) rep *= 2; /* warp-private copies for small tables */
      sm.replicas = rep;
      sm.total_bytes = static_cast<int32_t>(per_replica * rep);
    };
    int kernel;
    if (p.query_desc_type == B2Q_NonGroupedAggregate || p.query_desc_type == B2Q_Estimator) {
      kernel = B2Q_KERNEL_NON_GROUPED;
      use_smem_table();
    } else if (p.query_desc_type == B2Q_GroupByBaselineHash) {
      kernel = B2Q_KERNEL_BASELINE_GLOBAL;
    } else if (per_replica <= budget && p.entry_count <= (1 << 22)) {
      kernel = B2Q_KERNEL_PERFECT_SMEM;
      use_smem_table();
    } else {
      kernel = B2Q_KERNEL_PERFECT_GLOBAL;
    }
    if (eo_.force_kernel) {
      int f = eo_.force_kernel;
      if (f == B2Q_KERNEL_BASELINE_PROBE && kernel == B2Q_KERNEL_BASELINE_GLOBAL) f = kernel; /* the executor reads the option: per-row probe instead of the radix passes */
      const bool ok = (f == kernel) || (f == B2Q_KERNEL_PERFECT_GLOBAL && kernel == B2Q_KERNEL_PERFECT_SMEM);
      if (!ok) reject(B2Q_ERR_INVALID_ARGUMENT, "force_kernel is not applicable to this query");
      if (f == B2Q_KERNEL_PERFECT_GLOBAL) { sm.use_smem = 0; sm.replicas = 1; sm.total_bytes = 0; }
      kernel = f;
    }
    p.kernel = kernel;
    /* a dimension-sized join table rides in shared memory (TMA-staged once per CTA) when it fits beside the group
     * table; replicas give way first (they only relieve same-address serialisation) */
    sm.join_off = -1;
    sm.join_bytes = 0;
    static const bool stage = []() { const char* e = getenv("B2Q_JOIN_SMEM"); return !e || atoi(e) != 0; }();
    if (join_ && stage && p.join_entry_count > 0) {
      const int64_t room = 216 * 1024; /* of the 227 KB a CTA may opt in to */
      auto try_stage = [&](int64_t slot_bytes) -> bool {
        const int64_t jb = ((p.join_entry_count * slot_bytes + 15) / 16) * 16;
        int rep = sm.replicas;
        if (sm.use_smem) while (rep > 1 && int64_t(sm.replica_bytes) * rep + jb + 128 > room) rep /= 2;
        const int64_t base = sm.use_smem ? int64_t(sm.replica_bytes) * rep : 0;
        const int64_t off = ((base + 127) / 128) * 128;
        if (off + jb > room) return false;
        if (sm.use_smem) sm.replicas = rep;
        sm.join_off = static_cast<int32_t>(off);
        sm.join_bytes = static_cast<int32_t>(jb);
        sm.total_bytes = static_cast<int32_t>(off + jb);
        return true;
      };
      /* measured (c2join / c2joins, 1e9 rows): a table that fits with its 8-byte slots is a little faster that way
       * (4.02 vs 4.18 ms); the 16-bit slots are what lets a 1e5-row dimension fit at all (4.42 vs 5.60 ms from L2) */
      bool staged = try_stage(q.prog.join.packed_col >= 0 ? 8 : 4);
      if (staged) q.prog.join.slot16 = 0;
      else if (q.prog.join.slot16) staged = try_stage(2);
      if (!staged) q.prog.join.slot16 = 0; /* 16-bit slots exist only in shared memory */
    } else {
      q.prog.join.slot16 = 0;
    }
  }
};

}  // namespace

/* One INNER hash-join level: the unit is re-expressed over a combined table — columns [0, n_outer) of the scanned
 * table followed by the inner table's — so that ranges, layouts and the device program are planned by the same code;
 * every combined fragment carries the inner table's chunk stats for the inner columns. */
struct JoinedInput {
  std::vector<B2QExpr> exprs;
  B2QExecUnit u{};
  std::vector<B2QTypeInfo> col_types;
  std::vector<int8_t> enc;
  std::vector<std::vector<const void*>> bufs;
  std::vector<std::vector<B2QChunkStats>> stats;
  std::vector<B2QFragmentInfo> frags;
  B2QTableInfo t{};
  int n_outer = 0, outer_col = -1, inner_col = -1;
  bool left = false;
};

static void build_joined_input(const B2QExecUnit& u, const B2QTableInfo& outer, JoinedInput& ji) {
  auto bad = [](int32_t code, const char* m) { throw PlanError{code, m}; };
  if (u.num_join_quals != 1) bad(B2Q_ERR_UNSUPPORTED, "more than one join level is outside this path");
  if (u.join_type != 0 && u.join_type != 1) bad(B2Q_ERR_UNSUPPORTED, "only INNER and LEFT joins are on this path");
  const bool left = u.join_type == 1;
  if (!u.inner_table) bad(B2Q_ERR_INVALID_ARGUMENT, "join without an inner table");
  const B2QTableInfo& inner = *u.inner_table;
  if (inner.num_fragments > 1) bad(B2Q_ERR_INVALID_ARGUMENT, "the inner table must come as one concatenated fragment (ColumnFetcher::getAllTableColumnFragments)");
  if (inner.deleted_column_plus1) bad(B2Q_ERR_UNSUPPORTED, "inner table with a deleted-rows column");
  if (inner.num_cols <= 0 || outer.num_cols <= 0) bad(B2Q_ERR_INVALID_ARGUMENT, "table without columns");
  /* the same checks Planner::validate() makes on the outer table, before anything of the inner one is read */
  if (!inner.col_types || !outer.col_types) bad(B2Q_ERR_INVALID_ARGUMENT, "col_types is null");
  if (inner.num_fragments < 0 || (inner.num_fragments && !inner.fragments)) bad(B2Q_ERR_INVALID_ARGUMENT, "inner table: fragments");
  if (inner.num_fragments) {
    const B2QFragmentInfo& f0 = inner.fragments[0];
    if (f0.num_tuples < 0) bad(B2Q_ERR_INVALID_ARGUMENT, "inner table: negative row count");
    if (!f0.col_stats) bad(B2Q_ERR_INVALID_ARGUMENT, "inner table: fragment without chunk stats");
    if (f0.num_tuples > 0 && !f0.col_buffers) bad(B2Q_ERR_INVALID_ARGUMENT, "inner table: fragment without column buffers");
  }
  if (outer.num_fragments < 0 || (outer.num_fragments && !outer.fragments)) bad(B2Q_ERR_INVALID_ARGUMENT, "fragments");
  for (int f = 0; f < outer.num_fragments; ++f)
    if (!outer.fragments[f].col_stats) bad(B2Q_ERR_INVALID_ARGUMENT, "fragment without chunk stats");
  ji.n_outer = outer.num_cols;
  ji.exprs.assign(u.exprs, u.exprs + std::max(u.num_exprs, 0));
  for (B2QExpr& e : ji.exprs) {
    if (e.kind != B2Q_EXPR_COLUMN_VAR) continue;
    if (e.rte_idx == 1) {
      if (e.col_id < 0 || e.col_id >= inner.num_cols) bad(B2Q_ERR_INVALID_ARGUMENT, "inner column id out of range");
      if (left && e.ti.notnull) bad(B2Q_ERR_INVALID_ARGUMENT, "LEFT join: inner ColumnVars must be nullable");
      e.col_id += ji.n_outer;
      e.rte_idx = 0;
    } else if (e.rte_idx != 0) bad(B2Q_ERR_UNSUPPORTED, "rte_idx beyond one join level");
  }
  ji.u = u;
  ji.u.exprs = ji.exprs.data();
  ji.u.num_join_quals = 0;
  ji.u.inner_table = nullptr;
  if (u.join_qual < 0 || u.join_qual >= u.num_exprs) bad(B2Q_ERR_INVALID_ARGUMENT, "join qual index out of range");
  const B2QExpr& q = ji.exprs[u.join_qual];
  if (q.kind != B2Q_EXPR_BIN_OPER || q.op != B2Q_kEQ) bad(B2Q_ERR_UNSUPPORTED, "join qual must be an equality");
  if (q.left < 0 || q.left >= u.num_exprs || q.right < 0 || q.right >= u.num_exprs) bad(B2Q_ERR_INVALID_ARGUMENT, "join qual operand out of range");
  const B2QExpr& a = ji.exprs[q.left];
  const B2QExpr& b = ji.exprs[q.right];
  if (a.kind != B2Q_EXPR_COLUMN_VAR || b.kind != B2Q_EXPR_COLUMN_VAR) bad(B2Q_ERR_UNSUPPORTED, "join qual must compare two ColumnVars");
  const bool a_inner = a.col_id >= ji.n_outer, b_inner = b.col_id >= ji.n_outer;
  if (a_inner == b_inner) bad(B2Q_ERR_UNSUPPORTED, "join qual must compare an outer with an inner column");
  ji.outer_col = a_inner ? b.col_id : a.col_id;
  ji.inner_col = (a_inner ? a.col_id : b.col_id) - ji.n_outer;
  if (ji.outer_col < 0 || ji.outer_col >= ji.n_outer) bad(B2Q_ERR_INVALID_ARGUMENT, "outer join column out of range");
  ji.col_types.assign(outer.col_types, outer.col_types + outer.num_cols);
  ji.col_types.insert(ji.col_types.end(), inner.col_types, inner.col_types + inner.num_cols);
  if (left) for (int c = 0; c < inner.num_cols; ++c) ji.col_types[ji.n_outer + c].notnull = 0; /* codegenOuterJoinNullPlaceholder */
  ji.left = left;
  ji.enc.assign(ji.col_types.size(), 0);
  for (int c = 0; c < outer.num_cols; ++c) if (outer.col_encoded_sizes) ji.enc[c] = outer.col_encoded_sizes[c];
  for (int c = 0; c < inner.num_cols; ++c) if (inner.col_encoded_sizes) ji.enc[ji.n_outer + c] = inner.col_encoded_sizes[c];
  const B2QFragmentInfo* inf = inner.num_fragments ? &inner.fragments[0] : nullptr;
  const int nf = std::max(outer.num_fragments, 0);
  ji.bufs.resize(nf);
  ji.stats.resize(nf);
  ji.frags.resize(nf);
  for (int f = 0; f < nf; ++f) {
    const B2QFragmentInfo& of = outer.fragments[f];
    if (of.col_buffers) ji.bufs[f].assign(of.col_buffers, of.col_buffers + outer.num_cols);
    else ji.bufs[f].assign(static_cast<size_t>(outer.num_cols), nullptr); /* another device's fragment: chunk stats only */
    ji.stats[f].assign(of.col_stats, of.col_stats + outer.num_cols);
    for (int c = 0; c < inner.num_cols; ++c) {
      ji.bufs[f].push_back(nullptr); /* inner columns are resolved by the executor, not through the fragment */
      B2QChunkStats empty{};
      empty.int_min = INT64_MAX; empty.int_max = INT64_MIN; empty.fp_min = DBL_MAX; empty.fp_max = -DBL_MAX;
      ji.stats[f].push_back(inf ? inf->col_stats[c] : empty);
      if (left) ji.stats[f].back().has_nulls = 1; /* is_outer_join_proj (ExpressionRange.cpp:521-525, :642-652) */
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

int32_t make_query(const B2QExecUnit* u, const B2QTableInfo* t, const B2QExecutionOptions* eo, size_t guess,
                   bool has_card, bool filter_deleted, B2QQuery* out, std::string* err) {
  try {
    if (!u || !t || !eo || !out) throw PlanError{B2Q_ERR_INVALID_ARGUMENT, "null argument"};
    if (!u->num_join_quals) {
      Planner(*u, *t, *eo, guess, has_card, filter_deleted).run(*out);
      out->n_outer_cols = t->num_cols;
      out->join_inner_key_col = -1;
      out->plan.join_outer_col = out->plan.join_inner_col = -1;
      out->prog.join.fk_col = -1;
      return B2Q_OK;
    }
    JoinedInput ji;
    build_joined_input(*u, *t, ji);
    Planner pl(ji.u, ji.t, *eo, guess, has_card, filter_deleted);
    pl.set_join(ji.n_outer, ji.outer_col, ji.inner_col, *u->inner_table, ji.left);
    pl.run(*out);
    out->n_outer_cols = ji.n_outer;
    out->join_inner_key_col = ji.inner_col;
    return B2Q_OK;
  } catch (const PlanError& e) {
    if (err) *err = e.msg;
    return e.code;
  }
}

}  // namespace b2q
