// Host side of the drop-in: constraint / analyzer constructors (same validation as the reference's
// constructors), partial-state merge, and finalize = the O(1) Rust that follows `collect()` in every
// reference evaluate(): ratio / assertion / status / message, restated with identical format strings.
#include "plan.hpp"

#include <algorithm>
#include <cmath>
#include <map>
#include <unordered_map>
#include <set>

namespace tg {

int Plan::add_agg(Agg a) {
    for (size_t i = 0; i < aggs.size(); ++i)
        if (aggs[i].key == a.key) {
            if (a.kind == A_NUM || a.kind == A_DISTINCT) aggs[i].flags |= a.flags;  // union of what the slots need
            return (int)i;
        }
    aggs.push_back(std::move(a));
    return (int)aggs.size() - 1;
}

void Plan::reset_partials() {
    for (auto& a : aggs) a.reset_state();
}

// ---- aggregate constructors ----
static Agg mk_rows() {
    Agg a;
    a.kind = A_ROWS;
    a.key = "rows";
    return a;
}
static Agg mk_valid(const std::string& c) {
    Agg a;
    a.kind = A_VALID;
    a.key = "valid|" + c;
    a.cols = {c};
    return a;
}
// NUM aggregate flags (scan_defs.h UF_*): 1 moments (mean/sum/stddev/variance), 2 min/max, 4 wrapping i64 sum
static int stat_flags(int stat) {
    switch (stat) {
        case TG_STAT_MIN: case TG_STAT_MAX: return 2;
        case TG_STAT_MEAN: case TG_STAT_STDDEV: case TG_STAT_VARIANCE: return 1;
        case TG_STAT_SUM: return 1 | 4;
        default: return 2;  // median / percentile: min and max come with the sketch
    }
}
static Agg mk_num(const std::string& c, int flags) {
    Agg a;
    a.kind = A_NUM;
    a.key = "num|" + c;
    a.cols = {c};
    a.flags = flags;
    return a;
}
static Agg mk_pair(const std::string& x, const std::string& y) {
    Agg a;
    a.kind = A_PAIR;
    a.key = "pair|" + x + "|" + y;
    a.cols = {x, y};
    return a;
}
static Agg mk_spearman(const std::string& x, const std::string& y) {
    Agg a;
    a.kind = A_SPEARMAN;
    a.key = "spearman|" + x + "|" + y;
    a.cols = {x, y};
    return a;
}
static Agg mk_pred(const std::string& expr) {
    Agg a;
    a.kind = A_PRED;
    a.key = "pred|" + expr;
    a.text = expr;
    try {
        a.expr = parse_sql_expr(expr);
    } catch (Error& e) {
        a.expr = nullptr;  // reported at evaluation like a DataFusion planning error
        a.ctor_err = e.code;
        a.ctor_err_msg = e.msg;
        a.err = e.code;
        a.err_msg = e.msg;
    }
    return a;
}
static Agg mk_regex(const std::string& c, const std::string& pattern, bool icase, bool trim) {
    Agg a;
    a.kind = A_REGEX;
    a.flags = (icase ? 1 : 0) | (trim ? 2 : 0);
    a.key = "regex|" + c + "|" + std::to_string(a.flags) + "|" + pattern;
    a.cols = {c};
    a.text = pattern;
    return a;
}
// flags bit 0: some slot needs the singleton-group count (u2: GROUP BY .. HAVING COUNT(*) = 1); without it the
// dense path can count with non-returning atomics
static Agg mk_distinct(const std::vector<std::string>& cols, bool need_singles = false) {
    Agg a;
    a.kind = A_DISTINCT;
    a.flags = need_singles ? 1 : 0;
    a.key = "distinct";
    for (auto& c : cols) a.key += "|" + c;
    a.cols = cols;
    return a;
}
static Agg mk_kll(const std::string& c, int k) {
    Agg a;
    a.kind = A_KLL;
    a.key = "kll|" + c + "|" + std::to_string(k);
    a.cols = {c};
    a.iparam = k;
    return a;
}

static void check_threshold_security(double t) {
    if (!(t >= 0.0 && t <= 1.0)) throw Error(TG_ERR_SECURITY, "Threshold must be between 0.0 and 1.0");
}

// ---- slot constructors ----

// constraints/completeness.rs:96-110 (panics on bad threshold; we return an error)
int plan_add_completeness(Plan& p, const std::vector<std::string>& cols, double threshold, int op, int op_n) {
    if (!(threshold >= 0.0 && threshold <= 1.0))
        throw Error(TG_ERR_VALIDATION, "Threshold must be between 0.0 and 1.0");
    Slot s;
    s.kind = SL_COMPLETENESS;
    s.name = "completeness";
    s.columns = cols;
    s.threshold = threshold;
    s.op = op;
    s.op_n = op_n;
    for (auto& c : cols) s.aggs.push_back(p.add_agg(mk_valid(c)));
    p.slots.push_back(std::move(s));
    return (int)p.slots.size() - 1;
}

int plan_add_size(Plan& p, tg_assertion a) {
    Slot s;
    s.kind = SL_SIZE;
    s.name = "size";
    s.assertion = a;
    s.aggs.push_back(p.add_agg(mk_rows()));
    p.slots.push_back(std::move(s));
    return (int)p.slots.size() - 1;
}

static const char* stat_name(int kind, double pct) {  // statistics.rs:70-87
    switch (kind) {
        case TG_STAT_MIN: return "minimum";
        case TG_STAT_MAX: return "maximum";
        case TG_STAT_MEAN: return "mean";
        case TG_STAT_SUM: return "sum";
        case TG_STAT_STDDEV: return "standard deviation";
        case TG_STAT_VARIANCE: return "variance";
        case TG_STAT_MEDIAN: return "median";
        case TG_STAT_PERCENTILE: return std::fabs(pct - 0.5) < 2.220446049250313e-16 ? "median" : "percentile";
    }
    return "?";
}
static const char* stat_constraint_name(int kind) {  // statistics.rs:89-101
    switch (kind) {
        case TG_STAT_MIN: return "min";
        case TG_STAT_MAX: return "max";
        case TG_STAT_MEAN: return "mean";
        case TG_STAT_SUM: return "sum";
        case TG_STAT_STDDEV: return "standard_deviation";
        case TG_STAT_VARIANCE: return "variance";
        case TG_STAT_MEDIAN: return "median";
        case TG_STAT_PERCENTILE: return "percentile";
    }
    return "?";
}

constexpr int KLL_K_FOR_PERCENTILE = 512;

// constraints/statistics.rs:140-170 (new: validate identifier, percentile range)
int plan_add_statistic(Plan& p, const std::string& col, int stat, double pct, tg_assertion a) {
    validate_identifier(col);
    if (stat == TG_STAT_PERCENTILE && !(pct >= 0.0 && pct <= 1.0))
        throw Error(TG_ERR_SECURITY, "Percentile must be between 0.0 and 1.0");
    if (stat < TG_STAT_MIN || stat > TG_STAT_PERCENTILE) throw Error(TG_ERR_INVALID_ARG, "unknown statistic kind");
    Slot s;
    s.kind = SL_STAT;
    s.name = stat_constraint_name(stat);
    s.columns = {col};
    StatReq r{stat, stat == TG_STAT_MEDIAN ? 0.5 : pct, a, -1};
    s.aggs.push_back(p.add_agg(mk_num(col, stat_flags(stat))));
    if (stat == TG_STAT_MEDIAN || stat == TG_STAT_PERCENTILE) r.agg_kll = p.add_agg(mk_kll(col, KLL_K_FOR_PERCENTILE));
    s.stats.push_back(r);
    p.slots.push_back(std::move(s));
    return (int)p.slots.size() - 1;
}

int plan_add_multi_statistic(Plan& p, const std::string& col, const std::vector<StatReq>& stats) {
    validate_identifier(col);
    Slot s;
    s.kind = SL_MULTISTAT;
    s.name = "multi_statistical";
    s.columns = {col};
    int fl = 0;
    for (auto& r : stats) fl |= stat_flags(r.kind);
    s.aggs.push_back(p.add_agg(mk_num(col, fl)));
    for (auto r : stats) {
        if (r.kind == TG_STAT_PERCENTILE && !(r.percentile >= 0.0 && r.percentile <= 1.0))
            throw Error(TG_ERR_SECURITY, "Percentile must be between 0.0 and 1.0");
        if (r.kind == TG_STAT_MEDIAN) r.percentile = 0.5;
        if (r.kind == TG_STAT_MEDIAN || r.kind == TG_STAT_PERCENTILE)
            r.agg_kll = p.add_agg(mk_kll(col, KLL_K_FOR_PERCENTILE));
        s.stats.push_back(r);
    }
    p.slots.push_back(std::move(s));
    return (int)p.slots.size() - 1;
}

void regex_check_supported(const std::string& pattern, bool icase);  // regex_dfa.cpp (throws)

// constraints/format.rs:490-520
int plan_add_format(Plan& p, const std::string& col, int kind, const char* arg, int flag, double threshold,
                    tg_format_options opt) {
    validate_identifier(col);
    check_threshold_security(threshold);
    std::string pattern = format_pattern(kind, arg, flag);
    validate_regex_pattern_text(pattern);
    regex_check_supported(pattern, !opt.case_sensitive);  // Regex::new must succeed (security.rs:166-173)
    Slot s;
    s.kind = SL_FORMAT;
    s.name = format_name(kind);
    s.columns = {col};
    s.sub_kind = kind;
    s.has_arg = arg != nullptr;
    s.arg = arg ? arg : "";
    s.flag = flag;
    s.threshold = threshold;
    s.fopt = opt;
    s.pattern = pattern;
    s.aggs.push_back(p.add_agg(mk_regex(col, pattern, !opt.case_sensitive, opt.trim_before_check != 0)));
    p.slots.push_back(std::move(s));
    return (int)p.slots.size() - 1;
}

static const char* uniq_name(int kind) {
    switch (kind) {
        case TG_UNIQ_FULL: return "full_uniqueness";
        case TG_UNIQ_DISTINCTNESS: return "distinctness";
        case TG_UNIQ_UNIQUE_VALUE_RATIO: return "unique_value_ratio";
        case TG_UNIQ_PRIMARY_KEY: return "primary_key";
        case TG_UNIQ_WITH_NULLS: return "unique_with_nulls";
        case TG_UNIQ_COMPOSITE: return "unique_composite";
    }
    return "?";
}

// constraints/uniqueness.rs:262-308
int plan_add_uniqueness(Plan& p, const std::vector<std::string>& cols, int kind, double threshold,
                        tg_assertion a, int null_handling) {
    if (cols.empty())
        throw Error(TG_ERR_VALIDATION, "Validation failed for constraint 'unified_uniqueness': At least one column must be specified");
    for (auto& c : cols) validate_identifier(c);
    if (kind == TG_UNIQ_FULL || kind == TG_UNIQ_WITH_NULLS || kind == TG_UNIQ_COMPOSITE) {
        if (!(threshold >= 0.0 && threshold <= 1.0))
            throw Error(TG_ERR_VALIDATION, "Validation failed for constraint 'unified_uniqueness': Threshold must be between 0.0 and 1.0");
    }
    if (kind < TG_UNIQ_FULL || kind > TG_UNIQ_COMPOSITE) throw Error(TG_ERR_INVALID_ARG, "unknown uniqueness kind");
    Slot s;
    s.kind = SL_UNIQ;
    s.name = uniq_name(kind);
    s.columns = cols;
    s.sub_kind = kind;
    s.threshold = threshold;
    s.assertion = a;
    s.null_handling = null_handling;
    s.aggs.push_back(p.add_agg(mk_distinct(cols, kind == TG_UNIQ_UNIQUE_VALUE_RATIO)));
    p.slots.push_back(std::move(s));
    return (int)p.slots.size() - 1;
}

// constraints/correlation.rs:140-260
int plan_add_correlation(Plan& p, const std::string& c1, const std::string& c2, int kind, tg_assertion a) {
    validate_identifier(c1);
    validate_identifier(c2);
    Slot s;
    s.kind = SL_CORR;
    s.columns = {c1, c2};
    s.sub_kind = kind;
    s.assertion = a;
    switch (kind) {
        case TG_CORR_PEARSON: s.name = "correlation"; break;
        case TG_CORR_COVARIANCE: s.name = "covariance"; break;
        case TG_CORR_INDEPENDENCE:
            if (!(a.a >= 0.0 && a.a <= 1.0))
                throw Error(TG_ERR_CONFIGURATION, "Max correlation must be between 0.0 and 1.0");
            s.name = "independence";
            break;
        case TG_CORR_SPEARMAN: s.name = "spearman_correlation"; break;
        case TG_CORR_KENDALL: s.name = "kendall_correlation"; break;
        case TG_CORR_MUTUAL_INFORMATION: s.name = "mutual_information"; break;
        case TG_CORR_RANGE:
            if (a.a > a.b) throw Error(TG_ERR_CONFIGURATION, "Invalid correlation range: min must be <= max");
            s.name = "correlation_range";
            s.assertion.kind = TG_ASSERT_BETWEEN;
            break;
        default: throw Error(TG_ERR_INVALID_ARG, "unknown correlation kind");
    }
    if (kind == TG_CORR_PEARSON || kind == TG_CORR_COVARIANCE || kind == TG_CORR_INDEPENDENCE || kind == TG_CORR_RANGE)
        s.aggs.push_back(p.add_agg(mk_pair(c1, c2)));
    p.slots.push_back(std::move(s));
    return (int)p.slots.size() - 1;
}

// constraints/custom_sql.rs:60-98
int plan_add_custom_sql(Plan& p, const std::string& expr, const char* hint) {
    validate_sql_expression(expr);
    Slot s;
    s.kind = SL_SQL;
    s.name = "custom_sql";
    s.arg = expr;
    s.has_hint = hint != nullptr;
    s.hint = hint ? hint : "";
    s.aggs.push_back(p.add_agg(mk_pred(expr)));
    p.slots.push_back(std::move(s));
    return (int)p.slots.size() - 1;
}

// constraints/foreign_key.rs:66-149
int plan_add_foreign_key(Plan& p, const std::string& child, const std::string& parent, int allow_nulls,
                         int max_examples) {
    Slot s;
    s.kind = SL_FK;
    s.name = "foreign_key";
    s.columns = {child, parent};
    s.allow_nulls = allow_nulls;
    s.max_examples = max_examples;
    Agg a;
    a.kind = A_FK;
    a.key = "fk|" + child + "|" + parent + "|" + std::to_string(allow_nulls) + "|" + std::to_string(max_examples);
    a.flags = allow_nulls;
    a.iparam = max_examples;
    // parse_qualified_column: exactly one dot; both parts validated
    auto split = [](const std::string& q, std::string& t, std::string& c) {
        size_t d = q.find('.');
        if (d == std::string::npos || q.find('.', d + 1) != std::string::npos) return false;
        t = q.substr(0, d);
        c = q.substr(d + 1);
        return true;
    };
    std::string ct, cc, pt, pc;
    if (!split(child, ct, cc)) {
        a.err = TG_ERR_VALIDATION;
        a.err_msg = "Constraint evaluation failed for 'foreign_key': Foreign key column must be qualified (table.column): '" + child + "'";
    } else if (!split(parent, pt, pc)) {
        a.err = TG_ERR_VALIDATION;
        a.err_msg = "Constraint evaluation failed for 'foreign_key': Foreign key column must be qualified (table.column): '" + parent + "'";
    } else {
        try {
            validate_identifier(ct);
            validate_identifier(cc);
            validate_identifier(pt);
            validate_identifier(pc);
        } catch (Error& e) {
            a.err = e.code;
            a.err_msg = "Security error: " + e.msg;
        }
        a.cols = {ct, cc, pt, pc};
    }
    a.ctor_err = a.err;
    a.ctor_err_msg = a.err_msg;
    s.aggs.push_back(p.add_agg(std::move(a)));
    p.slots.push_back(std::move(s));
    return (int)p.slots.size() - 1;
}

int plan_add_analyzer(Plan& p, int kind, const char* col, const char* col2, const char* expr) {
    Slot s;
    s.kind = SL_ANALYZER;
    s.sub_kind = kind;
    std::string c = col ? col : "", c2 = col2 ? col2 : "";
    auto need_col = [&]() {
        if (!col) throw Error(TG_ERR_INVALID_ARG, "analyzer requires a column");
    };
    switch (kind) {
        case TG_AN_SIZE:
            s.name = "size";
            s.metric_key = "size";
            s.aggs.push_back(p.add_agg(mk_rows()));
            break;
        case TG_AN_COMPLETENESS:
            need_col();
            s.name = "completeness";
            s.metric_key = "completeness." + c;
            s.columns = {c};
            s.aggs.push_back(p.add_agg(mk_valid(c)));
            break;
        case TG_AN_DISTINCTNESS:
            need_col();
            s.name = "distinctness";
            s.metric_key = "distinctness." + c;
            s.columns = {c};
            s.aggs.push_back(p.add_agg(mk_distinct({c})));
            break;
        case TG_AN_APPROX_COUNT_DISTINCT:  // analyzers/advanced/approx_count_distinct.rs:100-176
            need_col();
            s.name = "approx_count_distinct";
            s.metric_key = "approx_count_distinct." + c;
            s.columns = {c};
            s.aggs.push_back(p.add_agg(mk_distinct({c})));
            break;
        case TG_AN_MEAN:
        case TG_AN_MIN:
        case TG_AN_MAX:
        case TG_AN_SUM:
        case TG_AN_STDDEV: {
            need_col();
            const char* nm = kind == TG_AN_MEAN ? "mean" : kind == TG_AN_MIN ? "min" : kind == TG_AN_MAX ? "max"
                           : kind == TG_AN_SUM ? "sum" : "standard_deviation";
            s.name = nm;
            // StandardDeviationAnalyzer has no metric_key override (SURVEY appendix C)
            s.metric_key = kind == TG_AN_STDDEV ? std::string(nm) : std::string(nm) + "." + c;
            s.columns = {c};
            s.aggs.push_back(p.add_agg(mk_num(c, kind == TG_AN_MIN || kind == TG_AN_MAX ? 2 : kind == TG_AN_STDDEV ? 1 : (1 | 4))));
        } break;
        case TG_AN_CORR_PEARSON:
        case TG_AN_COVARIANCE:
        case TG_AN_CORR_SPEARMAN: {
            if (!col || !col2) throw Error(TG_ERR_INVALID_ARG, "correlation analyzer requires two columns");
            validate_identifier(c);
            validate_identifier(c2);
            s.name = "correlation";
            const char* t = kind == TG_AN_CORR_PEARSON ? "pearson" : kind == TG_AN_COVARIANCE ? "covariance" : "spearman";
            s.metric_key = std::string("correlation_") + t + "_" + c + "_" + c2;
            s.columns = {c, c2};
            s.aggs.push_back(p.add_agg(kind == TG_AN_CORR_SPEARMAN ? mk_spearman(c, c2) : mk_pair(c, c2)));
        } break;
        case TG_AN_COMPLIANCE: {
            if (!expr) throw Error(TG_ERR_INVALID_ARG, "compliance analyzer requires a predicate");
            s.name = "compliance";
            s.metric_key = "compliance";
            s.arg = expr;
            // ComplianceAnalyzer wraps the predicate in parentheses (compliance.rs:153-159)
            s.aggs.push_back(p.add_agg(mk_pred(expr)));
        } break;
        default: throw Error(TG_ERR_INVALID_ARG, "unknown analyzer kind (use tg_plan_add_kll / _grouped_completeness)");
    }
    p.slots.push_back(std::move(s));
    return (int)p.slots.size() - 1;
}

int plan_add_kll(Plan& p, const std::string& col, int k, const std::vector<double>& q) {
    if (k < 2) throw Error(TG_ERR_INVALID_ARG, "k must be at least 2");
    for (double x : q)
        if (!(x >= 0.0 && x <= 1.0)) throw Error(TG_ERR_INVALID_ARG, "Quantile phi must be in [0, 1]");
    Slot s;
    s.kind = SL_KLL;
    s.name = "kll_sketch";
    s.metric_key = "kll_sketch";
    s.columns = {col};
    s.k = k;
    s.quantiles = q;
    s.aggs.push_back(p.add_agg(mk_kll(col, k)));
    p.slots.push_back(std::move(s));
    return (int)p.slots.size() - 1;
}

// constraints/length.rs:20-60 (LengthAssertion), :150-226 (evaluate). kind: 0 Min(a) 1 Max(a) 2 Between(a, b)
// 3 Exactly(a) 4 NotEmpty
int plan_add_length(Plan& p, const std::string& col, int kind, int64_t a, int64_t b) {
    validate_identifier(col);
    if (kind < 0 || kind > 4 || a < 0 || b < 0) throw Error(TG_ERR_INVALID_ARG, "invalid length assertion");
    if (kind == 2 && a > b) throw Error(TG_ERR_INVALID_ARG, "min_length must be <= max_length");  // length.rs:136 assert!
    Slot s;
    s.kind = SL_LENGTH;
    s.columns = {col};
    s.sub_kind = kind;
    const std::string A = std::to_string(a), B = std::to_string(b);
    int64_t lo = 0, hi = INT64_MAX;
    switch (kind) {
        case 0: s.name = "min_length"; s.arg = "at least " + A + " characters"; lo = a; break;
        case 1: s.name = "max_length"; s.arg = "at most " + A + " characters"; hi = a; break;
        case 2: s.name = "length_between"; s.arg = "between " + A + " and " + B + " characters"; lo = a; hi = b; break;
        case 3: s.name = "exact_length"; s.arg = "exactly " + A + " characters"; lo = hi = a; break;
        default: s.name = "not_empty"; s.arg = "not empty"; lo = 1; break;
    }
    Agg g;
    g.kind = A_LENGTH;
    g.key = "length|" + col + "|" + std::to_string(lo) + "|" + std::to_string(hi);
    g.cols = {col};
    g.lo = lo;
    g.hi = hi;
    s.aggs.push_back(p.add_agg(std::move(g)));
    p.slots.push_back(std::move(s));
    return (int)p.slots.size() - 1;
}

// constraints/values.rs:217-296: COUNT(CASE WHEN c IN ('v', ..) THEN 1 END), COUNT(*) .. WHERE c IS NOT NULL
int plan_add_containment(Plan& p, const std::string& col, const std::vector<std::string>& allowed) {
    validate_identifier(col);
    Slot s;
    s.kind = SL_CONTAINMENT;
    s.name = "containment";
    s.columns = {col};
    std::string expr = col + " IN (";
    for (size_t i = 0; i < allowed.size(); ++i) {
        if (i) expr += ", ";
        expr += '\'';
        for (char c : allowed[i]) {
            expr += c;
            if (c == '\'') expr += '\'';  // values.rs:241 doubles single quotes
        }
        expr += '\'';
    }
    expr += ")";
    s.arg = expr;
    s.aggs.push_back(p.add_agg(mk_pred(expr)));
    s.aggs.push_back(p.add_agg(mk_valid(col)));
    p.slots.push_back(std::move(s));
    return (int)p.slots.size() - 1;
}

// constraints/values.rs:347-414: COUNT(CASE WHEN CAST(c AS DOUBLE) >= 0 THEN 1 END), COUNT(*) .. WHERE c IS NOT NULL
int plan_add_non_negative(Plan& p, const std::string& col) {
    validate_identifier(col);
    Slot s;
    s.kind = SL_NON_NEGATIVE;
    s.name = "non_negative";
    s.columns = {col};
    s.arg = col + " >= 0";
    s.aggs.push_back(p.add_agg(mk_pred(s.arg)));
    s.aggs.push_back(p.add_agg(mk_valid(col)));
    p.slots.push_back(std::move(s));
    return (int)p.slots.size() - 1;
}

// constraints/quantile.rs:165-224 (constructors), :282-482 (evaluate). Every quantile of a column reads the one KLL
// sketch the plan holds for it (APPROX_PERCENTILE_CONT's t-digest in the reference; §8c "parity unpinned": the values
// agree within the sketches' rank error, the status / message rules are the reference's).
int plan_add_quantile(Plan& p, const std::string& col, int mode, const std::vector<double>& quantiles,
                      const std::vector<tg_assertion>& assertions, int strict) {
    validate_identifier(col);
    if (mode < TG_QUANTILE_SINGLE || mode > TG_QUANTILE_UNIMPLEMENTED)
        throw Error(TG_ERR_INVALID_ARG, "unknown quantile validation kind");
    if (mode == TG_QUANTILE_SINGLE && quantiles.size() != 1)
        throw Error(TG_ERR_INVALID_ARG, "a single quantile check takes exactly one quantile");
    if (mode <= TG_QUANTILE_MULTIPLE && assertions.size() != quantiles.size())
        throw Error(TG_ERR_INVALID_ARG, "one assertion per quantile");
    for (double q : quantiles)  // QuantileCheck::new (:47-57)
        if (!(q >= 0.0 && q <= 1.0)) throw Error(TG_ERR_CONFIGURATION, "Quantile must be between 0.0 and 1.0");
    Slot s;
    s.kind = SL_QUANTILE;
    s.name = "quantile";
    s.columns = {col};
    s.sub_kind = mode;
    s.flag = strict;
    // should_use_exact (:244-277) counts the rows first in every mode, so an unknown table / column surfaces
    s.aggs.push_back(p.add_agg(mk_valid(col)));
    if (mode != TG_QUANTILE_UNIMPLEMENTED) {
        const int kll = p.add_agg(mk_kll(col, KLL_K_FOR_PERCENTILE));
        for (size_t i = 0; i < quantiles.size(); ++i)
            s.stats.push_back(StatReq{TG_STAT_PERCENTILE, quantiles[i],
                                      i < assertions.size() ? assertions[i] : tg_assertion{0, 0, 0}, kll});
    }
    p.slots.push_back(std::move(s));
    return (int)p.slots.size() - 1;
}

// constraints/approx_count_distinct.rs:40-134: SELECT APPROX_DISTINCT(c). The HyperLogLog estimate is replaced by
// the EXACT distinct count of the hash job (error 0 <= any HLL error bound; the reference's tests assert ranges).
int plan_add_approx_count_distinct(Plan& p, const std::string& col, tg_assertion a) {
    validate_identifier(col);
    Slot s;
    s.kind = SL_APPROX_DISTINCT;
    s.name = "approx_count_distinct";
    s.columns = {col};
    s.assertion = a;
    s.aggs.push_back(p.add_agg(mk_distinct({col})));
    p.slots.push_back(std::move(s));
    return (int)p.slots.size() - 1;
}

// constraints/values.rs:28-37 (DataType::pattern), :88-165: COUNT(CASE WHEN c ~ 'pattern' ..), COUNT(*) .. WHERE c IS
// NOT NULL; data_type: 0 Integer 1 Float 2 Boolean 3 Date 4 Timestamp 5 String
int plan_add_data_type(Plan& p, const std::string& col, int data_type, double threshold) {
    validate_identifier(col);
    if (!(threshold >= 0.0 && threshold <= 1.0)) throw Error(TG_ERR_VALIDATION, "Threshold must be between 0.0 and 1.0");
    static const char* patterns[] = {"^-?\\d+$", "^-?\\d*\\.?\\d+([eE][+-]?\\d+)?$", "^(true|false|TRUE|FALSE|True|False|0|1)$",
                                     "^\\d{4}-\\d{2}-\\d{2}$", "^\\d{4}-\\d{2}-\\d{2}[ T]\\d{2}:\\d{2}:\\d{2}", ".*"};
    if (data_type < 0 || data_type > 5) throw Error(TG_ERR_INVALID_ARG, "unknown data type");
    Slot s;
    s.kind = SL_DATA_TYPE;
    s.name = "data_type";
    s.columns = {col};
    s.threshold = threshold;
    s.pattern = patterns[data_type];
    s.aggs.push_back(p.add_agg(mk_regex(col, s.pattern, false, false)));
    p.slots.push_back(std::move(s));
    return (int)p.slots.size() - 1;
}

// constraints/column_count.rs:43-85: the table's schema width against an assertion
int plan_add_column_count(Plan& p, tg_assertion a) {
    Slot s;
    s.kind = SL_COLUMN_COUNT;
    s.name = "column_count";
    s.assertion = a;
    s.aggs.push_back(p.add_agg(mk_rows()));
    p.slots.push_back(std::move(s));
    return (int)p.slots.size() - 1;
}

// analyzers/advanced/histogram.rs:62-76 (num_buckets clamped to 1..1000), :184-345
int plan_add_histogram(Plan& p, const std::string& col, int num_buckets) {
    validate_identifier(col);
    Slot s;
    s.kind = SL_HISTOGRAM;
    s.name = "histogram";
    s.metric_key = "histogram." + col;
    s.columns = {col};
    s.k = std::min(std::max(num_buckets, 1), 1000);
    Agg num = mk_num(col, 3);  // moments + min/max
    s.aggs.push_back(p.add_agg(std::move(num)));
    Agg h;
    h.kind = A_HIST;
    h.key = "hist|" + col + "|" + std::to_string(s.k);
    h.cols = {col};
    h.iparam = s.k;
    s.aggs.push_back(p.add_agg(std::move(h)));
    p.slots.push_back(std::move(s));
    return (int)p.slots.size() - 1;
}

int plan_add_grouped_completeness(Plan& p, const std::string& col, const std::vector<std::string>& groups,
                                  int max_groups, int include_overall) {
    if (groups.empty()) throw Error(TG_ERR_INVALID_ARG, "at least one grouping column is required");
    Slot s;
    s.kind = SL_GROUPED;
    s.name = "completeness";
    s.metric_key = "completeness." + col + "_grouped_by_";
    for (size_t i = 0; i < groups.size(); ++i) s.metric_key += (i ? "_" : "") + groups[i];
    s.columns = {col};
    s.max_groups = max_groups;
    s.include_overall = include_overall;
    Agg a;
    a.kind = A_GROUPED;
    a.key = "grouped|" + col;
    a.cols = {col};
    for (auto& g : groups) {
        a.key += "|" + g;
        a.cols.push_back(g);
    }
    s.aggs.push_back(p.add_agg(std::move(a)));
    p.slots.push_back(std::move(s));
    return (int)p.slots.size() - 1;
}

int plan_add_value_histogram(Plan& p, const std::string& col) {
    Slot s;
    s.kind = SL_VALUE_HIST;
    s.name = "histogram";
    s.metric_key = "histogram." + col;
    s.columns = {col};
    Agg a;
    a.kind = A_GROUPED;
    a.key = "vhist|" + col;
    a.cols = {col, col};  // target and grouping column: a group's non-NULL count is its size, the NULL group counts the NULLs
    a.flags = 2;
    s.aggs.push_back(p.add_agg(std::move(a)));
    p.slots.push_back(std::move(s));
    return (int)p.slots.size() - 1;
}

// ---- partial (de)serialisation: [u64 n_aggs] then per agg: kind, err, u[8], f[8], blob_len, blob, err_len, err ----
size_t Plan::partial_size() const {
    size_t n = 8;
    for (auto& a : aggs) n += 8 + 8 + 64 + 64 + 8 + ((a.blob.size() + 7) & ~size_t(7)) + 8 + ((a.err_msg.size() + 7) & ~size_t(7));
    return n;
}

void Plan::partial_export(uint8_t* buf) const {
    uint8_t* p = buf;
    auto put64 = [&](uint64_t v) {
        memcpy(p, &v, 8);
        p += 8;
    };
    put64(aggs.size());
    for (auto& a : aggs) {
        put64((uint64_t)a.kind);
        put64((uint64_t)a.err);
        memcpy(p, a.u, 64);
        p += 64;
        memcpy(p, a.f, 64);
        p += 64;
        put64(a.blob.size());
        size_t padded = (a.blob.size() + 7) & ~size_t(7);
        memset(p, 0, padded);
        if (!a.blob.empty()) memcpy(p, a.blob.data(), a.blob.size());
        p += padded;
        put64(a.err_msg.size());
        padded = (a.err_msg.size() + 7) & ~size_t(7);
        memset(p, 0, padded);
        memcpy(p, a.err_msg.data(), a.err_msg.size());
        p += padded;
    }
}

// re-pivot shifted sums (n, Σ(x-K1), Σ(x-K1)²) onto pivot K0
static void repivot1(double n, double delta, double& s, double& q) {
    // d' = d + delta
    q = q + 2.0 * delta * s + n * delta * delta;
    s = s + n * delta;
}

void Plan::partial_merge(const uint8_t* buf, size_t nbytes) {
    const uint8_t* p = buf;
    const uint8_t* end = buf + nbytes;
    auto get64 = [&]() {
        if (p + 8 > end) throw Error(TG_ERR_INVALID_ARG, "partial blob truncated");
        uint64_t v;
        memcpy(&v, p, 8);
        p += 8;
        return v;
    };
    uint64_t n = get64();
    if (n != aggs.size()) throw Error(TG_ERR_INVALID_ARG, "partial blob does not belong to this plan (aggregate count differs)");
    for (auto& a : aggs) {
        uint64_t kind = get64();
        if ((int32_t)kind != a.kind) throw Error(TG_ERR_INVALID_ARG, "partial blob does not belong to this plan (aggregate kind differs)");
        tg_status err = (tg_status)get64();
        uint64_t u[8];
        double f[8];
        if (p + 128 > end) throw Error(TG_ERR_INVALID_ARG, "partial blob truncated");
        memcpy(u, p, 64);
        p += 64;
        memcpy(f, p, 64);
        p += 64;
        uint64_t blen = get64();
        size_t padded = (blen + 7) & ~size_t(7);
        if (p + padded > end) throw Error(TG_ERR_INVALID_ARG, "partial blob truncated");
        std::vector<uint8_t> blob(p, p + blen);
        p += padded;
        uint64_t elen = get64();
        padded = (elen + 7) & ~size_t(7);
        if (p + padded > end) throw Error(TG_ERR_INVALID_ARG, "partial blob truncated");
        std::string emsg((const char*)p, elen);
        p += padded;
        merge_state((int)(&a - aggs.data()), err, emsg, u, f, blob);
    }
}

// one shard's state of aggregate i folded into ours (AnalyzerState::merge, analyzers/traits.rs:154-179)
void Plan::merge_state(int i, tg_status err, const std::string& emsg, const uint64_t* u, const double* f, const std::vector<uint8_t>& blob) {
    Agg& a = aggs[i];
    if (err != TG_OK && a.err == TG_OK) {
        a.err = err;
        a.err_msg = emsg;
    }
    {
        switch (a.kind) {
            case A_ROWS:
                a.u[0] += u[0];
                a.u[1] = std::max(a.u[1], u[1]);  // schema width: the same on every shard
                break;
            case A_VALID:
            case A_REGEX:
            case A_LENGTH:
                for (int i = 0; i < 8; ++i) a.u[i] += u[i];
                break;
            case A_HIST:
                // bucket bounds come from the shard's own min / max: the counts only add up when those agree. Shards
                // with different ranges leave the aggregate PENDING (u[7] = 1): the host layer then re-counts every
                // shard against the merged (global) min / max and installs the sums (two-phase histogram,
                // tg_plan_histogram_pending / _rebucket / _install); finalize reports an error while it is pending.
                if (u[7]) a.u[7] = 1;
                if (blob.empty()) break;  // that shard held no values
                if (a.blob.empty() && !a.u[7]) {
                    a.blob = blob;
                    a.f[0] = f[0];
                    a.f[1] = f[1];
                } else if (!a.u[7] && a.f[0] == f[0] && a.f[1] == f[1] && a.blob.size() == blob.size()) {
                    for (size_t i = 0; i + 8 <= blob.size(); i += 8) {
                        uint64_t x, y;
                        memcpy(&x, a.blob.data() + i, 8);
                        memcpy(&y, blob.data() + i, 8);
                        x += y;
                        memcpy(a.blob.data() + i, &x, 8);
                    }
                } else {
                    a.u[7] = 1;
                    a.blob.clear();
                }
                break;
            case A_PRED:
                a.u[0] += u[0];
                a.u[1] |= u[1];
                a.u[2] += u[2];
                break;
            case A_DISTINCT:
            case A_FK:
                // exact because the key space is hash-partitioned across shards before counting
                for (int i = 0; i < 8; ++i) a.u[i] += u[i];
                if (a.kind == A_FK) {
                    // examples: concatenate up to the cap (blob = [count u64][len-prefixed strings])
                    if (a.blob.empty()) a.blob = blob;
                    else if (!blob.empty()) {
                        uint64_t c0, c1;
                        memcpy(&c0, a.blob.data(), 8);
                        memcpy(&c1, blob.data(), 8);
                        const uint8_t* q = blob.data() + 8;
                        for (uint64_t i = 0; i < c1 && (int64_t)c0 < (int64_t)a.iparam; ++i) {
                            uint32_t L;
                            memcpy(&L, q, 4);
                            a.blob.insert(a.blob.end(), q, q + 4 + L);
                            q += 4 + L;
                            ++c0;
                        }
                        memcpy(a.blob.data(), &c0, 8);
                    }
                }
                break;
            case A_NUM: {
                if (u[0] == 0) break;  // other side empty
                if (a.u[0] == 0) {
                    memcpy(a.u, u, 64);
                    memcpy(a.f, f, 64);
                    break;
                }
                double s = f[1], q = f[2];
                repivot1((double)u[0], f[0] - a.f[0], s, q);
                a.f[1] += s;
                a.f[2] += q;
                a.f[5] += f[5];
                a.u[1] += u[1];  // wrapping i64 sum
                if (a.u[4]) {
                    a.u[2] = (uint64_t)std::min((int64_t)a.u[2], (int64_t)u[2]);
                    a.u[3] = (uint64_t)std::max((int64_t)a.u[3], (int64_t)u[3]);
                }
                a.f[3] = std::fmin(a.f[3], f[3]);
                a.f[4] = std::fmax(a.f[4], f[4]);
                a.u[0] += u[0];
            } break;
            case A_PAIR:
            case A_SPEARMAN: {
                if (u[0] == 0) break;
                if (a.u[0] == 0) {
                    memcpy(a.u, u, 64);
                    memcpy(a.f, f, 64);
                    break;
                }
                const double nn = (double)u[0], dx = f[0] - a.f[0], dy = f[1] - a.f[1];
                // dx' = dx + a, dy' = dy + b
                double sx = f[2], sy = f[3], sxx = f[4], syy = f[5], sxy = f[6];
                sxy = sxy + dx * sy + dy * sx + nn * dx * dy;
                repivot1(nn, dx, sx, sxx);
                repivot1(nn, dy, sy, syy);
                a.f[2] += sx;
                a.f[3] += sy;
                a.f[4] += sxx;
                a.f[5] += syy;
                a.f[6] += sxy;
                a.u[0] += u[0];
            } break;
            case A_KLL:
                a.u[0] += u[0];
                kll_blob_merge(a.blob, blob);
                break;
            case A_GROUPED:
                grouped_blob_merge(a.blob, blob);
                break;
        }
    }
}

// two-phase histogram: the HIST aggregates whose shards disagreed on [min, max]
std::vector<int> Plan::histogram_pending() const {
    std::vector<int> out;
    for (size_t i = 0; i < aggs.size(); ++i)
        if (aggs[i].kind == A_HIST && aggs[i].u[7] && aggs[i].err == TG_OK) out.push_back((int)i);
    return out;
}
void Plan::histogram_install(int agg_id, const uint64_t* counts, int nb) {
    if (agg_id < 0 || agg_id >= (int)aggs.size() || aggs[agg_id].kind != A_HIST) throw Error(TG_ERR_INVALID_ARG, "not a histogram aggregate");
    Agg& a = aggs[agg_id];
    const int want = std::min(std::max(a.iparam, 1), 1000);
    if (nb != want || !counts) throw Error(TG_ERR_INVALID_ARG, "histogram has " + std::to_string(want) + " buckets");
    a.blob.assign((size_t)nb * 8, 0);
    memcpy(a.blob.data(), counts, (size_t)nb * 8);
    for (auto& o : aggs)
        if (o.kind == A_NUM && o.cols.size() == 1 && o.cols[0] == a.cols[0]) {
            a.f[0] = o.f[3];
            a.f[1] = o.f[4];
        }
    a.u[7] = 0;
}

// ---- grouped blob: [u64 n_entries] then per entry: u32 key_len, key bytes (fields joined by \x1f), u64 total, u64 non_null.
// Merging appends the other shard's entries (GroupedCompletenessState::merge adds the counts of equal keys,
// grouped_completeness.rs:37-84; here equal keys are summed when the state is read — grouped_blob_compact — so that merging
// 8 shards costs 8 appends, not 8 rebuilds of a string-keyed map).
void grouped_blob_compact(std::vector<uint8_t>& b) {
    if (b.size() < 8) return;
    uint64_t n;
    memcpy(&n, b.data(), 8);
    struct Ent {
        const uint8_t* key;
        uint32_t len;
        uint64_t total, nn;
    };
    // open-addressing index over the entries (FNV-1a of the key bytes): no per-entry allocation — a state read costs
    // microseconds even with thousands of groups
    size_t cap = 16;
    while (cap < (size_t)n * 2) cap <<= 1;
    std::vector<uint32_t> slot(cap, 0xFFFFFFFFu);
    std::vector<Ent> ents;
    ents.reserve((size_t)n);
    const uint8_t* p = b.data() + 8;
    bool dup = false;
    for (uint64_t i = 0; i < n; ++i) {
        uint32_t L;
        memcpy(&L, p, 4);
        p += 4;
        uint64_t t, nn;
        memcpy(&t, p + L, 8);
        memcpy(&nn, p + L + 8, 8);
        uint64_t h = 0xcbf29ce484222325ull;
        for (uint32_t k = 0; k < L; ++k) h = (h ^ p[k]) * 0x100000001b3ull;
        size_t q = (size_t)(h ^ (h >> 29)) & (cap - 1);
        while (true) {
            const uint32_t at = slot[q];
            if (at == 0xFFFFFFFFu) {
                slot[q] = (uint32_t)ents.size();
                ents.push_back(Ent{p, L, t, nn});
                break;
            }
            if (ents[at].len == L && memcmp(ents[at].key, p, L) == 0) {
                ents[at].total += t;
                ents[at].nn += nn;
                dup = true;
                break;
            }
            q = (q + 1) & (cap - 1);
        }
        p += L + 16;
    }
    if (!dup) return;
    std::vector<uint8_t> out(8);
    const uint64_t m = ents.size();
    memcpy(out.data(), &m, 8);
    out.reserve(b.size());
    for (auto& e : ents) {
        const size_t o = out.size();
        out.resize(o + 4 + e.len + 16);
        memcpy(out.data() + o, &e.len, 4);
        memcpy(out.data() + o + 4, e.key, e.len);
        memcpy(out.data() + o + 4 + e.len, &e.total, 8);
        memcpy(out.data() + o + 4 + e.len + 8, &e.nn, 8);
    }
    b.swap(out);
}

void grouped_blob_merge(std::vector<uint8_t>& into, const std::vector<uint8_t>& other) {
    if (other.size() < 8) return;
    if (into.size() < 8) {
        into = other;
        return;
    }
    uint64_t a, b;
    memcpy(&a, into.data(), 8);
    memcpy(&b, other.data(), 8);
    a += b;
    memcpy(into.data(), &a, 8);
    into.insert(into.end(), other.begin() + 8, other.end());
    if (into.size() > ((size_t)8 << 20)) grouped_blob_compact(into);  // long merge chains (incremental runs) stay bounded
}

// ------------------------------------------------------------------ finalize ----

static void set_error(Slot& s, const Agg& a) {
    s.status = TG_FAILURE;
    s.has_metric = false;
    s.has_message = true;
    s.message = "Error evaluating constraint: " + a.err_msg;
    s.ares.error = 2;
}
static void skipped(Slot& s, const std::string& m) {
    s.status = TG_SKIPPED;
    s.has_metric = false;
    s.has_message = true;
    s.message = m;
}
static void success_metric(Slot& s, double v) {
    s.status = TG_SUCCESS;
    s.has_metric = true;
    s.metric = v;
    s.has_message = false;
}
static void failure_metric(Slot& s, double v, const std::string& m) {
    s.status = TG_FAILURE;
    s.has_metric = true;
    s.metric = v;
    s.has_message = true;
    s.message = m;
}
static void failure(Slot& s, const std::string& m) {
    s.status = TG_FAILURE;
    s.has_metric = false;
    s.has_message = true;
    s.message = m;
}

static std::string join(const std::vector<std::string>& v, const char* sep) {
    std::string r;
    for (size_t i = 0; i < v.size(); ++i) {
        if (i) r += sep;
        r += v[i];
    }
    return r;
}

// Σ(x-x̄)² from the shifted sums: m2 = Σd² - (Σd)²/n with d = x - K.
//  * a rounding-negative m2 is 0;
//  * a NaN or an infinite value in the column makes Σd and Σd² NaN / infinite and m2 NaN (DataFusion's VARIANCE is NaN);
//  * finite values whose squared deviations overflow leave Σd finite (an infinite value would make it infinite or NaN)
//    but Σd² = +inf, and inf - inf would read NaN: the variance is beyond the double range, +inf (as DataFusion's).
static double central_m2(double n, double sd, double sdd) {
    const double m2 = sdd - sd * sd / n;
    if (m2 < 0.0) return 0.0;
    if (std::isnan(m2) && std::isfinite(sd) && sdd == INFINITY) return INFINITY;
    return m2;
}

// value of a SQL aggregate over the A_NUM state, with DataFusion result typing
// (constraints/statistics.rs:278-308): returns false when the SQL result is NULL
static bool stat_value(const Agg& a, int kind, double* out) {
    const uint64_t n = a.u[0];
    const bool is_i64 = a.u[4] != 0;
    switch (kind) {
        case TG_STAT_MIN:
            if (n == 0) return false;
            *out = is_i64 ? (double)(int64_t)a.u[2] : a.f[3];
            return true;
        case TG_STAT_MAX:
            if (n == 0) return false;
            *out = is_i64 ? (double)(int64_t)a.u[3] : a.f[4];
            return true;
        case TG_STAT_MEAN:
            if (n == 0) return false;
            *out = a.f[5] / (double)n;
            return true;
        case TG_STAT_SUM:
            if (n == 0) return false;
            *out = is_i64 ? (double)(int64_t)a.u[1] : a.f[5];
            return true;
        case TG_STAT_STDDEV:
        case TG_STAT_VARIANCE: {
            if (n < 2) return false;
            double nn = (double)n;
            double var = central_m2(nn, a.f[1], a.f[2]) / (nn - 1.0);
            *out = kind == TG_STAT_STDDEV ? std::sqrt(var) : var;
            return true;
        }
    }
    return false;
}

bool slot_has_row_mask(const Slot& s) {
    switch (s.kind) {
        case SL_COMPLETENESS: return s.columns.size() == 1;
        case SL_SQL:
        case SL_CONTAINMENT:
        case SL_NON_NEGATIVE:
        case SL_FORMAT:
        case SL_DATA_TYPE:
        case SL_LENGTH: return true;
        case SL_ANALYZER: return s.sub_kind == TG_AN_COMPLETENESS || s.sub_kind == TG_AN_COMPLIANCE;
        default: return false;
    }
}

void plan_request_row_mask(Plan& p, int slot) {
    if (slot < 0 || slot >= (int)p.slots.size()) throw Error(TG_ERR_INVALID_ARG, "slot index out of range");
    Slot& s = p.slots[slot];
    if (!slot_has_row_mask(s))
        throw Error(TG_ERR_UNSUPPORTED, "row verdicts are not available for the '" + s.name + "' slot (row-level constraints only)");
    s.mask_requested = true;
    s.mask_built = false;
    // the first aggregate holds the per-row decision (predicate, pattern, length range); COUNT(c) needs no bits: the column's
    // validity bitmap is its verdict
    p.aggs[s.aggs[0]].row_bits = true;
}

const Slot& key_rows_slot(const Plan& p, int slot, int kind) {
    if (slot < 0 || slot >= (int)p.slots.size()) throw Error(TG_ERR_INVALID_ARG, "slot index out of range");
    const Slot& s = p.slots[slot];
    if (s.kind != SL_UNIQ && s.kind != SL_FK)
        throw Error(TG_ERR_UNSUPPORTED, "key-level row verdicts are not available for the '" + s.name + "' slot (uniqueness and foreign-key constraints only)");
    const bool fits = s.kind == SL_UNIQ ? kind == TG_KEY_ROWS_DUPLICATE || kind == TG_KEY_ROWS_FIRST : kind == TG_KEY_ROWS_ORPHAN;
    if (!fits)
        throw Error(TG_ERR_INVALID_ARG, "key-level row verdict kind " + std::to_string(kind) + " does not apply to the '" + s.name +
                                            "' slot (uniqueness: DUPLICATE or FIRST; foreign key: ORPHAN)");
    return s;
}

void plan_request_key_rows(Plan& p, int slot, int kind) {
    key_rows_slot(p, slot, kind);
    Slot& s = p.slots[slot];
    s.key_rows_requested |= (uint8_t)(1u << kind);
    s.mask_built = false;
    p.aggs[s.aggs[0]].key_rows |= (uint8_t)(1u << kind);
}

static void finalize_completeness(Plan& p, Slot& s) {
    // per-column evaluate_column (completeness.rs:137-246)
    struct ColRes {
        int status;
        bool has_metric;
        double metric;
        std::string msg;
    };
    std::vector<ColRes> rs;
    for (size_t i = 0; i < s.columns.size(); ++i) {
        const Agg& a = p.aggs[s.aggs[i]];
        if (a.err != TG_OK) {  // `?` propagates the first error
            set_error(s, a);
            s.ares.error = 0;
            return;
        }
        ColRes r{};
        const double total = (double)a.u[0], nn = (double)a.u[1];
        if (total == 0.0) {
            r.status = TG_SKIPPED;
            r.msg = "No data to validate";
        } else {
            double c = nn / total;
            r.has_metric = true;
            r.metric = c;
            if (c >= s.threshold) r.status = TG_SUCCESS;
            else {
                r.status = TG_FAILURE;
                r.msg = "Column '" + s.columns[i] + "' completeness " + fmt_f64_prec(c * 100.0, 2) +
                        "% is below threshold " + fmt_f64_prec(s.threshold * 100.0, 2) + "%";
            }
        }
        rs.push_back(r);
    }
    if (rs.empty()) {
        skipped(s, "No columns specified");
        return;
    }
    if (rs.size() == 1) {
        s.status = rs[0].status;
        s.has_metric = rs[0].has_metric;
        s.metric = rs[0].metric;
        s.has_message = !rs[0].msg.empty();
        s.message = rs[0].msg;
        return;
    }
    // core/unified.rs:52-121
    std::vector<bool> bools;
    std::vector<double> metrics;
    for (auto& r : rs) {
        bools.push_back(r.status == TG_SUCCESS);
        if (r.has_metric) metrics.push_back(r.metric);
    }
    bool ok = logical_evaluate(s.op, s.op_n, bools);
    s.has_metric = !metrics.empty();
    if (s.has_metric) {
        double sum = 0;
        for (double m : metrics) sum += m;
        s.metric = sum / (double)metrics.size();
    }
    if (ok) {
        s.status = TG_SUCCESS;
        if (s.op == TG_OP_ALL) {
            s.has_message = true;
            s.message = "All " + std::to_string(s.columns.size()) + " columns satisfy the constraint";
        } else if (s.op == TG_OP_ANY) {
            std::vector<std::string> passed;
            for (size_t i = 0; i < rs.size(); ++i)
                if (bools[i]) passed.push_back(s.columns[i]);
            s.has_message = true;
            s.message = "Columns " + join(passed, ", ") + " satisfy the constraint";
        } else {
            s.has_message = false;
        }
    } else {
        s.status = TG_FAILURE;
        std::vector<std::string> failed;
        for (size_t i = 0; i < rs.size(); ++i)
            if (!bools[i]) failed.push_back(s.columns[i]);
        s.has_message = true;
        s.message = "Constraint failed for columns: " + join(failed, ", ") + ". Required: " +
                    logical_description(s.op, s.op_n);
    }
}

static bool percentile_value(Plan& p, const StatReq& r, double* out) {
    if (r.agg_kll < 0) return false;
    const Agg& k = p.aggs[r.agg_kll];
    if (k.err != TG_OK || k.u[0] == 0) return false;
    return kll_blob_query(k.blob, r.percentile, out);
}

// DataFusion result typing for Int32 / Float32 columns: MIN / MAX / APPROX_PERCENTILE_CONT keep the column's type (the
// reference then fails its Int64 / Float64 downcasts), SUM widens to Int64 / Float64, AVG / STDDEV / VAR are Float64
static bool narrow_result(const Agg& a, int kind) {
    if ((a.narrow & 1) && (kind == TG_STAT_MIN || kind == TG_STAT_MAX || kind == TG_STAT_MEDIAN || kind == TG_STAT_PERCENTILE)) return true;
    return (a.narrow & 2) && kind == TG_STAT_SUM;  // SUM(UInt*) is UInt64
}

static void finalize_stat(Plan& p, Slot& s) {
    const Agg& a = p.aggs[s.aggs[0]];
    if (a.err != TG_OK) {
        set_error(s, a);
        return;
    }
    const StatReq& r = s.stats[0];
    if (narrow_result(a, r.kind)) {  // an Int32 / Float32 result array: neither downcast succeeds (statistics.rs:278-308)
        Agg er = a;
        er.err_msg = "Internal error: Failed to extract statistic value";
        set_error(s, er);
        return;
    }
    double v;
    bool ok;
    if (r.kind == TG_STAT_MEDIAN || r.kind == TG_STAT_PERCENTILE) {
        if (p.aggs[r.agg_kll].err != TG_OK) {
            set_error(s, p.aggs[r.agg_kll]);
            return;
        }
        ok = percentile_value(p, r, &v);
    } else {
        ok = stat_value(a, r.kind, &v);
    }
    const std::string name = stat_name(r.kind, r.percentile);
    if (!ok) {
        failure(s, name + " is null (no non-null values)");
        return;
    }
    if (assertion_evaluate(r.assertion, v)) success_metric(s, v);
    else failure_metric(s, v, name + " " + fmt_f64(v) + " does not " + assertion_description(r.assertion));
}

static void finalize_multistat(Plan& p, Slot& s) {
    const Agg& a = p.aggs[s.aggs[0]];
    if (a.err != TG_OK) {
        set_error(s, a);
        return;
    }
    std::vector<std::string> failures;
    std::vector<double> metrics;
    for (auto& r : s.stats) {
        if (narrow_result(a, r.kind)) {  // statistics.rs:481-485
            failures.push_back(std::string("Failed to compute ") + stat_name(r.kind, r.percentile));
            continue;
        }
        double v;
        bool ok = (r.kind == TG_STAT_MEDIAN || r.kind == TG_STAT_PERCENTILE) ? percentile_value(p, r, &v)
                                                                             : stat_value(a, r.kind, &v);
        const std::string name = stat_name(r.kind, r.percentile);
        if (!ok) {
            failures.push_back(name + " is null");
            continue;
        }
        metrics.push_back(v);
        if (!assertion_evaluate(r.assertion, v))
            failures.push_back(name + " is " + fmt_f64(v) + " which does not " + assertion_description(r.assertion));
    }
    if (failures.empty()) success_metric(s, metrics.empty() ? 0.0 : metrics[0]);
    else failure(s, join(failures, "; "));
}

// `{:?}` of an f64: Display plus ".0" when Display printed an integer
static std::string fmt_f64_debug(double v) {
    std::string t = fmt_f64(v);
    if (std::isfinite(v) && t.find_first_of(".e") == std::string::npos) t += ".0";
    return t;
}

// constraints/quantile.rs:285-482. An aggregate over no rows yields one NULL row which the reference reads with
// `.value(0)` (no null check, :311-316) => 0.0; mirrored.
static void finalize_quantile(Plan& p, Slot& s) {
    const Agg& rows = p.aggs[s.aggs[0]];
    if (rows.err != TG_OK) {
        set_error(s, rows);
        return;
    }
    if (s.sub_kind == TG_QUANTILE_UNIMPLEMENTED) {  // Distribution / Custom (:474-479)
        s.status = TG_SKIPPED;
        s.has_message = true;
        s.message = "Validation type not yet implemented";
        return;
    }
    std::vector<double> values;
    for (auto& r : s.stats) {
        if (p.aggs[r.agg_kll].err != TG_OK) {
            set_error(s, p.aggs[r.agg_kll]);
            return;
        }
        double v = 0.0;
        if (!percentile_value(p, r, &v)) v = 0.0;
        values.push_back(v);
    }
    if (s.sub_kind == TG_QUANTILE_SINGLE) {
        const StatReq& r = s.stats[0];
        const double v = values[0];
        if (assertion_evaluate(r.assertion, v)) success_metric(s, v);
        else failure_metric(s, v, "Quantile " + fmt_f64(r.percentile) + " is " + fmt_f64(v) + " which does not " +
                                      assertion_description(r.assertion));
    } else if (s.sub_kind == TG_QUANTILE_MULTIPLE) {
        std::vector<std::string> failures;
        for (size_t i = 0; i < s.stats.size(); ++i)
            if (!assertion_evaluate(s.stats[i].assertion, values[i]))
                failures.push_back("Q" + std::to_string((int32_t)(s.stats[i].percentile * 100.0)) + " is " +
                                   fmt_f64(values[i]) + " which does not " +
                                   assertion_description(s.stats[i].assertion));
        if (failures.empty()) {
            s.status = TG_SUCCESS;
        } else {
            failure(s, join(failures, "; "));
        }
    } else {  // Monotonic (:402-472)
        bool mono = true;
        for (size_t i = 1; i < values.size() && mono; ++i)
            mono = s.flag ? values[i] > values[i - 1] : values[i] >= values[i - 1];
        if (mono) {
            s.status = TG_SUCCESS;
        } else {
            std::vector<std::string> parts;
            for (double v : values) parts.push_back(fmt_f64_debug(v));
            failure(s, std::string("Quantiles are not ") + (s.flag ? "strictly" : "") + " monotonic: [" +
                           join(parts, ", ") + "]");
        }
    }
}

static void finalize_format(Plan& p, Slot& s) {
    const Agg& a = p.aggs[s.aggs[0]];
    if (a.err != TG_OK) {
        set_error(s, a);
        return;
    }
    const double matches = (double)(a.u[0] + (s.fopt.null_is_valid ? a.u[1] : 0));
    const double total = (double)a.u[2];
    if (total == 0.0) {
        skipped(s, "No data to validate");
        return;
    }
    const double ratio = matches / total;
    const bool detect = s.sub_kind == TG_FMT_CREDIT_CARD && s.flag;
    const bool ok = detect ? ratio <= s.threshold : ratio >= s.threshold;
    if (ok) {
        success_metric(s, ratio);
        return;
    }
    std::string msg;
    if (detect)
        msg = "Credit card detection ratio " + fmt_f64_prec(ratio, 3) + " exceeds threshold " +
              fmt_f64_prec(s.threshold, 3);
    else
        msg = "Format validation ratio " + fmt_f64_prec(ratio, 3) + " is below threshold " +
              fmt_f64_prec(s.threshold, 3) + " - values that " +
              format_description(s.sub_kind, s.pattern, s.has_arg ? s.arg.c_str() : nullptr, s.flag);
    failure_metric(s, ratio, msg);
}

static void finalize_uniq(Plan& p, Slot& s) {
    const Agg& a = p.aggs[s.aggs[0]];
    if (a.err != TG_OK) {
        set_error(s, a);
        return;
    }
    const bool multi = s.columns.size() > 1;
    const double total = (double)a.u[0];
    const uint64_t distinct_nonnull = a.u[1], singletons = a.u[2], any_null_rows = a.u[3], distinct_all = a.u[5];
    // COUNT(DISTINCT expr): single column ignores NULL; (a, b) is a struct value that is never NULL
    const uint64_t count_distinct_expr = multi ? distinct_all : distinct_nonnull;
    const std::string cols = join(s.columns, ", ");
    if (s.sub_kind == TG_UNIQ_FULL || s.sub_kind == TG_UNIQ_WITH_NULLS || s.sub_kind == TG_UNIQ_COMPOSITE) {
        uint64_t unique = count_distinct_expr;
        if (s.sub_kind == TG_UNIQ_WITH_NULLS && !multi) {
            if (s.null_handling == TG_NULLS_INCLUDE) unique = distinct_all;  // COALESCE(c,'<NULL>')
            else if (s.null_handling == TG_NULLS_DISTINCT) unique = distinct_nonnull + any_null_rows;
        }
        if (total == 0.0) {
            skipped(s, "No data to validate");
            return;
        }
        const double ratio = (double)unique / total;
        if (ratio >= s.threshold) success_metric(s, ratio);
        else
            failure_metric(s, ratio,
                           "Uniqueness ratio " + fmt_f64_prec(ratio, 3) + " is below threshold " +
                               fmt_f64_prec(s.threshold, 3) + " for columns: " + cols);
        return;
    }
    if (s.sub_kind == TG_UNIQ_DISTINCTNESS || s.sub_kind == TG_UNIQ_UNIQUE_VALUE_RATIO) {
        // distinctness multi-column concatenates COALESCE(.., '<NULL>') => NULL is a value
        const double count = s.sub_kind == TG_UNIQ_DISTINCTNESS ? (double)(multi ? distinct_all : distinct_nonnull)
                                                                : (double)singletons;
        if (total == 0.0) {
            skipped(s, "No data to validate");
            return;
        }
        const double ratio = count / total;
        if (assertion_evaluate(s.assertion, ratio)) success_metric(s, ratio);
        else
            failure_metric(s, ratio,
                           s.name + " ratio " + fmt_f64_prec(ratio, 3) + " does not satisfy " +
                               assertion_description(s.assertion) + " for columns: " + cols);
        return;
    }
    // primary key (uniqueness.rs:797-852)
    if (total == 0.0) {
        skipped(s, "No data to validate");
        return;
    }
    const double null_count = (double)any_null_rows, unique = (double)count_distinct_expr;
    if (null_count > 0.0)
        failure_metric(s, null_count / total,
                       "Primary key columns contain " + fmt_f64(null_count) + " NULL values: " + cols);
    else if (unique != total)
        failure_metric(s, (total - unique) / total,
                       "Primary key columns contain " + fmt_f64(total - unique) + " duplicate values: " + cols);
    else success_metric(s, 1.0);
}

// CORR / COVAR_SAMP of the pairwise-complete rows; NULL results read as 0.0 (correlation.rs:355-362)
static double pair_corr(const Agg& a) {
    const double n = (double)a.u[0];
    if (a.u[0] < 2) return 0.0;
    const double cxy = n * a.f[6] - a.f[2] * a.f[3];
    const double vx = n * a.f[4] - a.f[2] * a.f[2], vy = n * a.f[5] - a.f[3] * a.f[3];
    const double den = std::sqrt(vx * vy);
    if (!(den > 0.0)) return 0.0;
    return cxy / den;
}
static double pair_covar_samp(const Agg& a) {
    const double n = (double)a.u[0];
    if (a.u[0] < 2) return 0.0;
    return (a.f[6] - a.f[2] * a.f[3] / n) / (n - 1.0);
}

static void finalize_corr(Plan& p, Slot& s) {
    const std::string &c1 = s.columns[0], &c2 = s.columns[1];
    if (s.sub_kind == TG_CORR_SPEARMAN || s.sub_kind == TG_CORR_KENDALL || s.sub_kind == TG_CORR_MUTUAL_INFORMATION) {
        skipped(s, "Correlation type not yet implemented");
        return;
    }
    const Agg& a = p.aggs[s.aggs[0]];
    if (a.err != TG_OK) {
        set_error(s, a);
        return;
    }
    if (s.sub_kind == TG_CORR_INDEPENDENCE) {
        const double v = std::fabs(pair_corr(a));
        if (v <= s.assertion.a) success_metric(s, v);
        else
            failure_metric(s, v,
                           "Columns " + c1 + " and " + c2 + " have correlation " + fmt_f64(v) +
                               " exceeding independence threshold " + fmt_f64(s.assertion.a));
        return;
    }
    const bool cov = s.sub_kind == TG_CORR_COVARIANCE;
    const double v = cov ? pair_covar_samp(a) : pair_corr(a);
    if (assertion_evaluate(s.assertion, v)) success_metric(s, v);
    else
        failure_metric(s, v,
                       std::string(cov ? "covariance" : "Pearson correlation") + " between " + c1 + " and " + c2 +
                           " is " + fmt_f64(v) + " which does not " + assertion_description(s.assertion));
}

static void finalize_sql(Plan& p, Slot& s) {
    const Agg& a = p.aggs[s.aggs[0]];
    if (a.err != TG_OK) {
        // planning / binding problems are reported as a failed constraint (custom_sql.rs:212-232)
        failure(s, "SQL expression error: " + a.err_msg + ". Expression: '" + s.arg + "'");
        return;
    }
    if (a.u[1]) {
        failure(s, "SQL execution error: Arrow error: Divide by zero error. Expression: '" + s.arg + "'");
        return;
    }
    const double satisfied = (double)a.u[0], total = (double)a.u[2];
    if (total == 0.0) {
        skipped(s, "No data to validate");
        return;
    }
    const double ratio = satisfied / total;
    if (ratio == 1.0) {
        success_metric(s, ratio);
        return;
    }
    const int64_t failed = (int64_t)(total - satisfied);
    std::string msg = s.has_hint ? s.hint + " (" + std::to_string(failed) + " rows failed the condition)"
                                 : "Custom SQL condition not satisfied for " + std::to_string(failed) +
                                       " rows. Expression: '" + s.arg + "'";
    failure_metric(s, ratio, msg);
}

static void finalize_length(Plan& p, Slot& s) {
    const Agg& a = p.aggs[s.aggs[0]];
    if (a.err != TG_OK) {
        set_error(s, a);
        return;
    }
    const double rows = (double)a.u[2];
    if (rows == 0.0) {  // NULLIF(COUNT(*), 0) -> NULL ratio
        skipped(s, "No data to validate");
        return;
    }
    const double ratio = (double)(a.u[0] + a.u[1]) * 1.0 / rows;
    if (ratio >= 1.0) success_metric(s, ratio);
    else failure_metric(s, ratio, "Length constraint failed: " + fmt_f64_prec(ratio * 100.0, 2) + "% of values are " + s.arg);
}

// containment / non_negative share the shape: matching rows / non-null rows (values.rs:245-296, 363-414)
static void finalize_value_ratio(Plan& p, Slot& s, const char* what) {
    const Agg& pred = p.aggs[s.aggs[0]];
    const Agg& valid = p.aggs[s.aggs[1]];
    if (pred.err != TG_OK || valid.err != TG_OK) {
        set_error(s, pred.err != TG_OK ? pred : valid);
        return;
    }
    const double ok = (double)pred.u[0], total = (double)valid.u[1];
    if (total == 0.0) {
        skipped(s, "No non-null data to validate");
        return;
    }
    const double ratio = ok / total;
    if (ratio == 1.0) success_metric(s, ratio);
    else failure_metric(s, ratio, fmt_f64(total - ok) + what);
}

static void finalize_approx_distinct(Plan& p, Slot& s) {
    const Agg& a = p.aggs[s.aggs[0]];
    if (a.err != TG_OK) {
        set_error(s, a);
        return;
    }
    const double count = (double)a.u[1];  // 0 for an empty or all-NULL column (approx_count_distinct.rs:300-326)
    if (assertion_evaluate(s.assertion, count)) success_metric(s, count);
    else failure_metric(s, count, "Approximate distinct count " + fmt_f64(count) + " does not satisfy assertion " +
                                      assertion_description(s.assertion) + " for column '" + s.columns[0] + "'");
}

static void finalize_data_type(Plan& p, Slot& s) {
    const Agg& a = p.aggs[s.aggs[0]];
    if (a.err != TG_OK) {
        set_error(s, a);
        return;
    }
    const double matches = (double)a.u[0], total = (double)(a.u[2] - a.u[1]);  // non-null rows only (WHERE c IS NOT NULL)
    if (total == 0.0) {
        skipped(s, "No non-null data to validate");
        return;
    }
    const double ratio = matches / total;
    if (ratio >= s.threshold) success_metric(s, ratio);
    else failure_metric(s, ratio, "Data type conformance " + fmt_f64(ratio) + " is below threshold " + fmt_f64(s.threshold));
}

static void finalize_column_count(Plan& p, Slot& s) {
    const Agg& a = p.aggs[s.aggs[0]];
    if (a.err != TG_OK) {  // column_count.rs:47-53
        failure(s, "Constraint evaluation failed for 'column_count': Failed to access table 'data': " + a.err_msg);
        return;
    }
    const double n = (double)a.u[1];
    if (assertion_evaluate(s.assertion, n)) success_metric(s, n);
    else failure_metric(s, n, "Column count " + fmt_f64(n) + " does not satisfy assertion " + assertion_description(s.assertion));
}

static void finalize_fk(Plan& p, Slot& s) {
    const Agg& a = p.aggs[s.aggs[0]];
    if (a.err != TG_OK) {
        set_error(s, a);
        return;
    }
    const int64_t total = (int64_t)a.u[0], unique = (int64_t)a.u[1];
    if (total == 0) {
        s.status = TG_SUCCESS;
        s.has_metric = false;
        s.has_message = false;
        return;
    }
    std::vector<std::string> ex;
    if (a.blob.size() >= 8) {
        uint64_t c;
        memcpy(&c, a.blob.data(), 8);
        const uint8_t* q = a.blob.data() + 8;
        for (uint64_t i = 0; i < c; ++i) {
            uint32_t L;
            memcpy(&L, q, 4);
            ex.emplace_back((const char*)q + 4, L);
            q += 4 + L;
        }
    }
    std::string msg = "Foreign key constraint violation: " + std::to_string(total) + " values in '" + s.columns[0] +
                      "' do not exist in '" + s.columns[1] + "' (total: " + std::to_string(total) +
                      ", unique: " + std::to_string(unique) + ")";
    if (!ex.empty()) {
        std::string es;
        if (ex.size() <= 5) es = join(ex, ", ");
        else {
            std::vector<std::string> first(ex.begin(), ex.begin() + 5);
            es = join(first, ", ") + ", ... (" + std::to_string(ex.size() - 5) + " more)";
        }
        msg += ". Examples: [" + es + "]";
    }
    failure_metric(s, (double)total, msg);
}

static void analyzer_error(Slot& s, const Agg& a) {
    s.ares.error = 2;
    s.ares.metric_kind = 3;
    s.has_message = true;
    s.message = a.err_msg;
}

static void finalize_analyzer(Plan& p, Slot& s) {
    const Agg& a = p.aggs[s.aggs[0]];
    tg_analyzer_result& r = s.ares;
    r = tg_analyzer_result{};
    s.map.clear();
    s.has_message = false;
    if (a.err != TG_OK) {
        analyzer_error(s, a);
        return;
    }
    switch (s.sub_kind) {
        case TG_AN_SIZE:
            r.u[0] = a.u[0];
            r.metric_kind = 1;
            r.metric_long = (int64_t)a.u[0];
            r.metric_double = (double)a.u[0];
            break;
        case TG_AN_COMPLETENESS:
            r.u[0] = a.u[0];
            r.u[1] = a.u[1];
            r.metric_kind = 0;
            r.metric_double = a.u[0] == 0 ? 1.0 : (double)a.u[1] / (double)a.u[0];
            break;
        case TG_AN_APPROX_COUNT_DISTINCT:  // state {approx_distinct_count, total_count = COUNT(c)}; metric Long
            r.u[0] = a.u[1];
            r.u[1] = a.u[0] - a.u[3];
            r.metric_kind = 1;
            r.metric_long = (int64_t)a.u[1];
            break;
        case TG_AN_DISTINCTNESS: {
            // COUNT(c), COUNT(DISTINCT c): denominator is the non-null count (distinctness.rs:113-116)
            const uint64_t nonnull = a.u[0] - a.u[3];
            r.u[0] = nonnull;
            r.u[1] = a.u[1];
            r.metric_kind = 0;
            r.metric_double = nonnull == 0 ? 1.0 : (double)a.u[1] / (double)nonnull;
        } break;
        case TG_AN_MEAN:
            if (a.u[4]) {  // SUM(Int64) is Int64: the reference fails its Float64 downcast (mean.rs:119-125)
                r.error = 2;
                r.metric_kind = 3;
                s.has_message = true;
                s.message = "Invalid data: Expected Float64 array for sum";
                break;
            }
            r.f[0] = a.f[5];
            r.u[0] = a.u[0];
            if (a.u[0] == 0) {
                r.error = 1;
                r.metric_kind = 3;
            } else {
                r.metric_kind = 0;
                r.metric_double = a.f[5] / (double)a.u[0];
            }
            break;
        case TG_AN_MIN:
        case TG_AN_MAX: {
            if (a.narrow & 1) {  // min_max.rs:112-131: neither Float64 nor Int64
                r.error = 2;
                r.metric_kind = 3;
                s.has_message = true;
                s.message = std::string("Invalid data: Expected numeric array for ") + (s.sub_kind == TG_AN_MIN ? "min" : "max") + ", got " +
                            a.narrow_name;
                break;
            }
            const bool has = a.u[0] > 0;
            r.u[0] = r.u[1] = has;
            r.f[0] = a.u[4] ? (double)(int64_t)a.u[2] : a.f[3];
            r.f[1] = a.u[4] ? (double)(int64_t)a.u[3] : a.f[4];
            if (!has) {
                r.error = 1;
                r.metric_kind = 3;
            } else {
                r.metric_kind = 0;
                r.metric_double = s.sub_kind == TG_AN_MIN ? r.f[0] : r.f[1];
            }
        } break;
        case TG_AN_SUM:
            r.f[0] = a.u[4] ? (double)(int64_t)a.u[1] : a.f[5];
            r.u[0] = a.u[0] > 0;
            if (a.u[0] == 0) {
                r.f[0] = 0.0;
                r.error = 1;
                r.metric_kind = 3;
            } else {
                r.metric_kind = 0;
                r.metric_double = r.f[0];
            }
            break;
        case TG_AN_STDDEV: {
            // state fields as COUNT, SUM, SUM(c*c), AVG would give them (standard_deviation.rs:171-180)
            const double n = (double)a.u[0], K = a.f[0];
            r.u[0] = a.u[0];
            r.f[0] = a.f[5];
            r.f[1] = a.f[2] + 2.0 * K * a.f[1] + n * K * K;
            r.f[2] = a.u[0] ? a.f[5] / n : 0.0;
            if (a.u[0] == 0) {
                r.error = 1;
                r.metric_kind = 3;
                break;
            }
            r.metric_kind = 2;
            // metric map (standard_deviation.rs:239-279) from the shifted moments (better conditioned than
            // the reference's E[x^2]-E[x]^2, equal to it in exact arithmetic)
            const double m2 = central_m2(n, a.f[1], a.f[2]);
            const double pop_var = m2 / n;
            s.map.emplace_back("count", n);
            s.map.emplace_back("mean", r.f[2]);
            s.map.emplace_back("std_dev", std::sqrt(pop_var));
            s.map.emplace_back("variance", pop_var);
            if (a.u[0] > 1) {
                const double sv = m2 / (n - 1.0);
                s.map.emplace_back("sample_std_dev", std::sqrt(sv));
                s.map.emplace_back("sample_variance", sv);
            }
            if (std::fabs(r.f[2]) >= 2.220446049250313e-16)
                s.map.emplace_back("coefficient_of_variation", std::sqrt(pop_var) / std::fabs(r.f[2]));
            r.metric_double = std::sqrt(pop_var);
        } break;
        case TG_AN_CORR_PEARSON:
        case TG_AN_COVARIANCE:
        case TG_AN_CORR_SPEARMAN: {
            const double n = (double)a.u[0], Kx = a.f[0], Ky = a.f[1];
            r.u[0] = a.u[0];
            r.f[0] = a.f[2] + n * Kx;
            r.f[1] = a.f[3] + n * Ky;
            r.f[2] = a.f[4] + 2.0 * Kx * a.f[2] + n * Kx * Kx;
            r.f[3] = a.f[5] + 2.0 * Ky * a.f[3] + n * Ky * Ky;
            r.f[4] = a.f[6] + Kx * a.f[3] + Ky * a.f[2] + n * Kx * Ky;
            r.metric_kind = 0;
            if (a.u[0] < 2) {
                r.metric_double = NAN;  // correlation.rs:408-410
            } else if (s.sub_kind == TG_AN_COVARIANCE) {
                r.metric_double = (a.f[6] - a.f[2] * a.f[3] / n) / (n - 1.0);
            } else {
                const double num = n * a.f[6] - a.f[2] * a.f[3];
                const double den = std::sqrt((n * a.f[4] - a.f[2] * a.f[2]) * (n * a.f[5] - a.f[3] * a.f[3]));
                r.metric_double = (den == 0.0 || std::isnan(den)) ? 0.0 : num / den;
            }
        } break;
        case TG_AN_COMPLIANCE:
            if (a.u[1]) {
                r.error = 2;
                r.metric_kind = 3;
                s.has_message = true;
                s.message = "Arrow error: Divide by zero error";
                break;
            }
            r.u[0] = a.u[0];
            r.u[1] = a.u[2];
            r.metric_kind = 0;
            r.metric_double = a.u[2] == 0 ? 1.0 : (double)a.u[0] / (double)a.u[2];
            break;
    }
}

static std::string quantile_key(double q) {
    // quantile_{p} with p printed as Rust prints f64 (docs/reference/analyzers.md:327-356)
    return "quantile_" + fmt_f64(q);
}

static void finalize_kll(Plan& p, Slot& s) {
    const Agg& a = p.aggs[s.aggs[0]];
    tg_analyzer_result& r = s.ares;
    r = tg_analyzer_result{};
    s.map.clear();
    s.has_message = false;
    if (a.err != TG_OK) {
        analyzer_error(s, a);
        return;
    }
    uint64_t n = 0;
    double mn = 0, mx = 0;
    kll_blob_summary(a.blob, &n, &mn, &mx);
    r.u[0] = n;
    r.f[0] = mn;
    r.f[1] = mx;
    if (n == 0) {
        r.error = 1;
        r.metric_kind = 3;
        return;
    }
    r.metric_kind = 2;
    s.map.emplace_back("count", (double)n);
    s.map.emplace_back("min", mn);
    s.map.emplace_back("max", mx);
    for (double q : s.quantiles) {
        double v = 0;
        kll_blob_query(a.blob, q, &v);
        s.map.emplace_back(quantile_key(q), v);
    }
}

// HistogramState {buckets, min_value, max_value, total_count, sum, sum_squared} and MetricValue::Histogram with
// mean / std_dev (analyzers/advanced/histogram.rs:78-115, 300-358). Map keys: min, max, mean, std_dev, total_count,
// sum, sum_squared, bucket_{i}.lower / .upper / .count.
static void finalize_histogram(Plan& p, Slot& s) {
    const Agg& num = p.aggs[s.aggs[0]];
    const Agg& h = p.aggs[s.aggs[1]];
    tg_analyzer_result& r = s.ares;
    r = tg_analyzer_result{};
    s.map.clear();
    s.has_message = false;
    if (num.err != TG_OK || h.err != TG_OK) {
        analyzer_error(s, num.err != TG_OK ? num : h);
        return;
    }
    if (h.u[7] && !num.u[4] && num.u[0]) {
        r.error = 2;
        r.metric_kind = 3;
        s.has_message = true;
        s.message = "histogram shards with different value ranges: run the second phase (tg_plan_histogram_rebucket / _install) before finalize";
        return;
    }
    if (num.u[4]) {  // MIN(Int64) is Int64: the reference fails its Float64 downcast (histogram.rs:203-208)
        r.error = 2;
        r.metric_kind = 3;
        s.has_message = true;
        s.message = "Invalid data: Expected Float64 for min";
        return;
    }
    r.metric_kind = 2;
    const uint64_t n = num.u[0];
    r.u[0] = n;
    if (n == 0) {  // "No data": empty bucket list, zero stats (histogram.rs:245-254)
        for (const char* k : {"min", "max", "mean", "std_dev", "total_count", "sum", "sum_squared"}) s.map.emplace_back(k, 0.0);
        return;
    }
    const double mn = num.f[3], mx = num.f[4], K = num.f[0];
    const double sum = num.f[5];
    const double sum_sq = num.f[2] + 2.0 * K * num.f[1] + (double)n * K * K;  // Σx² from the shifted sums
    r.f[0] = mn;
    r.f[1] = mx;
    r.f[2] = sum;
    r.f[3] = sum_sq;
    const double mean = sum / (double)n;
    // std_dev as the reference computes it from Σx² (histogram.rs:106-113); the shifted form avoids its cancellation
    const double var = n > 1 ? (num.f[2] / (double)n) - (num.f[1] / (double)n) * (num.f[1] / (double)n) : 0.0;
    s.map.emplace_back("min", mn);
    s.map.emplace_back("max", mx);
    s.map.emplace_back("mean", mean);
    s.map.emplace_back("std_dev", n > 1 ? std::sqrt(var < 0 ? 0.0 : var) : 0.0);
    s.map.emplace_back("total_count", (double)n);
    s.map.emplace_back("sum", sum);
    s.map.emplace_back("sum_squared", sum_sq);
    const int nb = s.k;
    const double range = mx - mn, width = (range > 0.0 && nb > 1) ? range / (double)nb : 1.0;
    for (int i = 0; i < nb; ++i) {
        const double lower = mn + ((double)i * width);
        const double upper = i == nb - 1 ? mx + width * 0.001 : mn + ((double)(i + 1) * width);
        uint64_t c = 0;
        if (h.blob.size() >= (size_t)(i + 1) * 8) memcpy(&c, h.blob.data() + (size_t)i * 8, 8);
        const std::string pre = "bucket_" + std::to_string(i);
        s.map.emplace_back(pre + ".lower", lower);
        s.map.emplace_back(pre + ".upper", upper);
        s.map.emplace_back(pre + ".count", (double)c);
    }
}

static void finalize_grouped(Plan& p, Slot& s) {
    const Agg& a = p.aggs[s.aggs[0]];
    tg_analyzer_result& r = s.ares;
    r = tg_analyzer_result{};
    s.map.clear();
    s.has_message = false;
    if (a.err != TG_OK) {
        analyzer_error(s, a);
        return;
    }
    // groups sorted by completeness DESC, LIMIT max_groups+1 (grouped_completeness.rs:131-139), then the
    // first max_groups kept; overall = sum over the kept groups (:191-194)
    struct G {
        const uint8_t* key;
        uint32_t len;
        uint64_t total, nn;
        double ratio;
    };
    std::vector<G> gs;
    std::vector<uint8_t> state = a.blob;
    grouped_blob_compact(state);  // entries of equal keys (one per merged shard) add up
    if (state.size() >= 8) {
        uint64_t n;
        memcpy(&n, state.data(), 8);
        gs.reserve((size_t)n);
        const uint8_t* q = state.data() + 8;
        for (uint64_t i = 0; i < n; ++i) {
            uint32_t L;
            memcpy(&L, q, 4);
            q += 4;
            G g;
            g.key = q;
            g.len = L;
            q += L;
            memcpy(&g.total, q, 8);
            memcpy(&g.nn, q + 8, 8);
            g.ratio = (double)g.nn * 1.0 / (double)g.total;
            q += 16;
            gs.push_back(g);
        }
    }
    std::stable_sort(gs.begin(), gs.end(), [](const G& x, const G& y) {
        if (x.ratio != y.ratio) return x.ratio > y.ratio;
        const int c = memcmp(x.key, y.key, std::min(x.len, y.len));  // std::string's order: unsigned bytes, then length
        return c != 0 ? c < 0 : x.len < y.len;
    });
    const size_t total_groups = gs.size();
    const bool truncated = gs.size() > (size_t)s.max_groups;
    if (truncated) gs.resize(s.max_groups);
    uint64_t ot = 0, on = 0;
    r.metric_kind = 2;
    s.map.reserve(gs.size() + 3);
    for (auto& g : gs) {
        std::string k((const char*)g.key, g.len);
        for (auto& ch : k)
            if (ch == '\x1f') ch = '_';  // GroupedMetrics::to_metric_value joins key parts with '_' (grouped.rs:135-156)
        s.map.emplace_back(std::move(k), g.total == 0 ? 1.0 : (double)g.nn / (double)g.total);
        ot += g.total;
        on += g.nn;
    }
    if (s.include_overall) s.map.emplace_back("__overall__", ot == 0 ? 1.0 : (double)on / (double)ot);
    s.map.emplace_back("__metadata__.total_groups", (double)std::min(total_groups, (size_t)s.max_groups + 1));
    s.map.emplace_back("__metadata__.truncated", truncated ? 1.0 : 0.0);
    r.u[0] = ot;
    r.u[1] = on;
    r.u[2] = gs.size();
    r.metric_double = ot == 0 ? 1.0 : (double)on / (double)ot;
}

// HistogramConstraint::evaluate (constraints/histogram.rs:208-413): buckets = the non-NULL values with their counts, ordered by
// count DESC, value ASC; metric = the entropy of the ratios count / (total - nulls), summed in that order; no bucket at all =>
// Skipped("No data to analyze"). The assertion is a closure over the Histogram: it stays on the host side of the boundary,
// which reads the buckets through tg_plan_map_entry (value -> count) and u[0..2] = {total_count, null_count, distinct_count}.
static void finalize_value_hist(Plan& p, Slot& s) {
    const Agg& a = p.aggs[s.aggs[0]];
    tg_analyzer_result& r = s.ares;
    r = tg_analyzer_result{};
    s.map.clear();
    if (a.err != TG_OK) {
        set_error(s, a);
        return;
    }
    struct G {
        const uint8_t* key;
        uint32_t len;
        uint64_t count;
    };
    std::vector<G> gs;
    std::vector<uint8_t> state = a.blob;
    grouped_blob_compact(state);
    uint64_t total = 0, nulls = 0;
    if (state.size() >= 8) {
        uint64_t n;
        memcpy(&n, state.data(), 8);
        const uint8_t* q = state.data() + 8;
        for (uint64_t i = 0; i < n; ++i) {
            uint32_t L;
            memcpy(&L, q, 4);
            q += 4;
            G g{q, L, 0};
            q += L;
            uint64_t tot, nn;
            memcpy(&tot, q, 8);
            memcpy(&nn, q + 8, 8);
            q += 16;
            total += tot;
            if (nn == 0) {  // the NULL group (the target IS the grouping column: every other group has nn == tot > 0)
                nulls += tot;
                continue;
            }
            g.count = tot;
            gs.push_back(g);
        }
    }
    std::stable_sort(gs.begin(), gs.end(), [](const G& x, const G& y) {
        if (x.count != y.count) return x.count > y.count;
        const int c = memcmp(x.key, y.key, std::min(x.len, y.len));
        return c != 0 ? c < 0 : x.len < y.len;
    });
    r.metric_kind = 2;
    r.u[0] = total;
    r.u[1] = nulls;
    r.u[2] = gs.size();
    if (gs.empty()) {
        skipped(s, "No data to analyze");
        return;
    }
    double entropy = 0.0;
    const double denom = (double)(int64_t)(total - nulls);
    s.map.reserve(gs.size());
    for (auto& g : gs) {
        const double ratio = (double)(int64_t)g.count * 1.0 / denom;
        if (ratio > 0.0) entropy += -ratio * log(ratio);
        s.map.emplace_back(std::string((const char*)g.key, g.len), (double)g.count);
    }
    r.metric_double = entropy;
    success_metric(s, entropy);  // provisional: the host applies the assertion closure (INTEGRATION.md)
}

void Plan::finalize() {
    for (auto& s : slots) {
        s.has_message = false;
        s.message.clear();
        s.has_metric = false;
        s.metric = 0;
        switch (s.kind) {
            case SL_COMPLETENESS: finalize_completeness(*this, s); break;
            case SL_SIZE: {
                const Agg& a = aggs[s.aggs[0]];
                if (a.err != TG_OK) {
                    set_error(s, a);
                    break;
                }
                const double n = (double)a.u[0];
                if (assertion_evaluate(s.assertion, n)) success_metric(s, n);
                else failure_metric(s, n, "Size " + fmt_f64(n) + " does not " + assertion_description(s.assertion));
            } break;
            case SL_STAT: finalize_stat(*this, s); break;
            case SL_MULTISTAT: finalize_multistat(*this, s); break;
            case SL_FORMAT: finalize_format(*this, s); break;
            case SL_UNIQ: finalize_uniq(*this, s); break;
            case SL_CORR: finalize_corr(*this, s); break;
            case SL_SQL: finalize_sql(*this, s); break;
            case SL_FK: finalize_fk(*this, s); break;
            case SL_ANALYZER: finalize_analyzer(*this, s); break;
            case SL_KLL: finalize_kll(*this, s); break;
            case SL_GROUPED: finalize_grouped(*this, s); break;
            case SL_VALUE_HIST: finalize_value_hist(*this, s); break;
            case SL_LENGTH: finalize_length(*this, s); break;
            case SL_CONTAINMENT: finalize_value_ratio(*this, s, " values are not in the allowed set"); break;
            case SL_NON_NEGATIVE: finalize_value_ratio(*this, s, " values are negative"); break;
            case SL_APPROX_DISTINCT: finalize_approx_distinct(*this, s); break;
            case SL_DATA_TYPE: finalize_data_type(*this, s); break;
            case SL_COLUMN_COUNT: finalize_column_count(*this, s); break;
            case SL_HISTOGRAM: finalize_histogram(*this, s); break;
            case SL_QUANTILE: finalize_quantile(*this, s); break;
        }
    }
    executed = true;
}

// ---- *State structs as serde_json writes them: fields in declaration order, u64 as integers, f64 through ryu,
// Option::None and non-finite floats as null, unit enum variants as strings ----
std::string analyzer_state_json(const Plan& p, int slot_index) {
    if (slot_index < 0 || slot_index >= (int)p.slots.size()) throw Error(TG_ERR_INVALID_ARG, "slot out of range");
    if (!p.executed) throw Error(TG_ERR_INVALID_ARG, "plan has not been executed");
    const Slot& s = p.slots[slot_index];
    const tg_analyzer_result& r = s.ares;
    auto U = [](uint64_t v) { return std::to_string(v); };
    auto opt = [](bool has, double v) { return has ? json_f64(v) : std::string("null"); };
    if (s.kind == SL_HISTOGRAM) {
        // HistogramState (advanced/histogram.rs:78-91); HistogramBucket {lower_bound, upper_bound, count}
        std::string out = "{\"buckets\":[";
        const int nb = r.u[0] ? s.k : 0;
        auto get = [&](const std::string& key) {
            for (auto& kv : s.map)
                if (kv.first == key) return kv.second;
            return 0.0;
        };
        for (int i = 0; i < nb; ++i) {
            const std::string pre = "bucket_" + std::to_string(i);
            if (i) out += ",";
            out += "{\"lower_bound\":" + json_f64(get(pre + ".lower")) + ",\"upper_bound\":" + json_f64(get(pre + ".upper")) +
                   ",\"count\":" + U((uint64_t)get(pre + ".count")) + "}";
        }
        out += "],\"min_value\":" + json_f64(r.f[0]) + ",\"max_value\":" + json_f64(r.f[1]) + ",\"total_count\":" + U(r.u[0]) +
               ",\"sum\":" + json_f64(r.f[2]) + ",\"sum_squared\":" + json_f64(r.f[3]) + "}";
        return out;
    }
    if (s.kind != SL_ANALYZER || r.error == 2) return "";
    switch (s.sub_kind) {
        case TG_AN_SIZE: return "{\"count\":" + U(r.u[0]) + "}";
        case TG_AN_COMPLETENESS: return "{\"total_count\":" + U(r.u[0]) + ",\"non_null_count\":" + U(r.u[1]) + "}";
        case TG_AN_DISTINCTNESS: return "{\"total_count\":" + U(r.u[0]) + ",\"distinct_count\":" + U(r.u[1]) + "}";
        case TG_AN_MEAN: return "{\"sum\":" + json_f64(r.f[0]) + ",\"count\":" + U(r.u[0]) + "}";
        case TG_AN_MIN:
        case TG_AN_MAX: return "{\"min\":" + opt(r.u[0] != 0, r.f[0]) + ",\"max\":" + opt(r.u[1] != 0, r.f[1]) + "}";
        case TG_AN_SUM: return "{\"sum\":" + json_f64(r.f[0]) + ",\"has_values\":" + (r.u[0] ? "true" : "false") + "}";
        case TG_AN_STDDEV:
            return "{\"count\":" + U(r.u[0]) + ",\"sum\":" + json_f64(r.f[0]) + ",\"sum_squared\":" + json_f64(r.f[1]) + ",\"mean\":" +
                   json_f64(r.f[2]) + "}";
        case TG_AN_CORR_PEARSON:
        case TG_AN_COVARIANCE:
            return "{\"n\":" + U(r.u[0]) + ",\"sum_x\":" + json_f64(r.f[0]) + ",\"sum_y\":" + json_f64(r.f[1]) + ",\"sum_x2\":" +
                   json_f64(r.f[2]) + ",\"sum_y2\":" + json_f64(r.f[3]) + ",\"sum_xy\":" + json_f64(r.f[4]) +
                   ",\"x_ranks\":null,\"y_ranks\":null,\"correlation_type\":\"" +
                   (s.sub_kind == TG_AN_CORR_PEARSON ? "Pearson" : "Covariance") + "\"}";
        case TG_AN_COMPLIANCE: return "{\"compliant_count\":" + U(r.u[0]) + ",\"total_count\":" + U(r.u[1]) + "}";
        case TG_AN_APPROX_COUNT_DISTINCT: return "{\"approx_distinct_count\":" + U(r.u[0]) + ",\"total_count\":" + U(r.u[1]) + "}";
        default: return "";  // Spearman keeps its rank vectors on the device; KLL / grouped states are blobs
    }
}

}  // namespace tg
