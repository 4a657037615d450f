/*
 * oracle.cpp — CPU oracle for the local-score hot path of ninalu/urlearning-cpp.
 *
 * TEST INFRASTRUCTURE ONLY (see oracle.h).  Plain C++17, no third-party
 * dependencies, compiled with -ffp-contract=off so float/double expressions
 * round exactly as written (the reference is built without FMA contraction).
 *
 * Citations are relative to /root/reference/urlearning/.
 */
#include "oracle.h"

#include <algorithm>
#include <cfloat>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <fstream>
#include <limits>
#include <map>
#include <sstream>
#include <string>
#include <thread>
#include <unordered_map>
#include <unordered_set>
#include <vector>

static thread_local std::string g_err;
static int fail(const std::string &m) { g_err = m; return -1; }

/* fx * 2^e rounded once to float32 (the device's bic_finalize): fx to double rounded to odd (truncated, the lowest bit set when
 * that dropped anything), then rounded to nearest float32 -- a correct single rounding also for |fx| >= 2^53, where
 * (float)(double)fx rounds twice */
static float fixed_to_float(int64_t fx, int e) {
    const uint64_t mag = fx < 0 ? -(uint64_t)fx : (uint64_t)fx;
    int drop = 0;
    while ((mag >> drop) >= ((uint64_t)1 << 53)) drop++;
    uint64_t kept = mag >> drop;
    if (drop && (mag & (((uint64_t)1 << drop) - 1))) kept |= 1;           /* sticky bit: round to odd */
    const double d = std::ldexp((double)kept, drop + e);                   /* exact: kept < 2^53 */
    return (float)(fx < 0 ? -d : d);
}
extern "C" const char *orc_last_error(void) { return g_err.c_str(); }

/* ------------------------------------------------------------------ helpers */

/* boost::algorithm::trim with the classic locale: std::isspace set */
static std::string trim(const std::string &s) {
    size_t a = 0, b = s.size();
    while (a < b && std::isspace((unsigned char)s[a])) a++;
    while (b > a && std::isspace((unsigned char)s[b - 1])) b--;
    return s.substr(a, b - a);
}

/* boost::split(record, s, is_any_of(delim), token_compress_on)  — record.h:35-39.
 * token_compress_on merges adjacent delimiters; a leading/trailing delimiter still yields an
 * empty first/last token. */
static std::vector<std::string> split_compress(const std::string &s, char delim) {
    std::vector<std::string> out;
    std::string cur;
    size_t i = 0;
    while (true) {
        if (i == s.size()) { out.push_back(cur); break; }
        if (s[i] == delim) {
            out.push_back(cur);
            cur.clear();
            while (i < s.size() && s[i] == delim) i++;
            continue;
        }
        cur.push_back(s[i++]);
    }
    return out;
}

/* typedefs.h:681-687 */
static inline int cardinality(uint64_t v) { return __builtin_popcountll(v); }

/* typedefs.h:692-697 (Gosper's hack) */
static inline uint64_t next_permutation(uint64_t vs) {
    uint64_t temp = (vs | (vs - 1)) + 1;
    return temp | ((((temp & -temp) / (vs & -vs)) >> 1) - 1);
}

/* ------------------------------------------------------------------ tables */

struct orc_table {
    int64_t n = 0;
    int p = 0;
    std::vector<std::string> names;
    std::vector<std::vector<std::string>> records;            /* n rows of p strings */
    std::vector<std::vector<std::string>> values;             /* per variable: values in first-appearance order */
    std::vector<std::vector<int32_t>> codes;                  /* per variable: n codes */
};

/* record_file.h:39-54 (getline + trim + Record), bayesian_network.cpp:25-42 (names),
 * variable.h:43-48,58-64 (value dictionary in order of first appearance) */
extern "C" orc_table *orc_read_csv(const char *path, char delimiter, int has_header) {
    std::ifstream file(path);
    if (!file.good()) { fail(std::string("cannot open input file '") + path + "'"); return nullptr; }
    auto *t = new orc_table();
    std::string line;
    std::vector<std::string> header;
    if (has_header) {
        std::getline(file, line);
        header = split_compress(trim(line), delimiter);
    }
    while (std::getline(file, line)) t->records.push_back(split_compress(trim(line), delimiter));
    t->n = (int64_t)t->records.size();
    if (t->n == 0) { fail("input file has no records"); delete t; return nullptr; }
    t->p = (int)t->records[0].size(); /* bayesian_network.cpp:27 */
    for (int64_t r = 0; r < t->n; r++)
        if ((int)t->records[r].size() < t->p) {
            /* the reference indexes out of range here (UB); the oracle refuses */
            fail("ragged record at data line " + std::to_string(r + 1));
            delete t;
            return nullptr;
        }
    for (int i = 0; i < t->p; i++) {
        if (has_header && i < (int)header.size()) t->names.push_back(header[i]);
        else t->names.push_back("Variable_" + std::to_string(i)); /* bayesian_network.cpp:35 */
    }
    t->values.resize(t->p);
    t->codes.resize(t->p);
    for (int i = 0; i < t->p; i++) {
        std::unordered_map<std::string, int32_t> idx;
        t->codes[i].resize(t->n);
        for (int64_t r = 0; r < t->n; r++) {
            const std::string &s = t->records[r][i];
            auto it = idx.find(s);
            if (it == idx.end()) {
                it = idx.emplace(s, (int32_t)t->values[i].size()).first;
                t->values[i].push_back(s);
            }
            t->codes[i][r] = it->second;
        }
    }
    return t;
}
extern "C" void orc_table_free(orc_table *t) { delete t; }
extern "C" int64_t orc_table_n(const orc_table *t) { return t->n; }
extern "C" int orc_table_p(const orc_table *t) { return t->p; }
extern "C" const char *orc_table_name(const orc_table *t, int v) { return t->names[v].c_str(); }
extern "C" void orc_table_card(const orc_table *t, int32_t *c) {
    for (int i = 0; i < t->p; i++) c[i] = (int32_t)t->values[i].size();
}
extern "C" int orc_table_codes(const orc_table *t, uint8_t *out) {
    for (int i = 0; i < t->p; i++) {
        if (t->values[i].size() > 256) return fail("arity > 256");
        for (int64_t r = 0; r < t->n; r++) out[(int64_t)i * t->n + r] = (uint8_t)t->codes[i][r];
    }
    return 0;
}
extern "C" void orc_table_values(const orc_table *t, double *x) {
    for (int i = 0; i < t->p; i++)
        for (int64_t r = 0; r < t->n; r++) x[(int64_t)i * t->n + r] = strtod(t->records[r][i].c_str(), nullptr);
}

/* ---------------------------------------------------------------- skeleton */

/* boost::tokenizer<char_separator<char>> with dropped delimiters, empty tokens dropped */
static std::vector<std::string> tokenize(const std::string &s, const char *seps) {
    std::vector<std::string> out;
    std::string cur;
    for (char c : s) {
        if (strchr(seps, c)) { if (!cur.empty()) { out.push_back(cur); cur.clear(); } }
        else cur.push_back(c);
    }
    if (!cur.empty()) out.push_back(cur);
    return out;
}

/* skeleton.cpp:58-105 (matrix) and :19-57 (.arc list); dispatch score_main.cpp:319-329 */
extern "C" int orc_read_skeleton(const char *path, int p, uint64_t *edges) {
    for (int i = 0; i < p; i++) edges[i] = 0;
    if (path == nullptr || path[0] == 0) return 0;
    std::string fn(path);
    std::ifstream in(fn.c_str());
    /* the reference silently keeps a 1-variable default skeleton here (SURVEY Q11); we refuse */
    if (!in.good()) return fail("cannot open skeleton file '" + fn + "'");
    auto add_edge = [&](int i, int j) -> bool {
        if (i < 0 || j < 0 || i >= p || j >= p) return false;
        edges[i] |= 1ULL << j;
        edges[j] |= 1ULL << i;
        return true;
    };
    std::string line;
    if (fn.find(".arc") + 4 == fn.size()) { /* score_main.cpp:321 */
        while (std::getline(in, line)) {
            auto tok = tokenize(line, ",");
            if (tok.size() < 2) continue;
            int v1 = tok[0].size() > 2 ? atoi(tok[0].c_str() + 2) : 0; /* skeleton.cpp:43-44 */
            int v2 = tok[1].size() > 2 ? atoi(tok[1].c_str() + 2) : 0;
            if (!add_edge(v1 - 1, v2 - 1)) return fail("arc list vertex out of range");
        }
        return 1;
    }
    int row = 0;
    bool first = true;
    while (std::getline(in, line)) {
        auto tok = tokenize(line, ", \n\r");
        if (first) { first = false; if ((int)tok.size() != p) return fail("skeleton matrix width != variable count"); }
        int col = 0;
        for (auto &s : tok) {
            /* skeleton.cpp:91 writes `abs(atof(x)) > 0.05` with no using-directive in scope, so GCC binds ::abs(int): the
             * value is truncated first and only |x| >= 1 (or "TRUE") makes an edge.  Pinned by oracle/_ref. */
            if (s == "TRUE" || std::abs((int)atof(s.c_str())) > 0.05) {
                if (!add_edge(row, col)) return fail("skeleton matrix entry out of range (row " + std::to_string(row) + ")");
            }
            col++;
        }
        row++; /* blank lines count as rows, skeleton.cpp:84-99 */
    }
    return 1;
}

extern "C" uint64_t orc_two_hop(const uint64_t *edges, int p, int initialised, int v) {
    uint64_t all = p >= 64 ? ~0ULL : ((1ULL << p) - 1);
    auto nb = [&](int i) { return initialised ? edges[i] : all; }; /* skeleton.hpp:57-60 */
    uint64_t orig = nb(v), out = orig;
    for (int j = 0; j < p; j++)
        if (((orig >> j) & 1) && j != v) out |= nb(j); /* score_main.cpp:149-153 */
    return out;
}

/* -------------------------------------------------------------- enumeration */

extern "C" int orc_effective_max_parents(int maxParents, int p, int64_t n, int is_bic) {
    if (maxParents > p || maxParents < 1) maxParents = p - 1; /* score_main.cpp:296-298 */
    if (is_bic) {
        int nn = (int)n;
        int maxParentCount = (int)std::log(2 * nn / std::log((double)nn)); /* :301 */
        if (maxParentCount < maxParents) maxParents = maxParentCount;
    }
    return maxParents;
}

extern "C" int64_t orc_enumerate(int v, uint64_t neighbors, int p, int maxParents, uint64_t *out, int64_t cap) {
    int64_t cnt = 0;
    auto emit = [&](uint64_t m) { if (out && cnt < cap) out[cnt] = m; cnt++; };
    emit(0); /* score_calculator.cpp:56-61 */
    std::vector<int> idx;
    for (int i = 0; i < p; i++) if ((neighbors >> i) & 1) idx.push_back(i); /* :65-74 */
    int nn = (int)idx.size();
    if (nn >= 63) { fail("too many neighbours for a 64-bit varset"); return -1; }
    for (int layer = 1; layer <= maxParents; layer++) { /* :78 */
        if (layer > nn) break; /* (1<<layer)-1 >= 1<<nn: loop body never runs */
        uint64_t compact = (1ULL << layer) - 1, max = 1ULL << nn; /* :83-89 */
        while (compact < max) {
            uint64_t vars = 0;
            for (int i = 0; i < nn; i++) if ((compact >> i) & 1) vars |= 1ULL << idx[i]; /* :93-98 */
            if (!((vars >> v) & 1)) emit(vars); /* :100 */
            compact = next_permutation(compact); /* :119 */
        }
    }
    return cnt;
}

/* ------------------------------------------------------------ discrete BIC */

/* log_likelihood_calculator.h:30-38 */
static std::vector<float> log_cache(int64_t recordCount) {
    std::vector<float> c;
    c.push_back(0.0f);
    for (int i = 1; i < recordCount + 2; i++) c.push_back((float)(i * std::log((double)i)));
    return c;
}

extern "C" int64_t orc_bic_cells(const int32_t *card, int p, int v, uint64_t parents) {
    __int128 cells = card[v];
    for (int i = 0; i < p; i++)
        if ((parents >> i) & 1) { cells *= card[i]; if (cells > ((__int128)1 << 40)) return -1; }
    return (int64_t)cells;
}

extern "C" int orc_bic_counts(const uint8_t *codes, int64_t n, int p, const int32_t *card, int v, uint64_t parents,
                              int32_t *counts) {
    int64_t cells = orc_bic_cells(card, p, v, parents);
    if (cells < 0) return fail("contingency table too large");
    std::fill(counts, counts + cells, 0);
    std::vector<const uint8_t *> col;
    std::vector<int64_t> stride;
    int64_t base = card[v];
    for (int i = 0; i < p; i++)
        if ((parents >> i) & 1) { col.push_back(codes + (int64_t)i * n); stride.push_back(base); base *= card[i]; }
    const uint8_t *cv = codes + (int64_t)v * n;
    for (int64_t r = 0; r < n; r++) {
        int64_t idx = cv[r];
        for (size_t j = 0; j < col.size(); j++) idx += stride[j] * col[j][r];
        counts[idx]++;
    }
    return 0;
}

/* bic_scoring_function.cpp:20-30 — float product in ascending variable order */
static float bic_t(const int32_t *card, int p, int v, uint64_t parents) {
    float penalty = card[v] - 1;
    for (int pa = 0; pa < p; pa++)
        if ((parents >> pa) & 1) penalty *= card[pa];
    return penalty;
}

struct BicCtx {
    const uint8_t *codes; int64_t n; int p; const int32_t *card;
    std::vector<float> ilogi; float base;
};
static BicCtx make_bic(const uint8_t *codes, int64_t n, int p, const int32_t *card) {
    BicCtx c{codes, n, p, card, log_cache(n), 0.f};
    c.base = std::log((double)(int)n) / 2; /* bic_scoring_function.cpp:13 (float member <- double) */
    return c;
}

static int bic_score_one(const BicCtx &c, int v, uint64_t parents, int mode, std::vector<int32_t> &counts,
                         float *score_out, double *ll_out) {
    int64_t cells = orc_bic_cells(c.card, c.p, v, parents);
    if (cells < 0) return fail("contingency table too large");
    counts.resize(cells);
    if (orc_bic_counts(c.codes, c.n, c.p, c.card, v, parents, counts.data())) return -1;
    const int rv = c.card[v];
    float tVal = bic_t(c.card, c.p, v, parents);
    float score;
    if (mode == 0) {
        /* SURVEY Q4: FP64 sum of float table entries is exact (addends are multiples of 2^-23, totals
         * < 2^28 at N<=1e6) -> order independent; the int64 fixed-point mirror checks that claim. */
        double ll = 0;
        int64_t fx = 0;
        for (int64_t j = 0; j < cells; j += rv) {
            int32_t nij = 0;
            for (int k = 0; k < rv; k++) {
                int32_t cnt = counts[j + k];
                nij += cnt;
                ll += (double)c.ilogi[cnt];
                fx += (int64_t)std::ldexp((double)c.ilogi[cnt], 23);
            }
            ll -= (double)c.ilogi[nij];
            fx -= (int64_t)std::ldexp((double)c.ilogi[nij], 23);
        }
        if (std::ldexp((double)fx, -23) != ll) return fail("FP64 accumulation was not exact (N too large?)");
        if (ll_out) *ll_out = ll;
        score = (float)ll;
    } else {
        /* literal: float running sum, contingency-tree DFS order = variables ascending by index with the
         * child interleaved at its index position, values ascending (log_likelihood_calculator.cpp:41-77);
         * then n_ij terms subtracted (in ascending paIdx order here; the reference's order is
         * boost::unordered_map iteration order, :32-34). */
        std::vector<int> vars; /* S u {v} ascending */
        for (int i = 0; i < c.p; i++) if (((parents >> i) & 1) || i == v) vars.push_back(i);
        std::vector<int64_t> stride(vars.size());
        int64_t b = rv;
        for (size_t j = 0; j < vars.size(); j++) {
            if (vars[j] == v) stride[j] = 1;
            else { stride[j] = b; b *= c.card[vars[j]]; }
        }
        score = 0;
        std::vector<int> digit(vars.size(), 0);
        /* odometer with the FIRST variable as the most significant digit = DFS order */
        while (true) {
            int64_t idx = 0;
            for (size_t j = 0; j < vars.size(); j++) idx += stride[j] * digit[j];
            if (counts[idx] > 0) score += c.ilogi[counts[idx]];
            int j = (int)vars.size() - 1;
            while (j >= 0 && ++digit[j] == c.card[vars[j]]) { digit[j] = 0; j--; }
            if (j < 0) break;
        }
        for (int64_t j = 0; j < cells; j += rv) {
            int32_t nij = 0;
            for (int k = 0; k < rv; k++) nij += counts[j + k];
            if (nij > 0) score -= c.ilogi[nij];
        }
        if (ll_out) *ll_out = score;
    }
    score -= tVal * c.base; /* bic_scoring_function.cpp:73 */
    *score_out = score;
    return 0;
}

extern "C" int orc_bic_score(const uint8_t *codes, int64_t n, int p, const int32_t *card, int v, uint64_t parents,
                             int mode, float *score_out, double *ll_out) {
    BicCtx c = make_bic(codes, n, p, card);
    std::vector<int32_t> counts;
    return bic_score_one(c, v, parents, mode, counts, score_out, ll_out);
}

extern "C" int orc_bic_score_many(const uint8_t *codes, int64_t n, int p, const int32_t *card, int v,
                                  const uint64_t *parents, int64_t n_sets, int mode, int threads, float *out) {
    BicCtx c = make_bic(codes, n, p, card);
    if (threads < 1) threads = 1;
    std::vector<int> rc(threads, 0);
    std::vector<std::string> errs(threads);
    auto work = [&](int t) {
        std::vector<int32_t> counts;
        for (int64_t i = t; i < n_sets; i += threads)
            if (bic_score_one(c, v, parents[i], mode, counts, &out[i], nullptr)) { rc[t] = -1; errs[t] = g_err; return; }
    };
    std::vector<std::thread> th;
    for (int t = 1; t < threads; t++) th.emplace_back(work, t);
    work(0);
    for (auto &x : th) x.join();
    for (int t = 0; t < threads; t++) if (rc[t]) return fail(errs[t]);
    return 0;
}

/* ------------------------------------------------------------ discrete fNML */

/* fnml_scoring_function.h: `r2_1000` — the K=2 multinomial regret for N <= 1000.  The reference holds 12-digit decimal
 * literals; as float32 they equal the exactly computed values in regret_r2.inc (tools/gen_regret_table.py,
 * tests/test_fnml_tables.py compares them with the reference's header when it is present). */
static const uint32_t k_r2_bits[1001] = {
#include "regret_r2.inc"
};
/* fnml_scoring_function.h: reg2 */
static float fnml_reg2(int N) {
    if (N <= 1000) { float f; memcpy(&f, &k_r2_bits[N], 4); return f; }
    const double pi = 3.1415926535897932384626433832795;
    return exp(0.5 * log(N * pi / 2) + sqrt(8 / (9 * N * pi)) + (1.0 / 12 - 4 / (9 * pi)) / N);
}
/* fnml_scoring_function.h: reg — float32 recurrence C(N,k) = C(N,k-1) + C(N,k-2) / (k-2) * N */
static float fnml_reg(int N, int K) {
    if (K == 1) return 1.0;
    else if (K == 2) return fnml_reg2(N);
    float rk_2 = fnml_reg(N, 1);
    float rk_1 = fnml_reg(N, 2);
    float rk = 0;
    for (int k = 3; k <= K; ++k) {
        rk = rk_1 + rk_2 / (k - 2) * N;
        rk_2 = rk_1;
        rk_1 = rk;
    }
    return rk;
}
/* fnml_scoring_function.h: getRegretCache — one row: out[N] = (float)log(reg(N, r)), N = 0..n_max */
extern "C" void orc_log_regret(int64_t n_max, int r, float *out) {
    /* log(float) in C++ is the float overload (logf): the reference includes <math.h> and passes reg()'s float result */
    for (int64_t N = 0; N <= n_max; N++) out[N] = std::log(fnml_reg((int)N, r));
}

struct FnmlCtx { BicCtx b; std::vector<std::vector<float>> regret; /* by arity, built on demand */ };
static const std::vector<float> &fnml_row(FnmlCtx &c, int r) {
    if ((int)c.regret.size() <= r) c.regret.resize(r + 1);
    if (c.regret[r].empty()) { c.regret[r].resize(c.b.n + 1); orc_log_regret(c.b.n, r, c.regret[r].data()); }
    return c.regret[r];
}

/* fnml_scoring_function.cpp:28-74 with enableDeCamposPruning off (score_main.cpp:112): LL - sum_j regret[r_v][N_ij].
 * mode 0: the exact-integer contract (every float table entry in units of 2^-23, the regret entries rounded to that grid;
 *         one rounding to float32 at the end) — independent of summation order.
 * mode 1: literal float32: the log-likelihood as in orc_bic_score mode 1, tVal a float32 running sum over the parent
 *         configurations with a positive count (ascending paIdx here; boost::unordered_map order there), score -= tVal. */
static int fnml_score_one(const BicCtx &c, const std::vector<float> &reg, int v, uint64_t parents, int mode, std::vector<int32_t> &counts, float *score_out) {
    int64_t cells = orc_bic_cells(c.card, c.p, v, parents);
    if (cells < 0) return fail("contingency table too large");
    counts.resize(cells);
    if (orc_bic_counts(c.codes, c.n, c.p, c.card, v, parents, counts.data())) return -1;
    const int rv = c.card[v];
    if (mode == 0) {
        int64_t fx = 0;
        for (int64_t j = 0; j < cells; j += rv) {
            int32_t nij = 0;
            for (int k = 0; k < rv; k++) {
                int32_t cnt = counts[j + k];
                nij += cnt;
                fx += (int64_t)std::ldexp((double)c.ilogi[cnt], 23);
            }
            if (nij > 0) {
                fx -= (int64_t)std::ldexp((double)c.ilogi[nij], 23);
                fx -= std::llrint(std::ldexp((double)reg[nij], 23));
            }
        }
        *score_out = fixed_to_float(fx, -23);
        return 0;
    }
    float ll;
    { /* the log-likelihood of orc_bic_score mode 1 (penalty removed again would round twice: recompute) */
        std::vector<int> vars;
        for (int i = 0; i < c.p; i++) if (((parents >> i) & 1) || i == v) vars.push_back(i);
        std::vector<int64_t> stride(vars.size());
        int64_t b = rv;
        for (size_t j = 0; j < vars.size(); j++) {
            if (vars[j] == v) stride[j] = 1;
            else { stride[j] = b; b *= c.card[vars[j]]; }
        }
        float score = 0;
        std::vector<int> digit(vars.size(), 0);
        while (true) {
            int64_t idx = 0;
            for (size_t j = 0; j < vars.size(); j++) idx += stride[j] * digit[j];
            if (counts[idx] > 0) score += c.ilogi[counts[idx]];
            int j = (int)vars.size() - 1;
            while (j >= 0 && ++digit[j] == c.card[vars[j]]) { digit[j] = 0; j--; }
            if (j < 0) break;
        }
        for (int64_t j = 0; j < cells; j += rv) {
            int32_t nij = 0;
            for (int k = 0; k < rv; k++) nij += counts[j + k];
            if (nij > 0) score -= c.ilogi[nij];
        }
        ll = score;
    }
    float t = 0;
    for (int64_t j = 0; j < cells; j += rv) {
        int32_t nij = 0;
        for (int k = 0; k < rv; k++) nij += counts[j + k];
        if (nij > 0) t += reg[nij];
    }
    *score_out = ll - t;
    return 0;
}

extern "C" int orc_fnml_score_many(const uint8_t *codes, int64_t n, int p, const int32_t *card, int v,
                                   const uint64_t *parents, int64_t n_sets, int mode, int threads, float *out) {
    FnmlCtx c{make_bic(codes, n, p, card), {}};
    const std::vector<float> &reg = fnml_row(c, card[v]);
    if (threads < 1) threads = 1;
    std::vector<int> rc(threads, 0);
    std::vector<std::string> errs(threads);
    auto work = [&](int t) {
        std::vector<int32_t> counts;
        for (int64_t i = t; i < n_sets; i += threads)
            if (fnml_score_one(c.b, reg, v, parents[i], mode, counts, &out[i])) { rc[t] = -1; errs[t] = g_err; return; }
    };
    std::vector<std::thread> th;
    for (int t = 1; t < threads; t++) th.emplace_back(work, t);
    work(0);
    for (auto &x : th) x.join();
    for (int t = 0; t < threads; t++) if (rc[t]) return fail(errs[t]);
    return 0;
}

/* ------------------------------------------------------------ discrete BDeu */

/* bdeu_scoring_function.cpp:25-123 with enableDeCamposPruning off (score_main.cpp:112).
 *   lg (:25-37): r = prod card(pa) (int); a_ij = ess / r (float / int); lg_ij = lgamma(a_ij) stored as float; a_ijk likewise
 *   calculate (:125-168): every non-empty cell: score -= lg_ijk; score += (float)lgamma(a_ijk + n_ijk)   (float + int addition)
 *   :115-118: every non-empty parent configuration: score += lg_ij; score -= lgamma(a_ij + n_ij)
 * mode 0: every bracket [temp - lg_ijk], [lg_ij - lgamma(.)] in FP64, rounded to the 2^-30 grid, summed exactly, one final
 *         rounding to float32 — the order-independent contract the device implements (bic_kernels.cuh score_configs_bdeu).
 * mode 1: literal float32 running sum with lgammaf (lgamma(float) under <math.h> in C++ is the float overload): cells in
 *         contingency-tree DFS order, then configurations in ascending paIdx (boost::unordered_map order there). */
static int bdeu_score_one(const BicCtx &c, float ess, int v, uint64_t parents, int mode, std::vector<int32_t> &counts, float *score_out) {
    int64_t cells = orc_bic_cells(c.card, c.p, v, parents);
    if (cells < 0) return fail("contingency table too large");
    counts.resize(cells);
    if (orc_bic_counts(c.codes, c.n, c.p, c.card, v, parents, counts.data())) return -1;
    const int rv = c.card[v];
    int r = 1;
    for (int pa = 0; pa < c.p; pa++) if ((parents >> pa) & 1) r *= c.card[pa];
    const float a_ij = ess / r;
    int sg;
    const float lg_ij = lgamma_r(a_ij, &sg);
    r *= rv;
    const float a_ijk = ess / r;
    const float lg_ijk = lgamma_r(a_ijk, &sg);
    if (mode == 0) {
        int64_t fx = 0;
        for (int64_t j = 0; j < cells; j += rv) {
            int32_t nij = 0;
            for (int k = 0; k < rv; k++) {
                const int32_t cnt = counts[j + k];
                nij += cnt;
                if (cnt > 0) {
                    const float temp = lgamma_r(a_ijk + cnt, &sg);
                    fx += std::llrint(((double)temp - (double)lg_ijk) * 1073741824.0);
                }
            }
            if (nij > 0) fx += std::llrint(((double)lg_ij - lgamma_r(a_ij + nij, &sg)) * 1073741824.0);
        }
        *score_out = fixed_to_float(fx, -30);
        return 0;
    }
    std::vector<int> vars;
    for (int i = 0; i < c.p; i++) if (((parents >> i) & 1) || i == v) vars.push_back(i);
    std::vector<int64_t> stride(vars.size());
    int64_t b = rv;
    for (size_t j = 0; j < vars.size(); j++) {
        if (vars[j] == v) stride[j] = 1;
        else { stride[j] = b; b *= c.card[vars[j]]; }
    }
    /* the reference's calls are lgamma(float): under <math.h> in C++ that is the float overload, lgammaf */
    const float lg_ij_f = lgammaf_r(a_ij, &sg), lg_ijk_f = lgammaf_r(a_ijk, &sg);
    float score = 0;
    std::vector<int> digit(vars.size(), 0);
    while (true) {
        int64_t idx = 0;
        for (size_t j = 0; j < vars.size(); j++) idx += stride[j] * digit[j];
        if (counts[idx] > 0) {
            float temp = lgammaf_r(a_ijk + counts[idx], &sg);
            score -= lg_ijk_f;
            score += temp;
        }
        int j = (int)vars.size() - 1;
        while (j >= 0 && ++digit[j] == c.card[vars[j]]) { digit[j] = 0; j--; }
        if (j < 0) break;
    }
    for (int64_t j = 0; j < cells; j += rv) {
        int32_t nij = 0;
        for (int k = 0; k < rv; k++) nij += counts[j + k];
        if (nij > 0) {
            score += lg_ij_f;
            score -= lgammaf_r(a_ij + nij, &sg);
        }
    }
    *score_out = score;
    return 0;
}

extern "C" int orc_bdeu_score_many(const uint8_t *codes, int64_t n, int p, const int32_t *card, int v, float ess,
                                   const uint64_t *parents, int64_t n_sets, int mode, int threads, float *out) {
    BicCtx c = make_bic(codes, n, p, card);
    if (threads < 1) threads = 1;
    std::vector<int> rc(threads, 0);
    std::vector<std::string> errs(threads);
    auto work = [&](int t) {
        std::vector<int32_t> counts;
        for (int64_t i = t; i < n_sets; i += threads)
            if (bdeu_score_one(c, ess, v, parents[i], mode, counts, &out[i])) { rc[t] = -1; errs[t] = g_err; return; }
    };
    std::vector<std::thread> th;
    for (int t = 1; t < threads; t++) th.emplace_back(work, t);
    work(0);
    for (auto &x : th) x.join();
    for (int t = 0; t < threads; t++) if (rc[t]) return fail(errs[t]);
    return 0;
}

/* --------------------------------------------------------- continuous cBIC */

/* arma::mean (arrayops::accumulate: two running sums over even/odd elements, then /n) */
static double arma_mean(const double *x, int64_t n) {
    double a1 = 0, a2 = 0;
    int64_t i, j;
    for (i = 0, j = 1; j < n; i += 2, j += 2) { a1 += x[i]; a2 += x[j]; }
    if (i < n) a1 += x[i];
    return (a1 + a2) / (double)n;
}
/* arma::var, norm_type 0 (N-1): op_var::direct_var */
static double arma_var(const double *x, int64_t n) {
    if (n < 2) return 0;
    double m = arma_mean(x, n), acc2 = 0, acc3 = 0;
    for (int64_t i = 0; i < n; i++) { double t = m - x[i]; acc2 += t * t; acc3 += t; }
    return (acc2 - acc3 * acc3 / (double)n) / (double)(n - 1);
}

/* BIC_OLS.cpp:66-80 */
extern "C" void orc_standardise(const double *x, int64_t n, int p, double *z) {
    std::vector<double> c(n);
    for (int i = 0; i < p; i++) {
        const double *col = x + (int64_t)i * n;
        double mean_x = arma_mean(col, n);
        for (int64_t j = 0; j < n; j++) c[j] = col[j] - mean_x; /* x -= mean_x */
        double dev = std::sqrt(arma_var(c.data(), n));
        for (int64_t j = 0; j < n; j++) z[(int64_t)i * n + j] = (col[j] - mean_x) / dev; /* :76-77 */
    }
}

extern "C" void orc_gram(const double *z, int64_t n, int p, double *g) {
    for (int a = 0; a < p; a++)
        for (int b = a; b < p; b++) {
            const double *x = z + (int64_t)a * n, *y = z + (int64_t)b * n;
            long double s = 0; /* extended accumulation: this is the yardstick the GPU Gram is held to */
            for (int64_t r = 0; r < n; r++) s += (long double)x[r] * y[r];
            g[a * p + b] = g[b * p + a] = (double)s;
        }
}

/* arma::solve for a square system: LU with partial pivoting (LAPACK dgesv semantics) */
static bool solve_lu(std::vector<double> &a, std::vector<double> &b, int k) {
    for (int c = 0; c < k; c++) {
        int piv = c;
        for (int r = c + 1; r < k; r++) if (std::fabs(a[r * k + c]) > std::fabs(a[piv * k + c])) piv = r;
        if (a[piv * k + c] == 0) return false;
        if (piv != c) { for (int j = 0; j < k; j++) std::swap(a[c * k + j], a[piv * k + j]); std::swap(b[c], b[piv]); }
        for (int r = c + 1; r < k; r++) {
            double f = a[r * k + c] / a[c * k + c];
            for (int j = c; j < k; j++) a[r * k + j] -= f * a[c * k + j];
            b[r] -= f * b[c];
        }
    }
    for (int r = k - 1; r >= 0; r--) {
        double s = b[r];
        for (int j = r + 1; j < k; j++) s -= a[r * k + j] * b[j];
        b[r] = s / a[r * k + r];
    }
    return true;
}

static std::vector<int> parent_list(int p, int v, uint64_t parents) {
    std::vector<int> pv;
    for (int i = 0; i < p; i++) if (i != v && ((parents >> i) & 1)) pv.push_back(i); /* BIC_OLS.cpp:289-297 */
    return pv;
}

/* BIC_OLS.cpp:277-389.  mlpack 3.x LinearRegression(X, Y, lambda=0, intercept=false):
 *   cov = X X^T ; beta = solve(cov, X Y^T) ; ComputeError = ||Y - beta^T X||^2 / n_points. */
extern "C" double orc_cbic_the_score_residual(const double *z, int64_t n, int p, int v, uint64_t parents, double lambda) {
    std::vector<int> pv = parent_list(p, v, parents);
    int k = (int)pv.size();
    if (k == 0) return 0.0; /* :302-305 */
    const double *y = z + (int64_t)v * n;
    std::vector<double> cov(k * k), rhs(k);
    for (int a = 0; a < k; a++) {
        const double *xa = z + (int64_t)pv[a] * n;
        for (int b = a; b < k; b++) {
            const double *xb = z + (int64_t)pv[b] * n;
            double s = 0;
            for (int64_t r = 0; r < n; r++) s += xa[r] * xb[r];
            cov[a * k + b] = cov[b * k + a] = s;
        }
        double s = 0;
        for (int64_t r = 0; r < n; r++) s += xa[r] * y[r];
        rhs[a] = s;
    }
    if (!solve_lu(cov, rhs, k)) return std::numeric_limits<double>::quiet_NaN();
    double cost = 0;
    for (int64_t r = 0; r < n; r++) {
        double pred = 0;
        for (int a = 0; a < k; a++) pred += rhs[a] * z[(int64_t)pv[a] * n + r];
        double t = y[r] - pred;
        cost += t * t;
    }
    double error_L2 = cost / (double)n;
    int num_err = (int)n;
    return num_err * std::log(error_L2) + lambda * std::log((double)num_err) * k - 0.0; /* :366 */
}

extern "C" double orc_cbic_the_score_gram(const double *g, int64_t n, int p, int v, uint64_t parents, double lambda) {
    std::vector<int> pv = parent_list(p, v, parents);
    int k = (int)pv.size();
    if (k == 0) return 0.0;
    /* Cholesky G_SS = L L^T, w = L^-1 g_Sv, RSS = G_vv - w.w */
    std::vector<double> L(k * k, 0.0), w(k);
    for (int i = 0; i < k; i++) {
        for (int j = 0; j <= i; j++) {
            double s = g[pv[i] * p + pv[j]];
            for (int t = 0; t < j; t++) s -= L[i * k + t] * L[j * k + t];
            if (i == j) L[i * k + i] = std::sqrt(s);
            else L[i * k + j] = s / L[j * k + j];
        }
        double s = g[pv[i] * p + v];
        for (int t = 0; t < i; t++) s -= L[i * k + t] * w[t];
        w[i] = s / L[i * k + i];
    }
    double rss = g[v * p + v];
    for (int i = 0; i < k; i++) rss -= w[i] * w[i];
    int num_err = (int)n;
    return num_err * std::log(rss / (double)n) + lambda * std::log((double)num_err) * k - 0.0;
}

typedef std::unordered_map<uint64_t, float> FloatMap;

/* BIC_OLS.cpp:125-172, literal, with arma::uvec(n) zero-filled (Armadillo >= 10.5; SURVEY Q5).
 * VARSET_CLEAR is XOR (typedefs.h:657). */
static float fbss_literal(uint64_t parents, FloatMap &cache, const std::vector<uint64_t> &parent_vec, int num_parents,
                          std::unordered_set<uint64_t> &checked, uint64_t &optimal_subset) {
    float best = 0;
    for (int idx = 0; idx < num_parents; idx++) {
        const int varIdx = (int)parent_vec[idx];
        uint64_t thin = parents;
        thin ^= (1ULL << varIdx);
        if (checked.find(thin) != checked.end()) continue;
        auto it = cache.find(thin);
        if (it != cache.end()) {
            if (it->second > best) { best = it->second; optimal_subset = it->first; }
        } else {
            std::vector<uint64_t> nv(num_parents - 1, 0);
            int j = 0;
            for (int i = 0; i < num_parents; i++) {
                if (varIdx == (int)parent_vec[i]) continue;
                nv[j++] = parent_vec[i];
                uint64_t the_subset = parents;
                float s = fbss_literal(thin, cache, nv, num_parents - 1, checked, the_subset);
                checked.insert(thin);
                if (s > best) { best = s; optimal_subset = the_subset; }
            }
        }
    }
    return best;
}

/* The evident intent of :125-172: best cached score among proper subsets reached by removing one
 * parent at a time, recursing only through sets that are NOT in the cache; never below 0. */
static float fbss_clean(uint64_t parents, const FloatMap &cache, std::unordered_map<uint64_t, float> &memo) {
    float best = 0;
    for (uint64_t m = parents; m; m &= m - 1) {
        uint64_t thin = parents & ~(m & -m);
        if (thin == 0) continue; /* checked is seeded with the empty set, :231 */
        auto it = cache.find(thin);
        float s;
        if (it != cache.end()) s = it->second;
        else {
            auto mm = memo.find(thin);
            if (mm != memo.end()) s = mm->second;
            else { s = fbss_clean(thin, cache, memo); memo[thin] = s; }
        }
        if (s > best) best = s;
    }
    return best;
}

extern "C" int orc_cbic_accept(int v, int p, const uint64_t *masks, const float *the_scores, int64_t n_sets,
                               int accept_mode, uint8_t *stored, float *value) {
    FloatMap cache;
    std::unordered_map<uint64_t, float> memo; /* F() of uncached sets; valid because layers ascend */
    for (int64_t i = 0; i < n_sets; i++) {
        uint64_t parents = masks[i];
        float the_score = the_scores[i];
        std::vector<uint64_t> pv;
        for (int j = 0; j < p; j++) if (j != v && ((parents >> j) & 1)) pv.push_back(j);
        int num_parents = (int)pv.size();
        pv.resize(p, 0); /* uvec(variableCount).fill(0), BIC_OLS.cpp:178-179 */
        stored[i] = 0;
        value[i] = -the_score;
        float ret;
        bool callee_stored = false;
        if (num_parents > 0 && the_score >= 0.0f) ret = -the_score; /* :213-224, bic_threshold = 0 (:57) */
        else {
            float best;
            if (accept_mode == 1) {
                std::unordered_set<uint64_t> checked;
                checked.insert(0);
                uint64_t subset = parents;
                best = fbss_literal(parents, cache, pv, num_parents, checked, subset);
            } else best = fbss_clean(parents, cache, memo);
            if (num_parents > 0 && best + 0.0f >= -the_score) ret = -the_score; /* :234-246 */
            else { cache[parents] = -the_score; callee_stored = true; ret = -the_score; } /* :249 */
        }
        /* caller: score_calculator.cpp:59-61 (empty: <1) and :111-113 (<0) */
        bool caller_stores = (parents == 0) ? (ret < 1) : (ret < 0);
        if (caller_stores) cache[parents] = ret;
        if (callee_stored || caller_stores) stored[i] = 1;
    }
    return 0;
}

/* ------------------------------------------------------------------- prune */

/* score_calculator.cpp:137-148 */
struct CompareSecond {
    bool operator()(const std::pair<uint64_t, float> &lhs, const std::pair<uint64_t, float> &rhs) const {
        float val = lhs.second - rhs.second;
        if (std::fabs(val) > 2 * std::numeric_limits<float>::epsilon()) return val > 0;
        return lhs.first < rhs.first;
    }
};

/* score_calculator.cpp:150-197 */
extern "C" int orc_prune(const uint64_t *masks, const float *scores, int64_t m, int highestCompletedLayer, uint8_t *keep) {
    std::vector<std::pair<uint64_t, float>> pairs(m);
    std::unordered_map<uint64_t, int64_t> pos;
    for (int64_t i = 0; i < m; i++) { pairs[i] = {masks[i], scores[i]}; pos[masks[i]] = i; keep[i] = 1; }
    std::sort(pairs.begin(), pairs.end(), CompareSecond());
    std::vector<char> pruned(m, 0);
    for (int64_t i = 0; i < m; i++) {
        if (pruned[i]) continue;
        uint64_t pi = pairs[i].first;
        if (cardinality(pi) > highestCompletedLayer) { pruned[i] = 1; continue; } /* marked, NOT erased (:177-180) */
        for (int64_t j = i + 1; j < m; j++) {
            if (pruned[j]) continue;
            uint64_t pj = pairs[j].first;
            if ((pi & pj) == pi) { pruned[j] = 1; keep[pos[pj]] = 0; } /* cache.erase(pj) */
        }
    }
    return 0;
}

/* -------------------------------------------------------------------- .pss */

static std::string lexical_float(float f) { /* boost::lexical_cast<std::string>(float): 9 significant digits */
    char buf[64];
    snprintf(buf, sizeof buf, "%.9g", (double)f);
    return buf;
}

extern "C" int64_t orc_score_file(const orc_options *o) {
    std::string sf(o->function ? o->function : "BIC");
    for (auto &ch : sf) ch = (char)std::tolower((unsigned char)ch); /* score_main.cpp:294 */
    const bool is_fnml = sf == "fnml", is_bdeu = sf == "bdeu";
    const bool log_bound = sf == "bic";                     /* score_main.cpp:300-304: only BIC bounds the parent limit */
    bool is_bic = sf == "bic" || is_fnml || is_bdeu, is_cbic = sf == "cbic";   /* is_bic: discrete input */
    if (!is_bic && !is_cbic) return fail("oracle supports -f BIC|fNML|BDeu|cBIC only");
    orc_table *t = orc_read_csv(o->input, o->delimiter ? o->delimiter : ',', o->has_header);
    if (!t) return -1;
    const int p = t->p;
    const int64_t n = t->n;
    if (p > 63) { orc_table_free(t); return fail("p > 63 is not representable in the reference (uint64 varset)"); }
    int maxParents = orc_effective_max_parents(o->max_parents, p, n, log_bound);
    std::vector<uint64_t> edges(p);
    int init = orc_read_skeleton(o->skeleton, p, edges.data());
    if (init < 0) { orc_table_free(t); return -1; }
    std::vector<int32_t> card(p);
    orc_table_card(t, card.data());
    std::vector<uint8_t> codes;
    std::vector<double> x, z, g;
    if (is_bic) {
        codes.resize((size_t)n * p);
        if (orc_table_codes(t, codes.data())) { orc_table_free(t); return -1; }
    } else {
        x.resize((size_t)n * p); z.resize((size_t)n * p);
        orc_table_values(t, x.data());
        orc_standardise(x.data(), n, p, z.data());
        if (o->cbic_from_gram) { g.resize((size_t)p * p); orc_gram(z.data(), n, p, g.data()); }
    }
    int threads = o->threads < 1 ? 1 : o->threads;
    std::vector<std::string> blocks(p);
    std::vector<int64_t> counts(p, 0);
    std::vector<int> rc(p, 0);
    std::vector<std::string> errs(p);
    auto do_var = [&](int v) {
        uint64_t nb = orc_two_hop(edges.data(), p, init, v);
        int64_t m = orc_enumerate(v, nb, p, maxParents, nullptr, 0);
        if (m < 0) { rc[v] = -1; errs[v] = g_err; return; }
        std::vector<uint64_t> masks(m);
        orc_enumerate(v, nb, p, maxParents, masks.data(), m);
        std::vector<float> val(m);
        std::vector<uint8_t> stored(m, 1);
        if (is_bic) {
            FnmlCtx fc{make_bic(codes.data(), n, p, card.data()), {}};
            const BicCtx &c = fc.b;
            const std::vector<float> *reg = is_fnml ? &fnml_row(fc, card[v]) : nullptr;
            std::vector<int32_t> cnt;
            for (int64_t i = 0; i < m; i++) {
                if (is_bdeu ? bdeu_score_one(c, o->ess > 0 ? o->ess : 1.0f, v, masks[i], o->bic_mode, cnt, &val[i])
                    : is_fnml ? fnml_score_one(c, *reg, v, masks[i], o->bic_mode, cnt, &val[i])
                            : bic_score_one(c, v, masks[i], o->bic_mode, cnt, &val[i], nullptr)) { rc[v] = -1; errs[v] = g_err; return; }
                stored[i] = masks[i] == 0 ? (val[i] < 1) : (val[i] < 0); /* score_calculator.cpp:59,111 */
            }
        } else {
            std::vector<float> ts(m);
            for (int64_t i = 0; i < m; i++)
                ts[i] = (float)(o->cbic_from_gram ? orc_cbic_the_score_gram(g.data(), n, p, v, masks[i], o->lambda)
                                                  : orc_cbic_the_score_residual(z.data(), n, p, v, masks[i], o->lambda));
            orc_cbic_accept(v, p, masks.data(), ts.data(), m, o->accept_mode, stored.data(), val.data());
        }
        /* compact to the stored entries */
        std::vector<uint64_t> km; std::vector<float> ks;
        for (int64_t i = 0; i < m; i++) if (stored[i]) { km.push_back(masks[i]); ks.push_back(val[i]); }
        if (o->prune) {
            std::vector<uint8_t> keep(km.size());
            orc_prune(km.data(), ks.data(), (int64_t)km.size(), maxParents, keep.data());
            std::vector<uint64_t> km2; std::vector<float> ks2;
            for (size_t i = 0; i < km.size(); i++) if (keep[i]) { km2.push_back(km[i]); ks2.push_back(ks[i]); }
            km.swap(km2); ks.swap(ks2);
        }
        /* canonical order (|S|, mask) — the reference's order is boost::unordered_map iteration order */
        std::vector<size_t> ord(km.size());
        for (size_t i = 0; i < ord.size(); i++) ord[i] = i;
        std::sort(ord.begin(), ord.end(), [&](size_t a, size_t b) {
            int ca = cardinality(km[a]), cb = cardinality(km[b]);
            return ca != cb ? ca < cb : km[a] < km[b];
        });
        std::string &out = blocks[v];
        char buf[64];
        out += "VAR " + t->names[v] + "\n"; /* score_main.cpp:177-178 */
        out += "META arity=" + std::to_string(card[v]) + "\n";
        for (size_t ii = 0; ii < ord.size(); ii++) {
            size_t i = ord[ii];
            snprintf(buf, sizeof buf, "%f ", ks[i]); /* :191 */
            out += buf;
            for (int q = 0; q < p; q++) if ((km[i] >> q) & 1) { out += t->names[q]; out += " "; }
            out += "\n";
        }
        out += "\n";
        counts[v] = (int64_t)km.size();
    };
    std::vector<std::thread> th;
    for (int tt = 0; tt < threads; tt++)
        th.emplace_back([&, tt]() { for (int v = 0; v < p; v++) if (v % threads == tt) do_var(v); }); /* :136-139 */
    for (auto &x2 : th) x2.join();
    for (int v = 0; v < p; v++) if (rc[v]) { orc_table_free(t); return fail(errs[v]); }
    std::ofstream out(o->output, std::ios_base::out | std::ios_base::binary);
    if (!out.good()) { orc_table_free(t); return fail("cannot open output file"); }
    /* score_main.cpp:387-388 */
    out << "META pss_version = 0.1\nMETA input_file=" << o->input << "\nMETA num_records=" << (int)n << "\n";
    out << "META parent_limit=" << maxParents << "\nMETA score_type=" << sf << "\nMETA ess=" << lexical_float(o->ess > 0 ? o->ess : 1.0f) << "\n\n";
    int64_t total = 0;
    for (int v = 0; v < p; v++) { out << blocks[v]; total += counts[v]; }
    out.close();
    orc_table_free(t);
    return total;
}
