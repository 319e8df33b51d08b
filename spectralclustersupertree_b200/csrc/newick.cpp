// Newick text straight into the flat forest store (SURVEY.md 8(f)-3).
//
// The reference reads its input with load_trees (/root/reference/src/sc_supertree/load.py:21-22: one
// cogent3.make_tree per line) and keeps PhyloNode objects; at 10^4 taxa x 10^3 trees that is 1.3 million
// Python objects before the first kernel runs.  scs_forest_parse_newick parses the same file into the arrays
// of scs_forest_create without building a node object.  Grammar and label rules are those of
// spectralclustersupertree_b200/tree.py::make_tree (the parser behind this package's load_trees), which
// follows what the reference's tests rely on from cogent3: ':x' is a branch length
// (tests/test_spectral_cluster_supertree.py:186-187), a numeric label on an internal node is its support
// (:217-219), any other internal label is a name (unused here), [comments] are skipped, labels may be quoted
// with ' or " (a doubled quote stands for itself).  Global taxon id = rank of the tip name among all tip
// names, sorted as Python sorts str (code point order = byte order of UTF-8).
//
// Lines are independent, so they are parsed by the host threads in parallel, each with its own name table;
// the tables are merged afterwards.

#include <algorithm>
#include <cerrno>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <new>
#include <string>
#include <charconv>
#include <unordered_map>
#include <vector>

#include <omp.h>

#include "forest.hpp"
#include "scs_b200.h"

namespace {

struct ParsedTree {
    std::vector<int32_t> parent, tip;  // tip: thread-local name id, -1 for internal nodes
    std::vector<double> length, support;
    int thread = 0;
};

struct NameTable {
    std::unordered_map<std::string, int32_t> id;
    std::vector<std::string> names;
    int32_t intern(const std::string &name) {
        auto it = id.find(name);
        if (it != id.end()) return it->second;
        const int32_t fresh = static_cast<int32_t>(names.size());
        id.emplace(name, fresh);
        names.push_back(name);
        return fresh;
    }
};

bool is_space(unsigned char c) { return c == ' ' || c == '\t' || c == '\n' || c == '\r' || c == '\v' || c == '\f'; }
bool is_struct(char c) { return c == '(' || c == ')' || c == ',' || c == ':' || c == ';'; }

// The common case first: a plain decimal number parsed in place by std::from_chars (correctly rounded like strtod, a
// fraction of its cost on 17-digit branch lengths).  Anything it does not consume whole -- a leading '+', blanks,
// hexadecimal forms -- is left to as_number below, which decides as before.
bool as_plain_number(const char *first, const char *last, double *out) {
    if (first == last) return false;
    const char c = *first;
    if (!((c >= '0' && c <= '9') || c == '-' || c == '.')) return false;  // inf / nan / '+...' take the slow path
    double v;
    const std::from_chars_result r = std::from_chars(first, last, v, std::chars_format::general);
    if (r.ec != std::errc() || r.ptr != last) return false;  // out of range: strtod's +-HUGE_VAL / 0 semantics below
    *out = v;
    return true;
}

// float(label) of Python for the forms that occur in Newick files; false if the label is not a number
bool as_number(const std::string &given, double *out) {
    if (given.empty()) return false;
    // float() allows single underscores between digits ("1_000.5"); strtod does not know them
    std::string stripped;
    if (given.find('_') != std::string::npos) {
        for (size_t i = 0; i < given.size(); ++i) {
            if (given[i] != '_') {
                stripped.push_back(given[i]);
                continue;
            }
            const bool between_digits = i > 0 && i + 1 < given.size() && given[i - 1] >= '0' && given[i - 1] <= '9' &&
                                        given[i + 1] >= '0' && given[i + 1] <= '9';
            if (!between_digits) return false;
        }
    }
    const std::string &label = stripped.empty() ? given : stripped;
    errno = 0;
    char *end = nullptr;
    const double v = std::strtod(label.c_str(), &end);
    if (end != label.c_str() + label.size()) return false;
    if (label.find_first_of("xXpP") != std::string::npos) return false;  // strtod takes hex floats, float() does not
    *out = v;
    return true;
}

// One line -> one tree.  Returns nullptr, or a static message describing the syntax error.
const char *parse_line(const char *s, const char *e, NameTable &table, ParsedTree &tree) {
    std::vector<int32_t> open;  // internal nodes whose ')' has not been seen yet
    int32_t cur = -1;           // completed node that a following label / length applies to
    bool expect_length = false, finished = false, has_root = false;
    std::vector<uint8_t> has_label;  // internal node already carries a name or a support value
    const double nan = std::nan("");
    auto new_node = [&](int32_t tip) -> int32_t {
        const int32_t k = static_cast<int32_t>(tree.parent.size());
        tree.parent.push_back(open.empty() ? -1 : open.back());
        tree.tip.push_back(tip);
        tree.length.push_back(nan);
        tree.support.push_back(nan);
        has_label.push_back(0);
        return k;
    };
    std::string label;
    const char *p = s;
    while (p < e) {
        const char ch = *p;
        char kind = 0;  // structural character, or 'L' for a label
        const char *plain_begin = nullptr, *plain_end = nullptr;  // an unquoted label, where it lies in the text
        if (is_struct(ch)) {
            kind = ch;
            ++p;
        } else if (is_space(static_cast<unsigned char>(ch))) {
            ++p;
            continue;
        } else if (ch == '[') {
            int depth = 1;
            ++p;
            while (p < e && depth) {
                depth += *p == '[';
                depth -= *p == ']';
                ++p;
            }
            if (depth) return "unterminated [comment]";
            continue;
        } else if (ch == '\'' || ch == '"') {
            label.clear();
            ++p;
            while (true) {
                if (p >= e) return "unterminated quoted label";
                if (*p == ch) {
                    if (p + 1 < e && p[1] == ch) {
                        label.push_back(ch);
                        p += 2;
                        continue;
                    }
                    ++p;
                    break;
                }
                label.push_back(*p++);
            }
            kind = 'L';
        } else {
            const char *q = p;
            while (q < e && !is_struct(*q) && *q != '[' && !is_space(static_cast<unsigned char>(*q))) ++q;
            plain_begin = p;
            plain_end = q;
            if (!expect_length) label.assign(p, q);
            p = q;
            kind = 'L';
        }
        if (finished) return "text after the final ';'";
        switch (kind) {
        case '(':
            if (cur >= 0) return "'(' directly after a node";
            if (open.empty() && has_root) return "more than one top-level node";
            has_root = true;
            open.push_back(new_node(-1));
            break;
        case ',':
            if (open.empty()) return "',' outside parentheses";
            if (cur < 0) new_node(table.intern(std::string()));
            cur = -1;
            expect_length = false;
            break;
        case ')':
            if (open.empty()) return "unbalanced ')'";
            if (cur < 0) new_node(table.intern(std::string()));
            cur = open.back();
            open.pop_back();
            expect_length = false;
            break;
        case ':':
            if (cur < 0) {
                if (open.empty() && has_root) return "more than one top-level node";
                has_root = true;
                cur = new_node(table.intern(std::string()));
            }
            expect_length = true;
            break;
        case ';':
            finished = true;
            break;
        default:  // a label
            if (expect_length) {
                double number;
                if (!(plain_begin && as_plain_number(plain_begin, plain_end, &number))) {
                    if (plain_begin) label.assign(plain_begin, plain_end);
                    if (!as_number(label, &number)) return "invalid branch length";
                }
                tree.length[cur] = number;
                expect_length = false;
            } else if (cur < 0) {
                if (open.empty() && has_root) return "more than one top-level node";
                has_root = true;
                cur = new_node(table.intern(label));
            } else if (tree.tip[cur] < 0 && !has_label[cur]) {
                double number;
                if (as_number(label, &number)) tree.support[cur] = number;
                has_label[cur] = 1;
            } else {
                return "unexpected label";
            }
        }
    }
    if (!open.empty()) return "unbalanced '('";
    if (!has_root) return "empty Newick string";
    return nullptr;
}

thread_local std::string g_parse_error;

}  // namespace

extern "C" {

const char *scs_newick_last_error(void) { return g_parse_error.c_str(); }

int scs_forest_parse_newick(const char *text, size_t bytes, scs_forest **out, char **names_out, size_t *names_bytes,
                            int *num_taxa_out) {
    if (!text || !out || !names_out || !names_bytes) return SCS_ERR_INVALID;
    *out = nullptr;
    *names_out = nullptr;
    *names_bytes = 0;
    g_parse_error.clear();
    // lines as Python's file iteration yields them: split at '\n', no empty line after a final newline
    std::vector<std::pair<size_t, size_t>> lines;
    for (size_t at = 0; at < bytes;) {
        const void *nl = std::memchr(text + at, '\n', bytes - at);
        const size_t end = nl ? static_cast<size_t>(static_cast<const char *>(nl) - text) : bytes;
        lines.emplace_back(at, end);
        at = end + 1;
    }
    const int T = static_cast<int>(lines.size());
    const int threads = std::max(1, std::min(scs_host_threads(), T));
    std::vector<ParsedTree> trees(static_cast<size_t>(T));
    std::vector<NameTable> tables(static_cast<size_t>(threads));
    int bad_line = -1;
    const char *bad_what = nullptr;
#pragma omp parallel for schedule(dynamic, 4) num_threads(threads) if (bytes > (1u << 16))
    for (int t = 0; t < T; ++t) {
        const int me = omp_get_thread_num();
        trees[t].thread = me;
        const char *err = parse_line(text + lines[t].first, text + lines[t].second, tables[me], trees[t]);
        if (err) {
#pragma omp critical(scs_newick_error)
            if (bad_line < 0 || t < bad_line) {
                bad_line = t;
                bad_what = err;
            }
        }
    }
    if (bad_line >= 0) {
        g_parse_error = "line " + std::to_string(bad_line + 1) + ": " + bad_what;
        return SCS_ERR_INPUT;
    }
    // global names: sorted, unique; per-thread map local id -> global id
    std::vector<std::string> names;
    for (const NameTable &tb : tables) names.insert(names.end(), tb.names.begin(), tb.names.end());
    std::sort(names.begin(), names.end());
    names.erase(std::unique(names.begin(), names.end()), names.end());
    std::vector<std::vector<int32_t>> global(tables.size());
    for (size_t w = 0; w < tables.size(); ++w) {
        global[w].resize(tables[w].names.size());
        for (size_t i = 0; i < tables[w].names.size(); ++i)
            global[w][i] = static_cast<int32_t>(std::lower_bound(names.begin(), names.end(), tables[w].names[i]) - names.begin());
    }
    std::vector<int64_t> offsets(static_cast<size_t>(T) + 1, 0);
    for (int t = 0; t < T; ++t) offsets[t + 1] = offsets[t] + static_cast<int64_t>(trees[t].parent.size());
    const int64_t M = offsets[T];
    std::vector<int32_t> parent(M), taxon(M);
    std::vector<double> length(M), support(M), weight(static_cast<size_t>(T), 1.0);
#pragma omp parallel for schedule(dynamic, 8) num_threads(threads) if (M > (1 << 16))
    for (int t = 0; t < T; ++t) {
        const ParsedTree &tr = trees[t];
        const int64_t base = offsets[t];
        const std::vector<int32_t> &map = global[tr.thread];
        for (size_t k = 0; k < tr.parent.size(); ++k) {
            parent[base + k] = tr.parent[k];
            // a node without children is a tip even if it was opened with '(' ... it cannot be: ')' adds one
            taxon[base + k] = tr.tip[k] >= 0 ? map[tr.tip[k]] : -1;
            length[base + k] = tr.length[k];
            support[base + k] = tr.support[k];
        }
    }
    const int rc = scs_forest_create(T, offsets.data(), parent.data(), length.data(), support.data(), taxon.data(),
                                     weight.data(), static_cast<int>(names.size()), out);
    if (rc) {
        g_parse_error = scs_forest_last_error();
        if (g_parse_error.empty()) g_parse_error = "the parsed trees are not a valid forest";
        return rc;
    }
    size_t total = 0;
    for (const std::string &nm : names) total += nm.size() + 1;
    char *buf = static_cast<char *>(std::malloc(total ? total : 1));
    if (!buf) {
        scs_forest_destroy(*out);
        *out = nullptr;
        return SCS_ERR_INVALID;
    }
    size_t at = 0;
    for (const std::string &nm : names) {  // NUL-separated: a name may contain any other byte
        std::memcpy(buf + at, nm.data(), nm.size());
        at += nm.size();
        buf[at++] = '\0';
    }
    *names_out = buf;
    *names_bytes = total;
    if (num_taxa_out) *num_taxa_out = static_cast<int>(names.size());
    return SCS_OK;
}

/* The flat supertree as Newick text, straight from the arrays (replaces building node objects for
 * PhyloNode.write, /root/reference/src/sc_supertree/cli.py:39): children in index order, tip labels quoted as
 * cogent3 quotes them (single quotes around a label with blanks or Newick punctuation, a quote doubled), no
 * branch lengths (the supertree has none), terminated by ';'. */
static int flat_tree_newick(int64_t num_nodes, const int32_t *parent, const int32_t *taxon, const char *names,
                            size_t names_bytes, int num_taxa, const double *value, int digits, char **text_out,
                            size_t *text_bytes) {
    if (num_nodes <= 0 || !parent || !taxon || !names || !text_out || !text_bytes || num_taxa < 0) return SCS_ERR_INVALID;
    if (value && (digits < 0 || digits > 17)) return SCS_ERR_INVALID;
    *text_out = nullptr;
    *text_bytes = 0;
    std::vector<const char *> label(static_cast<size_t>(num_taxa));
    std::vector<size_t> label_len(static_cast<size_t>(num_taxa));
    {
        size_t at = 0;
        for (int x = 0; x < num_taxa; ++x) {
            if (at >= names_bytes) return SCS_ERR_INVALID;
            label[x] = names + at;
            const void *end = std::memchr(names + at, '\0', names_bytes - at);
            if (!end) return SCS_ERR_INVALID;
            label_len[x] = static_cast<size_t>(static_cast<const char *>(end) - (names + at));
            at += label_len[x] + 1;
        }
    }
    // children of every node, in index order
    std::vector<int64_t> first(static_cast<size_t>(num_nodes) + 1, 0);
    if (parent[0] != -1) return SCS_ERR_INVALID;
    for (int64_t k = 1; k < num_nodes; ++k) {
        if (parent[k] < 0 || parent[k] >= k) return SCS_ERR_INVALID;
        first[parent[k] + 1] += 1;
    }
    for (int64_t k = 0; k < num_nodes; ++k) first[k + 1] += first[k];
    std::vector<int32_t> child(static_cast<size_t>(num_nodes));
    {
        std::vector<int64_t> cursor(first.begin(), first.end() - 1);
        for (int64_t k = 1; k < num_nodes; ++k) child[cursor[parent[k]]++] = static_cast<int32_t>(k);
    }
    std::string text;
    text.reserve(static_cast<size_t>(num_nodes) * 8);
    auto put_label = [&](int32_t x) {
        const char *s = label[x];
        const size_t n = label_len[x];
        bool plain = n > 0;
        for (size_t i = 0; i < n && plain; ++i) plain = std::strchr(" ()[]':;,\t\n", s[i]) == nullptr;
        if (plain || n == 0) {
            text.append(s, n);
            return;
        }
        text.push_back('\'');
        for (size_t i = 0; i < n; ++i) {
            if (s[i] == '\'') text.push_back('\'');
            text.push_back(s[i]);
        }
        text.push_back('\'');
    };
    // iterative depth-first walk: (node, next child to visit)
    std::vector<std::pair<int32_t, int64_t>> stack;
    stack.emplace_back(0, first[0]);
    if (first[1] == first[0]) {  // a single node
        if (taxon[0] >= 0 && taxon[0] < num_taxa) put_label(taxon[0]);
    } else {
        text.push_back('(');
        while (!stack.empty()) {
            auto &top = stack.back();
            const int32_t node = top.first;
            if (top.second == first[node + 1]) {
                text.push_back(')');
                if (value && node != 0 && std::isfinite(value[node])) {
                    char label[64];
                    const int len = std::snprintf(label, sizeof(label), "%.*f", digits, value[node]);
                    if (len < 0 || len >= static_cast<int>(sizeof(label))) return SCS_ERR_INVALID;
                    text.append(label, static_cast<size_t>(len));
                }
                stack.pop_back();
                continue;
            }
            if (top.second != first[node]) text.push_back(',');
            const int32_t c = child[top.second++];
            if (first[c + 1] == first[c]) {
                if (taxon[c] < 0 || taxon[c] >= num_taxa) return SCS_ERR_INVALID;
                put_label(taxon[c]);
            } else {
                text.push_back('(');
                stack.emplace_back(c, first[c]);
            }
        }
    }
    text.push_back(';');
    char *buf = static_cast<char *>(std::malloc(text.size() + 1));
    if (!buf) return SCS_ERR_INVALID;
    std::memcpy(buf, text.data(), text.size());
    buf[text.size()] = '\0';
    *text_out = buf;
    *text_bytes = text.size();
    return SCS_OK;
}

int scs_flat_tree_newick(int64_t num_nodes, const int32_t *parent, const int32_t *taxon, const char *names,
                         size_t names_bytes, int num_taxa, char **text_out, size_t *text_bytes) {
    return flat_tree_newick(num_nodes, parent, taxon, names, names_bytes, num_taxa, nullptr, 0, text_out, text_bytes);
}

/* The same with a numeric label after every internal non-root node whose value is finite: the support values of an
 * annotated supertree (scs_supertree_support), written as "%.*f" so that scs_forest_parse_newick reads them back as
 * supports. */
int scs_flat_tree_newick_values(int64_t num_nodes, const int32_t *parent, const int32_t *taxon, const char *names,
                                size_t names_bytes, int num_taxa, const double *value, int digits, char **text_out,
                                size_t *text_bytes) {
    if (!value) return SCS_ERR_INVALID;
    return flat_tree_newick(num_nodes, parent, taxon, names, names_bytes, num_taxa, value, digits, text_out, text_bytes);
}

void scs_free(void *ptr) { std::free(ptr); }

}  // extern "C"
