// ms-format gene trees for create_haplotypes (DESIGN.md section 10, "Gene trees"): the text's `//` blocks, one per
// chromosome; a block's tree lines, each an optional [n] prefix and one Newick tree; the regions the prefixes cut the
// chromosome into.  The Newick grammar and the node numbering are those of mutate.parse_newick (nodes in order of
// appearance, which is preorder), so that node indices, which address the draws, agree with the Python side.
#include <algorithm>
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <stdexcept>
#include <string>
#include <unordered_map>

#include "jlp_host.h"

namespace jlp {

namespace {

struct TreeLine {
    const char* s;              // the Newick text (after the prefix)
    uint64_t n;
    uint64_t len;               // the [n] prefix, 0 when absent
    uint64_t block, index;      // for messages
};

[[noreturn]] void fail(const std::string& m) { throw std::runtime_error(m); }

std::string where(const TreeLine& t) {
    return "block " + std::to_string(t.block + 1) + ", tree " + std::to_string(t.index + 1);
}

bool is_space(char ch) { return ch == ' ' || ch == '\t' || ch == '\n' || ch == '\r' || ch == '\v' || ch == '\f'; }

// one Newick tree as parse_newick reads it; labels of the childless nodes (the tips) go to tip_node by name
void parse_tree(const TreeLine& L, const std::unordered_map<std::string, uint32_t>& tip_of, uint32_t n_tips,
                uint32_t max_nodes, GeneTree& T) {
    const char* s = L.s;
    const uint64_t n = L.n;
    uint64_t i = 0;
    auto err = [&](const std::string& m) {
        fail("ms text, " + where(L) + ": Newick tree: " + m + " (at character " + std::to_string(i) + ")");
    };
    auto skip = [&]() {
        while (i < n) {
            if (is_space(s[i])) i++;
            else if (s[i] == '[') {
                const void* e = std::memchr(s + i, ']', n - i);
                if (!e) err("unterminated comment");
                i = (uint64_t)(static_cast<const char*>(e) - s) + 1;
            } else break;
        }
    };
    auto plain = [&](char ch) { return !std::strchr("(),:;[]'", ch) && !is_space(ch); };
    auto read_label = [&]() {
        skip();
        std::string out;
        if (i < n && s[i] == '\'') {
            i++;
            for (;;) {
                if (i >= n) err("unterminated quoted label");
                if (s[i] == '\'') {
                    if (i + 1 < n && s[i + 1] == '\'') { out += '\''; i += 2; continue; }
                    i++;
                    break;
                }
                out += s[i++];
            }
            return out;
        }
        const uint64_t j = i;
        while (i < n && plain(s[i])) i++;
        return std::string(s + j, i - j);
    };
    std::vector<std::string> label;
    std::vector<char> has_len;
    auto read_length = [&](uint32_t v) {
        skip();
        if (i < n && s[i] == ':') {
            i++;
            skip();
            const uint64_t j = i;
            while (i < n && plain(s[i])) i++;
            const std::string tok(s + j, i - j);
            char* end = nullptr;
            const double x = tok.empty() ? 0 : std::strtod(tok.c_str(), &end);
            if (tok.empty() || end != tok.c_str() + tok.size()) err("branch length '" + tok + "' is not a number");
            if (!std::isfinite(x)) err("branch length '" + tok + "' is not finite");
            T.branch_len[v] = x;
            has_len[v] = 1;
        }
    };
    auto add = [&](int32_t par) {
        if (T.parent.size() >= max_nodes) err("more than " + std::to_string(max_nodes) + " nodes");
        T.parent.push_back(par);
        T.branch_len.push_back(0.0);
        label.emplace_back();
        has_len.push_back(0);
        return (uint32_t)(T.parent.size() - 1);
    };
    skip();
    if (i >= n || s[i] != '(') err("the tree must start with '(' (a tree of more than one node)");
    std::vector<uint32_t> stack{add(-1)};
    i++;
    for (;;) {                                   // at the start of a child of stack.back()
        skip();
        if (i < n && s[i] == '(') {
            stack.push_back(add((int32_t)stack.back()));
            i++;
            continue;
        }
        uint32_t v = add((int32_t)stack.back());
        label[v] = read_label();
        if (label[v].empty()) err("every tip needs a label");
        read_length(v);
        for (;;) {                               // after a child
            skip();
            if (i >= n) err("unexpected end of the tree");
            if (s[i] == ',') { i++; break; }
            if (s[i] != ')') err(std::string("unexpected character '") + s[i] + "'");
            i++;
            v = stack.back();
            stack.pop_back();
            label[v] = read_label();
            read_length(v);
            if (stack.empty()) break;
        }
        if (stack.empty()) break;
    }
    skip();
    if (i >= n || s[i] != ';') err("the tree must end with ';'");
    i++;
    skip();
    if (i != n) err("text after the tree's ';' (one tree per line)");
    const uint32_t nn = (uint32_t)T.parent.size();
    std::vector<char> has_kid(nn, 0);
    for (uint32_t v = 1; v < nn; v++) {
        has_kid[T.parent[v]] = 1;
        if (!has_len[v]) fail("ms text, " + where(L) + ": Newick tree: node '" + label[v] + "' has no branch length");
        if (T.branch_len[v] < 0) fail("ms text, " + where(L) + ": Newick tree: node '" + label[v] + "' has a negative branch length");
    }
    T.branch_len[0] = 0.0;
    T.tip_node.assign(n_tips, UINT32_MAX);
    uint32_t tips = 0;
    for (uint32_t v = 0; v < nn; v++) {
        if (has_kid[v]) continue;
        tips++;
        const auto it = tip_of.find(label[v]);
        if (it == tip_of.end())
            fail("ms text, " + where(L) + ": tip label '" + label[v] + "' is not one of the haplotypes' names");
        if (T.tip_node[it->second] != UINT32_MAX) fail("ms text, " + where(L) + ": duplicate tip label '" + label[v] + "'");
        T.tip_node[it->second] = v;
    }
    if (tips != n_tips)
        fail("ms text, " + where(L) + ": the tree has " + std::to_string(tips) + " tips, the haplotypes are " +
             std::to_string(n_tips) + " (every tree needs the same tip labels)");
}

}  // namespace

void parse_ms(const char* text, uint64_t len, const std::vector<uint64_t>& chrom_len, const char* const* tip_names,
              uint32_t n_tips, uint32_t max_nodes, unsigned n_threads, GeneTrees& out) {
    // the lines: `//` starts a block, tree lines start with '[' or '('; everything else is ignored
    std::vector<TreeLine> lines;
    std::vector<uint64_t> block_first;           // each block's first tree line
    for (uint64_t a = 0; a < len;) {
        const void* e = std::memchr(text + a, '\n', len - a);
        const uint64_t b = e ? (uint64_t)(static_cast<const char*>(e) - text) : len;
        uint64_t m = b - a;
        if (m && text[a + m - 1] == '\r') m--;
        const char* s = text + a;
        if (m >= 2 && s[0] == '/' && s[1] == '/') {
            block_first.push_back(lines.size());
        } else if (m && (s[0] == '[' || s[0] == '(') && !block_first.empty()) {
            TreeLine t{s, m, 0, block_first.size() - 1, lines.size() - block_first.back()};
            const void* close = s[0] == '[' ? std::memchr(s, ']', m) : nullptr;
            uint64_t k = 1, v = 0;
            if (close) {
                const uint64_t c = (uint64_t)(static_cast<const char*>(close) - s);
                while (k < c && s[k] >= '0' && s[k] <= '9') {
                    if (v > (UINT64_MAX - 9) / 10) fail("ms text, " + where(t) + ": the [n] prefix is too large");
                    v = 10 * v + (uint64_t)(s[k] - '0');
                    k++;
                }
                if (k == c && c > 1) {                     // [digits]: the prefix; anything else is a Newick comment
                    if (v == 0) fail("ms text, " + where(t) + ": the [n] prefix must be a positive integer, not [0]");
                    t.len = v;
                    t.s = s + c + 1;
                    t.n = m - c - 1;
                }
            }
            lines.push_back(t);
        }
        a = b + 1;
    }
    if (lines.empty()) fail("the ms text has no trees (a '//' line followed by tree lines)");
    if (lines.size() >> 32) fail("the ms text has 2^32 or more trees");
    const uint64_t nb = block_first.size(), nc = chrom_len.size();
    if (nb != nc)
        fail("the ms text has " + std::to_string(nb) + " blocks ('//' lines), the reference has " + std::to_string(nc) +
             " chromosomes");
    block_first.push_back(lines.size());
    for (uint64_t bk = 0; bk < nb; bk++) {
        const uint64_t f = block_first[bk], l = block_first[bk + 1];
        const std::string name = "ms text, block " + std::to_string(bk + 1);
        if (f == l) fail(name + " has no trees");
        uint64_t with = 0;
        for (uint64_t j = f; j < l; j++) with += lines[j].len > 0;
        if (with && with != l - f) fail(name + " mixes trees with and without a [n] prefix");
        if (!with && l - f > 1) fail(name + " has " + std::to_string(l - f) + " trees without a [n] prefix (one at most)");
    }

    std::unordered_map<std::string, uint32_t> tip_of;
    for (uint32_t t = 0; t < n_tips; t++)
        if (!tip_of.emplace(tip_names[t], t).second) fail(std::string("duplicate haplotype name '") + tip_names[t] + "'");
    out.trees.assign(lines.size(), GeneTree{});
    parallel_for(lines.size(), std::max(1u, std::min<unsigned>(n_threads, (unsigned)std::min<uint64_t>(lines.size(), 1u << 16))),
                 [&](uint64_t j) { parse_tree(lines[j], tip_of, n_tips, max_nodes, out.trees[j]); });

    // regions: [floor(L c_{k-1} / S), floor(L c_k / S)) over the prefix sums c_k, empty ones dropped
    out.regions.assign(nc, {});
    for (uint64_t bk = 0; bk < nb; bk++) {
        const uint64_t f = block_first[bk], l = block_first[bk + 1], L = chrom_len[bk];
        if (L >> 32) fail("chromosomes of 2^32 bases or more are not supported");
        unsigned __int128 S = 0;
        for (uint64_t j = f; j < l; j++) S += lines[j].len;
        if (S == 0) S = 1;                                 // one tree without a prefix: the whole chromosome
        if (S >> 64) fail("ms text, block " + std::to_string(bk + 1) + ": the [n] prefixes sum to 2^64 or more");
        unsigned __int128 cum = 0;
        uint64_t start = 0;
        for (uint64_t j = f; j < l; j++) {
            cum += lines[j].len ? lines[j].len : 1;
            const uint64_t end = (uint64_t)((unsigned __int128)L * cum / S);
            if (end > start) out.regions[bk].push_back(TreeRegion{(uint32_t)start, (uint32_t)end, (uint32_t)j});
            start = end;
        }
    }
}

}  // namespace jlp
