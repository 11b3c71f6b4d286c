// Elimination-order heuristics on the interaction graph (host side).
//
// Replaces bn::Graph's constructor, ordering(), min_fill(), weighted_min_fill(),
// min_degree() and order_width() (reference code/graph.cpp:9-237).  north_star keeps
// this on the host and demands BIT-EXACT orders.  The reference breaks ties by the
// iteration order of libstdc++ `std::unordered_set<unsigned>` (SURVEY A.3), so this
// file deliberately uses the same containers and performs insertions, erasures and
// scans in the same sequence; only then do `*begin()`, the strict `<` scans and the
// fill-in edge insertions see the same element order.  Header-only so the C-ABI
// library (bnpp_elim_order) and the bn::Graph wrapper share one implementation.
#pragma once
#include <algorithm>
#include <cstdint>
#include <functional>
#include <queue>
#include <tuple>
#include <unordered_map>
#include <unordered_set>
#include <vector>

namespace bnpp {

enum Heuristic { H_MIN_FILL = 0, H_WEIGHTED_MIN_FILL = 1, H_MIN_DEGREE = 2 };

class InteractionGraph {
public:
    typedef std::unordered_set<unsigned> NodeSet;
    typedef std::unordered_map<unsigned, NodeSet> Adjacency;

    InteractionGraph() {}

    // scopes[f] = variable ids of factor f in scope order; card[id] = cardinality
    InteractionGraph(const std::vector<std::vector<unsigned>> &scopes, const std::vector<unsigned> &card) : card_(card)
    {
        // every scope variable becomes a node first (code/graph.cpp:11-18) ...
        for (const auto &sc : scopes)
            for (unsigned v : sc) adj_[v] = NodeSet();
        // ... then each factor contributes a clique, pairs (i, j > i) in scope order (code/graph.cpp:20-34)
        for (const auto &sc : scopes) {
            const size_t w = sc.size();
            for (size_t i = 0; i + 1 < w; ++i)
                for (size_t j = i + 1; j < w; ++j) {
                    adj_[sc[i]].insert(sc[j]);
                    adj_[sc[j]].insert(sc[i]);
                }
        }
    }

    const Adjacency &adjacency() const { return adj_; }
    Adjacency &adjacency() { return adj_; }

    bool has(unsigned id) const { return adj_.find(id) != adj_.end(); }

    // The reference dereferences find() unchecked and crashes on a node it does not know
    // (SURVEY A.2 i); here an unknown node simply has no neighbours.
    const NodeSet &neighbors(unsigned id) const
    {
        static const NodeSet none;
        Adjacency::const_iterator it = adj_.find(id);
        return it == adj_.end() ? none : it->second;
    }

    bool connected(unsigned a, unsigned b) const
    {
        Adjacency::const_iterator it = adj_.find(a);
        return it != adj_.end() && it->second.count(b) != 0;
    }

    // number (or cardinality-weighted number) of edges elimination of `id` would add
    unsigned fill_in(unsigned id, bool weighted) const
    {
        const NodeSet &nb = neighbors(id);
        unsigned score = 0;
        for (unsigned a : nb)
            for (unsigned b : nb)
                if (a < b && !connected(a, b)) score += weighted ? card_.at(a) * card_.at(b) : 1u;
        return score;
    }

    // code/graph.cpp:103-120
    unsigned pick_min_degree(const NodeSet &cand) const
    {
        unsigned best = *cand.begin();
        unsigned best_deg = (unsigned)adj_.size() + 1;
        for (unsigned id : cand) {
            const unsigned deg = (unsigned)neighbors(id).size();
            if (deg < best_deg) {
                best = id;
                best_deg = deg;
            }
        }
        return best;
    }

    // code/graph.cpp:122-153: the best score is seeded with |nodes|+1, NOT with the first candidate's score
    unsigned pick_min_fill(const NodeSet &cand) const
    {
        unsigned best = *cand.begin();
        unsigned best_fill = (unsigned)adj_.size() + 1;
        for (unsigned id : cand) {
            const unsigned f = fill_in(id, false);
            if (f < best_fill || (f == best_fill && neighbors(id).size() < neighbors(best).size())) {
                best = id;
                best_fill = f;
            }
        }
        return best;
    }

    // code/graph.cpp:155-195: seeded with the first candidate's real score
    unsigned pick_weighted_min_fill(const NodeSet &cand) const
    {
        unsigned best = *cand.begin();
        unsigned best_fill = fill_in(best, true);
        for (unsigned id : cand) {
            const unsigned f = fill_in(id, true);
            if (f < best_fill || (f == best_fill && neighbors(id).size() < neighbors(best).size())) {
                best = id;
                best_fill = f;
            }
        }
        return best;
    }

    // Removes `id`, connecting its neighbours pairwise; returns its degree at that moment.
    // Sequence of mutations as in code/graph.cpp:73-96.
    unsigned eliminate(unsigned id, bool erase_node_first)
    {
        const NodeSet nb = neighbors(id);   // a copy iterates exactly like the original
        if (erase_node_first) adj_.erase(id);          // order_width() erases the node first (code/graph.cpp:217-218)
        for (unsigned a : nb) adj_[a].erase(id);
        for (unsigned a : nb)
            for (unsigned b : nb)
                if (a != b && !connected(a, b)) {
                    adj_[a].insert(b);
                    adj_[b].insert(a);
                }
        if (!erase_node_first) adj_.erase(id);
        return (unsigned)nb.size();
    }

    // Graph::ordering, code/graph.cpp:41-101.  `vars` in the caller's order.
    std::vector<unsigned> ordering(const std::vector<unsigned> &vars, Heuristic h, unsigned &width) const
    {
        InteractionGraph g(*this);
        return g.ordering_in_place(vars, h, width);
    }

    // the same on this graph itself: the eliminated nodes are gone and the fill edges stay, so a second call orders
    // the rest of the variables after the first ones (constrained orders: summed variables, then MAP variables)
    std::vector<unsigned> ordering_in_place(const std::vector<unsigned> &vars, Heuristic h, unsigned &width)
    {
        InteractionGraph &g = *this;
        NodeSet cand;
        for (unsigned v : vars) cand.insert(v);
        std::vector<unsigned> order;
        order.reserve(vars.size());
        width = 0;
        while (!cand.empty()) {
            unsigned next;
            if (h == H_MIN_DEGREE) next = g.pick_min_degree(cand);
            else if (h == H_WEIGHTED_MIN_FILL) next = g.pick_weighted_min_fill(cand);
            else next = g.pick_min_fill(cand);
            order.push_back(next);
            const unsigned deg = g.eliminate(next, false);
            if (deg > width) width = deg;
            cand.erase(next);
        }
        return order;
    }

    // Graph::order_width, code/graph.cpp:197-237
    unsigned order_width(const std::vector<unsigned> &order) const
    {
        InteractionGraph g(*this);
        unsigned width = 0;
        for (unsigned v : order) {
            const unsigned deg = g.eliminate(v, true);
            if (deg > width) width = deg;
        }
        return width;
    }

    const std::vector<unsigned> &cardinalities() const { return card_; }

private:
    std::vector<unsigned> card_;
    Adjacency adj_;
};

// Same orders as InteractionGraph::ordering, computed faster (SURVEY §8f row 1: once the
// tables are fast, ordering is what an end-to-end query waits for).
//
// What decides the reference's order is (1) the iteration order of the CANDIDATE set --
// kept here as the very same std::unordered_set<unsigned> with the same insert / erase
// history -- and (2) per-candidate scores and degrees, which are order-independent sums.
// The iteration order of the adjacency sets never influences a decision, so adjacency is
// a bit matrix: fill-in = C(d,2) - (edges inside the neighbourhood) by popcounts, cached
// per node and recomputed only for nodes whose neighbourhood changed.  Scores wrap modulo
// 2^32 exactly like the reference's `unsigned` accumulators.
class FastOrderer {
public:
    explicit FastOrderer(const InteractionGraph &g) : card_(g.cardinalities())
    {
        unsigned maxid = 0;
        for (const auto &node : g.adjacency()) {
            maxid = std::max(maxid, node.first);
            for (unsigned b : node.second) maxid = std::max(maxid, b);
        }
        n_ = maxid + 1;
        words_ = (n_ + 63) / 64;
        bits_.assign((size_t)n_ * words_, 0);
        present_.assign(n_, 0);
        deg_.assign(n_, 0);
        lo_.assign(n_, words_);
        hi_.assign(n_, 0);
        for (const auto &node : g.adjacency()) {
            present_[node.first] = 1;
            ++alive_;
            for (unsigned b : node.second) set(node.first, b);
            deg_[node.first] = (unsigned)node.second.size();
        }
        score_.assign(n_, 0);
        dirty_.assign(n_, 1);
    }

    // The same graph straight from the factor scopes (no hash containers): nodes = every scope
    // variable, edges = the pairs of each scope (code/graph.cpp:11-34).
    FastOrderer(const std::vector<std::vector<unsigned>> &scopes, const std::vector<unsigned> &card) : card_(card)
    {
        unsigned maxid = 0;
        bool any = false;
        for (const auto &sc : scopes)
            for (unsigned v : sc) {
                maxid = std::max(maxid, v);
                any = true;
            }
        n_ = any ? maxid + 1 : 0;
        words_ = (n_ + 63) / 64;
        bits_.assign((size_t)n_ * words_, 0);
        present_.assign(n_, 0);
        deg_.assign(n_, 0);
        lo_.assign(n_, words_);
        hi_.assign(n_, 0);
        for (const auto &sc : scopes) {
            for (unsigned v : sc)
                if (!present_[v]) {
                    present_[v] = 1;
                    ++alive_;
                }
            for (size_t i = 0; i + 1 < sc.size(); ++i)
                for (size_t j = i + 1; j < sc.size(); ++j)
                    if (sc[i] != sc[j]) {
                        set(sc[i], sc[j]);
                        set(sc[j], sc[i]);
                    }
        }
        for (unsigned v = 0; v < n_; ++v) {
            unsigned d = 0;
            for (unsigned w = lo_[v]; w <= hi_[v] && w < words_; ++w) d += (unsigned)__builtin_popcountll(row(v)[w]);
            deg_[v] = d;
        }
        score_.assign(n_, 0);
        dirty_.assign(n_, 1);
    }

    // Every round of the reference scans ALL candidates in the iteration order of its
    // std::unordered_set and keeps the first strict improvement of (score, then degree).
    // Erasing from an unordered_set never reorders the remaining elements, so that order
    // is fixed once the set is filled: `seq`.  The scan's winner is then the minimum of
    // (score, degree, position in seq) -- kept in an ordered set whose keys are refreshed
    // only for the nodes an elimination touched, instead of O(candidates) work per round.
    // The one case where the scan is NOT that minimum -- plain min-fill seeds its best
    // score with |nodes|+1 (code/graph.cpp:122-153), so when no candidate scores below
    // the seed the first candidate survives unless a later one ties the seed with a smaller
    // degree -- falls back to the literal scan for that round.  The graph is eliminated in place: a second call orders
    // the rest of the variables with the fill edges of the first in place.
    std::vector<unsigned> ordering(const std::vector<unsigned> &vars, Heuristic h, unsigned &width)
    {
        std::unordered_set<unsigned> cand;
        for (unsigned v : vars) cand.insert(v);
        const std::vector<unsigned> seq(cand.begin(), cand.end());
        const size_t m = seq.size();
        std::vector<unsigned> order;
        order.reserve(m);
        width = 0;
        const bool weighted = (h == H_WEIGHTED_MIN_FILL);
        typedef std::tuple<unsigned, unsigned, unsigned> Key;      // (score, degree, position)
        // a min-heap with lazy deletion: a refreshed key is pushed, its stale copy is skipped when it surfaces
        std::priority_queue<Key, std::vector<Key>, std::greater<Key>> heap;
        std::vector<Key> key(m);
        std::vector<char> live(m, 1);
        std::vector<int> pos_of(n_, -1);                            // candidates that are graph nodes
        auto make_key = [&](unsigned pos) {
            const unsigned id = seq[pos];
            if (h == H_MIN_DEGREE) return Key(degree(id), 0u, pos);
            return Key(fill(id, weighted), degree(id), pos);
        };
        for (unsigned pos = 0; pos < m; ++pos) {
            if (seq[pos] < n_) pos_of[seq[pos]] = (int)pos;
            key[pos] = make_key(pos);
            heap.push(key[pos]);
        }
        touched_.clear();
        size_t left = m;
        while (left) {
            for (unsigned id : touched_) {
                const int pos = id < n_ ? pos_of[id] : -1;
                if (pos < 0 || !live[pos]) continue;
                const Key k = make_key((unsigned)pos);
                if (k != key[pos]) {
                    key[pos] = k;
                    heap.push(k);
                }
            }
            touched_.clear();
            while (!live[std::get<2>(heap.top())] || heap.top() != key[std::get<2>(heap.top())]) heap.pop();
            unsigned best_pos = std::get<2>(heap.top());
            if (h == H_MIN_FILL && std::get<0>(heap.top()) >= alive_ + 1) {
                // the literal scan of code/graph.cpp:122-153
                bool first = true;
                unsigned best = 0, best_fill = alive_ + 1;
                for (unsigned pos = 0; pos < m; ++pos) {
                    if (!live[pos]) continue;
                    const unsigned id = seq[pos];
                    if (first) {
                        best = id;
                        best_pos = pos;
                        first = false;
                    }
                    const unsigned f = fill(id, false);
                    if (f < best_fill || (f == best_fill && degree(id) < degree(best))) {
                        best = id;
                        best_pos = pos;
                        best_fill = f;
                    }
                }
            }
            const unsigned best = seq[best_pos];
            order.push_back(best);
            live[best_pos] = 0;
            --left;
            const unsigned d = eliminate(best);
            if (d > width) width = d;
        }
        return order;
    }

private:
    uint64_t *row(unsigned a) { return &bits_[(size_t)a * words_]; }
    const uint64_t *row(unsigned a) const { return &bits_[(size_t)a * words_]; }
    void set(unsigned a, unsigned b)
    {
        const unsigned w = b >> 6;
        row(a)[w] |= 1ull << (b & 63);
        if (w < lo_[a]) lo_[a] = w;
        if (w > hi_[a]) hi_[a] = w;
    }
    void clear(unsigned a, unsigned b) { row(a)[b >> 6] &= ~(1ull << (b & 63)); }
    bool test(unsigned a, unsigned b) const { return (row(a)[b >> 6] >> (b & 63)) & 1ull; }
    unsigned degree(unsigned id) const { return id < n_ ? deg_[id] : 0; }

    // lo_/hi_: the words of a row that ever held a bit (rows of a sparse graph are mostly empty words)
    template <class F>
    void for_each(unsigned v, F f) const
    {
        const uint64_t *r = row(v);
        for (unsigned w = lo_[v]; w <= hi_[v] && w < words_; ++w) {
            uint64_t x = r[w];
            while (x) {
                const unsigned b = (unsigned)__builtin_ctzll(x);
                x &= x - 1;
                f(w * 64 + b);
            }
        }
    }

    unsigned fill(unsigned id, bool weighted)
    {
        if (id >= n_ || !present_[id]) return 0;
        if (!dirty_[id]) return score_[id];
        const uint64_t *nw = row(id);
        uint64_t s;
        if (!weighted) {
            uint64_t inside = 0;   // ordered pairs (a, b) of neighbours that are adjacent
            for_each(id, [&](unsigned a) {
                const uint64_t *na = row(a);
                const unsigned w0 = std::max(lo_[a], lo_[id]), w1 = std::min(hi_[a], hi_[id]);
                for (unsigned w = w0; w <= w1 && w < words_; ++w) inside += (uint64_t)__builtin_popcountll(na[w] & nw[w]);
            });
            const uint64_t d = deg_[id];
            s = d * (d - (d ? 1 : 0)) / 2 - inside / 2;
        } else {
            uint64_t sum = 0, sq = 0, inside = 0;
            for_each(id, [&](unsigned a) {
                const uint64_t ca = card_.at(a);
                sum += ca;
                sq += ca * ca;
                const uint64_t *na = row(a);
                uint64_t acc = 0;
                const unsigned w0 = std::max(lo_[a], lo_[id]), w1 = std::min(hi_[a], hi_[id]);
                for (unsigned w = w0; w <= w1 && w < words_; ++w) {
                    uint64_t x = na[w] & nw[w];
                    while (x) {
                        const unsigned b = (unsigned)__builtin_ctzll(x);
                        x &= x - 1;
                        acc += card_.at(w * 64 + b);
                    }
                }
                inside += ca * acc;
            });
            s = (sum * sum - sq) / 2 - inside / 2;
        }
        score_[id] = (unsigned)s;   // the reference accumulates in `unsigned`
        dirty_[id] = 0;
        return score_[id];
    }

    unsigned eliminate(unsigned v)
    {
        if (v >= n_ || !present_[v]) return 0;
        std::vector<unsigned> nb;
        for_each(v, [&](unsigned a) { nb.push_back(a); });
        for (unsigned a : nb) {
            clear(a, v);
            --deg_[a];
            dirty_[a] = 1;
            touched_.push_back(a);
        }
        for (size_t i = 0; i < nb.size(); ++i)
            for (size_t j = i + 1; j < nb.size(); ++j) {
                const unsigned a = nb[i], b = nb[j];
                if (test(a, b)) continue;
                // a new edge changes the fill-in of every common neighbour of its end points
                const uint64_t *ra = row(a), *rb = row(b);
                const unsigned w0 = std::max(lo_[a], lo_[b]), w1 = std::min(hi_[a], hi_[b]);
                for (unsigned w = w0; w <= w1 && w < words_; ++w) {
                    uint64_t x = ra[w] & rb[w];
                    while (x) {
                        const unsigned c = (unsigned)__builtin_ctzll(x);
                        x &= x - 1;
                        if (!dirty_[w * 64 + c]) touched_.push_back(w * 64 + c);
                        dirty_[w * 64 + c] = 1;
                    }
                }
                set(a, b);
                set(b, a);
                ++deg_[a];
                ++deg_[b];
            }
        if (lo_[v] <= hi_[v]) std::fill(row(v) + lo_[v], row(v) + std::min(hi_[v] + 1, words_), 0);
        deg_[v] = 0;
        present_[v] = 0;
        --alive_;
        return (unsigned)nb.size();
    }

    std::vector<unsigned> card_;
    unsigned n_ = 0, words_ = 0, alive_ = 0;
    std::vector<uint64_t> bits_;
    std::vector<char> present_, dirty_;
    std::vector<unsigned> deg_, score_;
    std::vector<unsigned> lo_, hi_;     // per row: first and last word that ever held a bit (lo > hi: none)
    std::vector<unsigned> touched_;     // nodes whose score or degree the last elimination changed
};

}  // namespace bnpp
