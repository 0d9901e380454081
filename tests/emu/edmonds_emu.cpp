// edmonds_emu.cpp -- TEST INFRASTRUCTURE: host build of the matching in squarna_b200/csrc/sqrn_edmonds.cuh
// (SQRN_HOST_EMU), so that `pytest -m "not gpu"` checks it against NetworkX's max_weight_matching and
// squarna_b200/SQRNalgos.Edmonds on a box without a GPU.  The delta minima run for a simulated team of `width` lanes
// (1; 32: the warp tier; 256: the CTA and global tiers, which run the same item function with the node state in shared
// memory or in a workspace slot) and the partial keys are combined in the device's order.  It is not linked into
// libsqrn_b200.so; barriers and concurrency are only covered by the `-m gpu` tests.
#define SQRN_HOST_EMU 1
#include <stdlib.h>
#include "../../squarna_b200/csrc/sqrn_params.h"
#include "../../squarna_b200/csrc/sqrn_edmonds.cuh"

using namespace sqrn;

extern "C" int emu_ed_smem_max_n(long long budget) { return ed_smem_max_n((size_t)budget); }

// One graph through ed_item with a team of `width` lanes: mate (V) receives each node's partner node or -1.  Returns
// the number of pairs or the item's error code.
static int run_item(int V, const int32_t *pos, const int64_t *rowptr, const int32_t *adj, const int32_t *ep,
                    const double *wt, int64_t E, double maxw, int width, int32_t *pairs)
{
    const int64_t vbase[2] = {0, V}, ebase[2] = {0, E}, base = 0;
    int32_t n_out = 0;
    EdBatch eb{};
    eb.n_items = 1; eb.vbase = vbase; eb.ebase = ebase; eb.rowptr = rowptr;
    eb.pos = pos; eb.adj = adj; eb.ep = ep; eb.wt = wt; eb.maxw = &maxw;
    eb.out_base = &base; eb.out_pairs = pairs; eb.out_n = &n_out;
    const EdLayout L = ed_layout(V);
    std::vector<double> state(L.total / 8 + 2);
    std::vector<int32_t> est((size_t)ed_edge_words(V, E));
    unsigned char *st = (unsigned char *)state.data();
    if (width == 1) ed_item<HuEmuTeam<1>>(eb, 0, st, est.data(), nullptr);
    else if (width == 32) ed_item<HuEmuTeam<32>>(eb, 0, st, est.data(), nullptr);
    else if (width == 256) ed_item<HuEmuTeam<256>>(eb, 0, st, est.data(), nullptr);
    else return SQRN_E_BADARG;
    return n_out;
}

// The matching alone on a graph given as its edges in insertion order (node ids 0 .. n_nodes-1 in insertion order;
// every node has an edge): pairs [n_nodes/2][2] out as node ids, v < w, in node order.  Returns the pair count.
extern "C" int emu_matching(int n_nodes, int64_t n_edges, const int32_t *ends, const double *w, int width, int32_t *pairs)
{
    std::vector<int64_t> rowptr((size_t)n_nodes + 1, 0);
    for (int64_t k = 0; k < 2 * n_edges; k++) rowptr[(size_t)ends[k] + 1]++;
    for (int x = 0; x < n_nodes; x++) rowptr[(size_t)x + 1] += rowptr[(size_t)x];
    std::vector<int32_t> adj((size_t)(2 * n_edges + 1)), pos((size_t)n_nodes + 1);
    std::vector<int64_t> at(rowptr.begin(), rowptr.end() - 1);
    for (int64_t k = 0; k < 2 * n_edges; k++) adj[(size_t)at[(size_t)ends[k]]++] = (int32_t)k;
    double maxw = 0.0;
    for (int64_t e = 0; e < n_edges; e++) if (w[e] > maxw) maxw = w[e];
    for (int x = 0; x < n_nodes; x++) pos[(size_t)x] = x;
    if (n_edges == 0) return 0;
    return run_item(n_nodes, pos.data(), rowptr.data(), adj.data(), ends, w, n_edges, maxw, width, pairs);
}

// Same arguments as sqrn_edmonds_batch, plus the team width; the same checks.  Pairs sorted by v.
extern "C" int emu_edmonds(int64_t n_seqs, const int64_t *off, const int64_t *so, const int32_t *stems,
                           const double *scores, double power, int width, int64_t *pair_offsets, int32_t *pairs)
{
    pair_offsets[0] = 0;
    for (int64_t b = 0; b < n_seqs; b++) {
        const int N = (int)(off[b + 1] - off[b]);
        const int64_t ns = so[b + 1] - so[b];
        if (N > SQRN_MAX_LEN || (ns > 0 && !hu_stems_ok(N, stems + 3 * so[b], ns))) return SQRN_E_BADARG;
        std::vector<double> w;
        if (ns > 0 && !ed_weights(scores + so[b], ns, power, w)) return SQRN_E_BADARG;
        std::vector<int32_t> pos, adj, ep;
        std::vector<int64_t> rowptr;
        std::vector<double> wt;
        const double maxw = ed_seq_graph(N, stems + 3 * so[b], w.data(), ns, pos, rowptr, adj, ep, wt);
        int n = 0;
        int32_t *out = pairs + 2 * pair_offsets[b];
        if (!wt.empty()) {
            n = run_item((int)pos.size(), pos.data(), rowptr.data(), adj.data(), ep.data(), wt.data(),
                         (int64_t)wt.size(), maxw, width, out);
            if (n < 0) return SQRN_E_BADARG;
            std::vector<std::pair<int32_t, int32_t>> pr((size_t)n);
            for (int k = 0; k < n; k++) pr[(size_t)k] = {out[2 * k], out[2 * k + 1]};
            std::sort(pr.begin(), pr.end());
            for (int k = 0; k < n; k++) { out[2 * k] = pr[(size_t)k].first; out[2 * k + 1] = pr[(size_t)k].second; }
        }
        pair_offsets[b + 1] = pair_offsets[b] + n;
    }
    return SQRN_OK;
}
