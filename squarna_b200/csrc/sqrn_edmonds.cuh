// sqrn_edmonds.cuh -- the Edmonds builder of SQRNalgos (squarna_b200/SQRNalgos.py: Edmonds) on the device: NetworkX's
// max_weight_matching (networkx/algorithms/matching.py, Van Rantwijk's primal-dual blossom algorithm, maxcardinality
// False) on the graph of the stem pairs, ported statement for statement.  One team (a warp or a CTA) per sequence.
//
// The graph is what Graph.add_weighted_edges_from builds from the dict {(v, w): score} filled in stem order: an edge
// sits at the FIRST occurrence of its pair and weighs the LAST stem's score ** power; the nodes are numbered in order
// of first appearance (v before w), and a node's adjacency lists its edges in the order they were added.  That order
// decides every tie, and with weights that are powers of multiples of 0.25 ties are the normal case, so the port keeps
// every order the Python code has:
//   - `queue` is a LIFO stack; Blossom.leaves() is the explicit-stack DFS (copy childs, pop from the end);
//   - bestedgeto / mybestedges keep first-insertion order and replace only on strictly smaller slack;
//   - the delta scans visit the nodes in node order, then the live blossoms in creation order (the order of the
//     blossomparent and blossomdual dicts); each later candidate wins only when strictly smaller.  The scan is a team
//     minimum over a key (order-preserving image of the value with -0.0 read as +0.0, kind, order index) that is
//     unique per candidate, so the partial keys may meet in any order.  A blossom's order index is its position in
//     the creation list, which is compacted (keeping its order) when full, never its slot;
//   - the end-of-stage expansion walks the creation list; expandBlossom / augmentBlossom keep the index parity,
//     wrap-around and rotation of `childs` / `edges`, with explicit frames in place of Python's trampolines.
// Arithmetic is float64 without FMA: slack = (dual[v] + dual[w]) - 2 * wt, delta3 = kslack / 2.0, duals change by
// +-delta; `kslack <= 0` and the strict `<` everywhere else.
//
// Ids: nodes 0 .. V-1, blossom slot s is id V + s (at most V/2 blossoms are alive at once: each has >= 3 children).
// Edges: oriented edge o = 2e (v, w) or 2e + 1 (w, v) of edge e; tail ep[o], head ep[o ^ 1].  Only a warp's or a CTA's
// rank 0 runs the search (the Python control flow is sequential); the stage start, the delta minima and the dual
// updates run over the whole team.  State: ~124 bytes a node (EdLayout) in shared memory or in a workspace slot, and
// 4E + O(V) int32 per sequence (allowed-edge stamps, the mybestedges arena) in a workspace slot.  The same functions
// compile for the host (SQRN_HOST_EMU, tests/emu/edmonds_emu.cpp) with the team of sqrn_hungarian.cuh's HuEmuTeam.
#pragma once
#include <cfloat>
#include <cmath>
#include <unordered_map>
#include "sqrn_hungarian.cuh"

namespace sqrn {

constexpr int ED_WARP_MAX_N = 256;  // warp tier: sequences of up to this many positions
constexpr int ED_WPC = 4;           // warp tier: warps (sequences) per CTA
constexpr int ED_CTA_TW = 8;        // CTA and global tiers: 256 threads a sequence
constexpr int ED_SCAN = 256;        // prefix-count scratch: one entry per thread of the widest team
constexpr int ED_NCTRL = 16;        // control words shared by the team

// control words
enum { EC_QLEN, EC_AUG, EC_STAMP, EC_CLEN, EC_NFREE, EC_CTOP, EC_MTOP, EC_ERR };

__host__ __device__ constexpr int ed_nb(int v) { return v / 2 + 1; }             // blossom slots
__host__ __device__ constexpr int64_t ed_ccap(int v) { return 3 * ((int64_t)ed_nb(v) + v + ed_nb(v)) + 8; }

// The per-node state of a sequence of at most n nodes (offsets in bytes).
struct EdLayout {
    int V, NB;
    size_t ctrl, scan, dual, bdual, lab, ledge, bedge, par, bbase, inb, mate, cpos, nleaf, cst, clen, mst, mlen,
        clist, freel, queue, stk, bto, frame, carena, total;
};

__host__ __device__ inline EdLayout ed_layout(int n)
{
    EdLayout L{};
    const size_t V = (size_t)n, NB = (size_t)ed_nb(n), ids = V + NB;
    L.V = n; L.NB = (int)NB;
    size_t off = 0;
    L.ctrl = off; off += nu_al(4 * ED_NCTRL);
    L.scan = off; off += nu_al(4 * ED_SCAN);
    L.dual = off; off += nu_al(8 * V);
    L.bdual = off; off += nu_al(8 * NB);
    L.ledge = off; off += nu_al(4 * ids);
    L.bedge = off; off += nu_al(4 * ids);
    L.par = off; off += nu_al(4 * ids);
    L.bbase = off; off += nu_al(4 * ids);
    L.inb = off; off += nu_al(4 * V);
    L.mate = off; off += nu_al(4 * V);
    L.cpos = off; off += nu_al(4 * NB);
    L.nleaf = off; off += nu_al(4 * NB);
    L.cst = off; off += nu_al(4 * NB);
    L.clen = off; off += nu_al(4 * NB);
    L.mst = off; off += nu_al(4 * NB);
    L.mlen = off; off += nu_al(4 * NB);
    L.clist = off; off += nu_al(4 * 2 * NB);
    L.freel = off; off += nu_al(4 * NB);
    L.queue = off; off += nu_al(4 * (V + 2));
    L.stk = off; off += nu_al(4 * ids);
    L.bto = off; off += nu_al(4 * ids);
    L.frame = off; off += nu_al(4 * 8 * NB);
    L.carena = off; off += nu_al(4 * (size_t)ed_ccap(n));
    L.lab = off; off += nu_al(ids);
    L.total = off;
    return L;
}

// int32 words of a sequence's edge state: allowed-edge stamps [E], then the mybestedges arena
__host__ __device__ inline int64_t ed_mcap(int v, int64_t e) { return 4 * e + 4 * (int64_t)ed_nb(v) + 8; }
__host__ __device__ inline int64_t ed_edge_words(int v, int64_t e) { return (e + ed_mcap(v, e) + 3) & ~(int64_t)3; }

// Dynamic shared memory of a CTA: the CTA tier holds the state, the reduction scratch (one key a warp) and the item
// number; the global tier only the last two; the warp tier ED_WPC states.
__host__ __device__ inline size_t ed_cta_smem(int n, bool state) { return (state ? ed_layout(n).total : 0) + 16 * ED_CTA_TW + 16; }
__host__ __device__ inline size_t ed_warp_smem(int n) { return ED_WPC * ed_layout(n).total; }

// Longest sequence whose state fits `budget` bytes of dynamic shared memory per CTA (the CTA tier).
inline int ed_smem_max_n(size_t budget)
{
    int lo = 0, hi = SQRN_MAX_LEN;
    while (lo < hi) {
        const int m = (lo + hi + 1) / 2;
        if (ed_cta_smem(m, true) <= budget) lo = m; else hi = m - 1;
    }
    return lo;
}

// A batch as the kernels see it.  Sequence b: nodes [vbase[b], vbase[b+1]), its position pos[vbase[b] + x] and
// adjacency adj[rowptr[vbase[b] + b + x] .. rowptr[vbase[b] + b + x + 1]) (oriented edges, local ids); edges
// [ebase[b], ebase[b+1]): endpoints ep[2 ebase[b] + o], weights wt[ebase[b] + e]; maxw[b] = NetworkX's maxweight.
struct EdBatch {
    int n_items; const int32_t *order;          // sequences of this launch, longest first
    const int64_t *vbase, *ebase, *rowptr;
    const int32_t *pos, *adj, *ep;
    const double *wt, *maxw;
    const int64_t *out_base; int32_t *out_pairs; int32_t *out_n;   // sequence b: up to V/2 pairs at out_base[b]; < 0: error
    int *counter;
    unsigned char *ws; int64_t slot_bytes;      // team t's slot at ws + t * slot_bytes: [node state (global tier)] edge state
};

// The search state of one sequence; every member function but the parallel ones runs on rank 0 only.
struct EdSeq {
    int V, NB, nids;
    int64_t E;
    const int32_t *adj, *ep;
    const int64_t *rp;
    const double *wt;
    int *ctrl, *scan;
    double *dual, *bdual;
    int8_t *lab;
    int32_t *ledge, *bedge, *par, *bbase, *inb, *mate, *cpos, *nleaf, *cst, *clen, *mst, *mlen, *clist, *freel,
        *queue, *stk, *bto, *frame, *carena, *allow, *marena;
    int64_t ccap, mcap;

    __device__ __forceinline__ int tail(int o) const { return ep[o]; }
    __device__ __forceinline__ int head(int o) const { return ep[o ^ 1]; }
    __device__ __forceinline__ double slack(int o) const
    {
        return __dsub_rn(__dadd_rn(dual[tail(o)], dual[head(o)]), __dmul_rn(2.0, wt[o >> 1]));
    }
    __device__ __forceinline__ int32_t *childs(int s) const { return carena + cst[s]; }
    __device__ __forceinline__ int32_t *edges(int s) const { return carena + cst[s] + clen[s]; }
    __device__ __forceinline__ void fail(int code) { if (!ctrl[EC_ERR]) ctrl[EC_ERR] = code; }

    __device__ void push(int v)
    {
        if (ctrl[EC_QLEN] >= V + 2) { fail(-2); return; }
        queue[ctrl[EC_QLEN]++] = v;
    }

    // Blossom.leaves() of id b: f(v) for each leaf in the DFS order; stops early when f returns true.  Returns the
    // last leaf visited.
    template <class F> __device__ int leaves(int b, F f)
    {
        int n = 0, last = -1;
        const int s0 = b - V;
        for (int k = 0; k < clen[s0]; k++) stk[n++] = childs(s0)[k];
        while (n) {
            const int t = stk[--n];
            if (t >= V) { const int s = t - V; for (int k = 0; k < clen[s]; k++) stk[n++] = childs(s)[k]; }
            else { last = t; if (f(t)) break; }
        }
        return last;
    }

    __device__ void assignLabel(int w, int t, int o)
    {
        for (;;) {
            const int b = inb[w];
            lab[w] = lab[b] = (int8_t)t;
            ledge[w] = ledge[b] = o;
            bedge[w] = bedge[b] = -1;
            if (t == 1) {
                if (b >= V) leaves(b, [&](int v) { push(v); return false; });
                else push(b);
                return;
            }
            const int m = mate[bbase[b]];      // (base, mate[base]): assignLabel(mate[base], 1, base)
            w = head(m); t = 1; o = m;
        }
    }

    // the base vertex of a new blossom, or -1 (an augmenting path)
    __device__ int scanBlossom(int v, int w)
    {
        int np = 0, base = -1;
        while (v != -1) {
            int b = inb[v];
            if (lab[b] & 4) { base = bbase[b]; break; }
            stk[np++] = b;
            lab[b] = 5;
            if (ledge[b] == -1) v = -1;
            else {
                v = tail(ledge[b]);
                b = inb[v];
                v = tail(ledge[b]);
            }
            if (w != -1) { const int x = v; v = w; w = x; }
        }
        for (int k = 0; k < np; k++) lab[stk[k]] = 1;
        return base;
    }

    __device__ void carena_compact()
    {
        int64_t q = 0;
        for (int64_t p = 0; p < ctrl[EC_CTOP];) {
            const int s = carena[p], len = carena[p + 1];
            const int64_t size = 2 + 2 * (int64_t)len;
            if (cpos[s] >= 0 && cst[s] == p + 2) {
                if (q != p) for (int64_t k = 0; k < size; k++) carena[q + k] = carena[p + k];
                cst[s] = (int32_t)(q + 2);
                q += size;
            }
            p += size;
        }
        ctrl[EC_CTOP] = (int)q;
    }

    __device__ void marena_compact()
    {
        int64_t q = 0;
        for (int64_t p = 0; p < ctrl[EC_MTOP];) {
            const int s = marena[p], len = marena[p + 1];
            const int64_t size = 2 + (int64_t)len;
            if (cpos[s] >= 0 && mst[s] == p + 2) {
                if (q != p) for (int64_t k = 0; k < size; k++) marena[q + k] = marena[p + k];
                mst[s] = (int32_t)(q + 2);
                q += size;
            }
            p += size;
        }
        ctrl[EC_MTOP] = (int)q;
    }

    // one entry k of a sub-blossom's neighbour list (addBlossom's bestedgeto); n: entries so far at L
    __device__ __forceinline__ void best_to(int b, int k, int32_t *L, int &n)
    {
        int j = head(k);
        if (inb[j] == b) j = tail(k);
        const int bj = inb[j];
        if (bj != b && lab[bj] == 1 && (bto[bj] < 0 || slack(k) < slack(L[bto[bj]]))) {
            if (bto[bj] < 0) { bto[bj] = n; L[n++] = k; }
            else L[bto[bj]] = k;
        }
    }

    __device__ void addBlossom(int base, int o)
    {
        int v = tail(o), w = head(o);
        const int bb = inb[base];
        int bv = inb[v], bw = inb[w];
        if (ctrl[EC_NFREE] == 0) { fail(-2); return; }
        const int s = freel[--ctrl[EC_NFREE]], b = V + s;
        bbase[b] = base;
        par[b] = -1;
        par[bb] = b;
        // lengths of the two paths, then the lists written in their final order
        int kv = 0, kw = 0;
        for (int x = bv; x != bb; x = inb[tail(ledge[x])]) kv++;
        for (int x = bw; x != bb; x = inb[tail(ledge[x])]) kw++;
        const int len = 1 + kv + kw;
        if (ctrl[EC_CTOP] + 2 + 2 * (int64_t)len > ccap) carena_compact();
        if (ctrl[EC_CTOP] + 2 + 2 * (int64_t)len > ccap) { fail(-2); return; }
        const int64_t at = ctrl[EC_CTOP];
        carena[at] = s; carena[at + 1] = len;
        cst[s] = (int32_t)(at + 2); clen[s] = len;
        ctrl[EC_CTOP] = (int)(at + 2 + 2 * (int64_t)len);
        int32_t *ch = childs(s), *ed = edges(s);
        ch[0] = bb;
        ed[kv] = o;
        for (int i = 0; bv != bb; i++) {
            par[bv] = b;
            ch[kv - i] = bv;
            ed[kv - 1 - i] = ledge[bv];
            v = tail(ledge[bv]);
            bv = inb[v];
        }
        for (int i = 0; bw != bb; i++) {
            par[bw] = b;
            ch[kv + 1 + i] = bw;
            ed[kv + 1 + i] = ledge[bw] ^ 1;
            w = tail(ledge[bw]);
            bw = inb[w];
        }
        lab[b] = 1;
        ledge[b] = ledge[bb];
        bdual[s] = 0.0;
        // the creation list (compacted in order when full)
        if (ctrl[EC_CLEN] == 2 * NB) {
            int q = 0;
            for (int p = 0; p < ctrl[EC_CLEN]; p++)
                if (clist[p] >= 0) { cpos[clist[p]] = q; clist[q++] = clist[p]; }
            ctrl[EC_CLEN] = q;
        }
        cpos[s] = ctrl[EC_CLEN];
        clist[ctrl[EC_CLEN]++] = s;
        int nl = 0;
        for (int k = 0; k < len; k++) nl += ch[k] >= V ? nleaf[ch[k] - V] : 1;
        nleaf[s] = nl;
        mst[s] = -1;
        // relabel the leaves
        leaves(b, [&](int x) {
            if (lab[inb[x]] == 2) push(x);
            inb[x] = b;
            return false;
        });
        // b.mybestedges, written at the arena's top (at most one entry per other top-level blossom)
        const int64_t need = 2 + (E < (int64_t)nids ? E : (int64_t)nids);
        if (ctrl[EC_MTOP] + need > mcap) marena_compact();
        if (ctrl[EC_MTOP] + need > mcap) { fail(-2); return; }
        const int64_t mat = ctrl[EC_MTOP];
        int32_t *L = marena + mat + 2;
        int n = 0;
        for (int k = 0; k < len; k++) {
            const int c = ch[k];
            if (c >= V) {
                const int sc = c - V;
                if (mst[sc] >= 0) {
                    const int32_t *nb = marena + mst[sc];
                    const int m = mlen[sc];
                    mst[sc] = -1;
                    for (int q = 0; q < m; q++) best_to(b, nb[q], L, n);
                } else {
                    leaves(c, [&](int x) {
                        for (int64_t q = rp[x]; q < rp[x + 1]; q++) best_to(b, adj[q], L, n);
                        return false;
                    });
                }
            } else {
                for (int64_t q = rp[c]; q < rp[c + 1]; q++) best_to(b, adj[q], L, n);
            }
            bedge[c] = -1;
        }
        for (int q = 0; q < n; q++) {       // clear bestedgeto
            int j = head(L[q]);
            if (inb[j] == b) j = tail(L[q]);
            bto[inb[j]] = -1;
        }
        marena[mat] = s; marena[mat + 1] = n;
        mst[s] = (int32_t)(mat + 2); mlen[s] = n;
        ctrl[EC_MTOP] = (int)(mat + 2 + n);
        int best = -1;
        double bs = 0.0;
        for (int q = 0; q < n; q++) {
            const double ks = slack(L[q]);
            if (best < 0 || ks < bs) { best = L[q]; bs = ks; }
        }
        bedge[b] = best;
    }

    __device__ void remove_blossom(int b)
    {
        const int s = b - V;
        lab[b] = 0; ledge[b] = -1; bedge[b] = -1; par[b] = -1;
        clist[cpos[s]] = -1;
        cpos[s] = -1; cst[s] = -1; mst[s] = -1;
        freel[ctrl[EC_NFREE]++] = s;
    }

    __device__ static __forceinline__ int wrap(int j, int n) { return j < 0 ? j + n : j; }

    __device__ void expandBlossom(int b0, bool endstage)
    {
        int32_t *fb = frame, *fk = frame + NB;
        int depth = 0;
        fb[0] = b0; fk[0] = 0; depth = 1;
        while (depth) {
            const int b = fb[depth - 1], s = b - V;
            if (fk[depth - 1] < clen[s]) {
                const int c = childs(s)[fk[depth - 1]++];
                par[c] = -1;
                if (c >= V) {
                    if (endstage && bdual[c - V] == 0.0) {
                        if (depth == NB) { fail(-2); return; }
                        fb[depth] = c; fk[depth] = 0; depth++;
                        continue;
                    }
                    leaves(c, [&](int v) { inb[v] = c; return false; });
                } else {
                    inb[c] = c;
                }
                continue;
            }
            if (!endstage && lab[b] == 2) relabel_expanded(b);
            remove_blossom(b);
            depth--;
        }
    }

    // expandBlossom's relabelling of the sub-blossoms of an expanding T-blossom b (during a stage)
    __device__ void relabel_expanded(int b)
    {
        const int s = b - V, n = clen[s];
        const int32_t *ch = childs(s), *ed = edges(s);
        const int entry = inb[head(ledge[b])];
        int j = 0;
        while (ch[j] != entry) j++;
        int jstep;
        if (j & 1) { j -= n; jstep = 1; } else jstep = -1;
        int ovw = ledge[b];                     // (v, w)
        const int stamp = ctrl[EC_STAMP];
        while (j != 0) {
            const int opq = jstep == 1 ? ed[wrap(j, n)] : ed[wrap(j - 1, n)] ^ 1;    // (p, q)
            const int q = head(opq);
            lab[head(ovw)] = 0;
            lab[q] = 0;
            assignLabel(head(ovw), 2, ovw);
            allow[opq >> 1] = stamp;
            j += jstep;
            if (jstep == 1) ovw = ed[wrap(j, n)];
            else ovw = ed[wrap(j - 1, n)] ^ 1;
            allow[ovw >> 1] = stamp;
            j += jstep;
        }
        const int w = head(ovw), bw = ch[wrap(j, n)];
        lab[w] = lab[bw] = 2;
        ledge[w] = ledge[bw] = ovw;
        bedge[bw] = -1;
        j += jstep;
        while (ch[wrap(j, n)] != entry) {
            const int bv = ch[wrap(j, n)];
            if (lab[bv] == 1) { j += jstep; continue; }
            int v;
            if (bv >= V) v = leaves(bv, [&](int x) { return lab[x] != 0; });
            else v = bv;
            if (lab[v] != 0) {
                lab[v] = 0;
                lab[head(mate[bbase[bv]])] = 0;
                assignLabel(v, 2, ledge[v]);
            }
            j += jstep;
        }
    }

    __device__ void rotate(int32_t *a, int n, int i)
    {
        auto rev = [](int32_t *x, int lo, int hi) { for (hi--; lo < hi; lo++, hi--) { const int32_t t = x[lo]; x[lo] = x[hi]; x[hi] = t; } };
        rev(a, 0, i); rev(a, i, n); rev(a, 0, n);
    }

    __device__ void augmentBlossom(int b0, int v0)
    {
        // frame: b, v, t, i, j, jstep, owx, pc
        int depth = 0;
        auto F = [&](int d) { return frame + 8 * d; };
        { int32_t *f = F(0); f[0] = b0; f[1] = v0; f[7] = 0; depth = 1; }
        while (depth) {
            int32_t *f = F(depth - 1);
            const int b = f[0], s = b - V, n = clen[s];
            const int32_t *ch = childs(s), *ed = edges(s);
            auto call = [&](int t, int v) {
                if (depth == NB) { fail(-2); return; }
                int32_t *g = F(depth); g[0] = t; g[1] = v; g[7] = 0; depth++;
            };
            if (f[7] == 0) {
                int t = f[1];
                while (par[t] != b) t = par[t];
                f[2] = t; f[7] = 1;
                if (t >= V) { call(t, f[1]); continue; }
            }
            if (f[7] == 1) {
                int i = 0;
                while (ch[i] != f[2]) i++;
                f[3] = i; f[4] = i;
                if (i & 1) { f[4] -= n; f[5] = 1; } else f[5] = -1;
                f[7] = 2;
            }
            if (f[7] == 2) {
                if (f[4] == 0) {
                    const int i = f[3];
                    rotate(childs(s), n, i);
                    rotate(edges(s), n, i);
                    bbase[b] = bbase[childs(s)[0]];
                    depth--;
                    continue;
                }
                f[4] += f[5];
                const int t = ch[wrap(f[4], n)];
                f[6] = f[5] == 1 ? ed[wrap(f[4], n)] : ed[wrap(f[4] - 1, n)] ^ 1;    // (w, x)
                f[7] = 3;
                if (t >= V) { call(t, tail(f[6])); continue; }
            }
            if (f[7] == 3) {
                f[4] += f[5];
                const int t = ch[wrap(f[4], n)];
                f[7] = 4;
                if (t >= V) { call(t, head(f[6])); continue; }
            }
            // f[7] == 4
            mate[tail(f[6])] = f[6];
            mate[head(f[6])] = f[6] ^ 1;
            f[7] = 2;
        }
    }

    __device__ void augmentMatching(int o)
    {
        for (int side = 0; side < 2; side++) {
            int osj = o ^ side;                 // (s, j)
            int s_ = tail(osj);
            for (;;) {
                const int bs = inb[s_];
                if (bs >= V) augmentBlossom(bs, s_);
                mate[s_] = osj;
                if (ledge[bs] == -1) break;
                const int t = tail(ledge[bs]);
                const int bt = inb[t];
                const int l = ledge[bt];        // (s, j)
                s_ = tail(l);
                const int j = head(l);
                if (bt >= V) augmentBlossom(bt, j);
                mate[j] = l ^ 1;
                osj = l;
            }
        }
    }

    // the substage's labelling loop: until the queue is empty or the matching augmented
    __device__ void scan_queue()
    {
        const int stamp = ctrl[EC_STAMP];
        while (ctrl[EC_QLEN] > 0 && !ctrl[EC_AUG] && !ctrl[EC_ERR]) {
            const int v = queue[--ctrl[EC_QLEN]];
            for (int64_t q = rp[v]; q < rp[v + 1]; q++) {
                const int o = adj[q], w = head(o);
                const int bv = inb[v], bw = inb[w];
                if (bv == bw) continue;
                double kslack = 0.0;
                bool allowed = allow[o >> 1] == stamp;
                if (!allowed) {
                    kslack = slack(o);
                    if (kslack <= 0.0) { allow[o >> 1] = stamp; allowed = true; }
                }
                if (allowed) {
                    if (lab[bw] == 0) assignLabel(w, 2, o);
                    else if (lab[bw] == 1) {
                        const int base = scanBlossom(v, w);
                        if (base != -1) addBlossom(base, o);
                        else { augmentMatching(o); ctrl[EC_AUG] = 1; break; }
                    } else if (lab[w] == 0) { lab[w] = 2; ledge[w] = o; }
                } else if (lab[bw] == 1) {
                    if (bedge[bv] == -1 || kslack < slack(bedge[bv])) bedge[bv] = o;
                } else if (lab[w] == 0) {
                    if (bedge[w] == -1 || kslack < slack(bedge[w])) bedge[w] = o;
                }
            }
        }
    }
};

// The delta candidates: key (image of the value, kind << 30 | order index); kinds 0..3 are delta1..delta4.
__device__ __forceinline__ HuKey ed_key(double x, int kind, int idx)
{
    return HuKey{hu_image(x), (uint32_t)kind << 30 | (uint32_t)idx};
}

// One sequence (V >= 1 nodes, E >= 1 edges).  vst: the node state (EdLayout of at least V nodes); est: the edge state
// (ed_edge_words).  Writes the matched pairs (positions, v < w, in node order) or a negative error code to out_n.
template <class TM>
__device__ void ed_item(const EdBatch &eb, int seq, unsigned char *vst, int32_t *est, HuKey *red)
{
    constexpr int T = TM::T;
    const int rank = TM::rank();
    EdSeq S;
    const int64_t vb = eb.vbase[seq], eb0 = eb.ebase[seq];
    S.V = (int)(eb.vbase[seq + 1] - vb);
    S.NB = ed_nb(S.V);
    S.nids = S.V + S.NB;
    S.E = eb.ebase[seq + 1] - eb0;
    S.rp = eb.rowptr + vb + seq;
    S.adj = eb.adj;                                  // rp holds absolute offsets into adj
    S.ep = eb.ep + 2 * eb0;
    S.wt = eb.wt + eb0;
    const EdLayout L = ed_layout(S.V);               // this sequence's own offsets inside its (larger) slot
    S.ctrl = (int *)(vst + L.ctrl); S.scan = (int *)(vst + L.scan);
    S.dual = (double *)(vst + L.dual); S.bdual = (double *)(vst + L.bdual);
    S.lab = (int8_t *)(vst + L.lab);
    S.ledge = (int32_t *)(vst + L.ledge); S.bedge = (int32_t *)(vst + L.bedge); S.par = (int32_t *)(vst + L.par);
    S.bbase = (int32_t *)(vst + L.bbase); S.inb = (int32_t *)(vst + L.inb); S.mate = (int32_t *)(vst + L.mate);
    S.cpos = (int32_t *)(vst + L.cpos); S.nleaf = (int32_t *)(vst + L.nleaf); S.cst = (int32_t *)(vst + L.cst);
    S.clen = (int32_t *)(vst + L.clen); S.mst = (int32_t *)(vst + L.mst); S.mlen = (int32_t *)(vst + L.mlen);
    S.clist = (int32_t *)(vst + L.clist); S.freel = (int32_t *)(vst + L.freel); S.queue = (int32_t *)(vst + L.queue);
    S.stk = (int32_t *)(vst + L.stk); S.bto = (int32_t *)(vst + L.bto); S.frame = (int32_t *)(vst + L.frame);
    S.carena = (int32_t *)(vst + L.carena);
    S.allow = est; S.marena = est + S.E;
    S.ccap = ed_ccap(S.V); S.mcap = ed_mcap(S.V, S.E);
    const int V = S.V, NB = S.NB;
    const double maxw = eb.maxw[seq];

    // initial state
    for (int x = rank; x < V; x += T) { S.dual[x] = maxw; S.mate[x] = -1; S.inb[x] = x; }
    for (int x = rank; x < S.nids; x += T) { S.par[x] = -1; S.bbase[x] = x; S.bto[x] = -1; S.lab[x] = 0; }
    for (int s = rank; s < NB; s += T) { S.cpos[s] = -1; S.cst[s] = -1; S.mst[s] = -1; S.freel[s] = NB - 1 - s; }
    for (int64_t e = rank; e < S.E; e += T) S.allow[e] = 0;
    if (rank == 0) {
        for (int k = 0; k < ED_NCTRL; k++) S.ctrl[k] = 0;
        S.ctrl[EC_NFREE] = NB;
    }
    TM::sync();
    for (;;) {                                       // stages
        // stage start: clear labels and least-slack edges, forget mybestedges, a fresh allowed-edge stamp
        const int stamp = S.ctrl[EC_STAMP] + 1, ncl = S.ctrl[EC_CLEN];
        for (int x = rank; x < S.nids; x += T) { S.lab[x] = 0; S.ledge[x] = -1; S.bedge[x] = -1; }
        for (int p = rank; p < ncl; p += T) if (S.clist[p] >= 0) S.mst[S.clist[p]] = -1;
        TM::sync();
        if (rank == 0) { S.ctrl[EC_STAMP] = stamp; S.ctrl[EC_MTOP] = 0; S.ctrl[EC_QLEN] = 0; S.ctrl[EC_AUG] = 0; }
        // label the single top-level blossoms S, in node order: each thread takes a contiguous chunk, counts the
        // queue entries (a blossom's leaves, else the node), and after a prefix count writes them in order
        {
            const int chunk = (V + T - 1) / T, lo = rank * chunk < V ? rank * chunk : V, hi = lo + chunk < V ? lo + chunk : V;
            int cnt = 0;
            for (int v = lo; v < hi; v++)
                if (S.mate[v] < 0) { const int b = S.inb[v]; cnt += b >= V ? S.nleaf[b - V] : 1; }
            S.scan[rank] = cnt;
            TM::sync();
            if (rank == 0) {
                int acc = 0;
                for (int r = 0; r < T; r++) { const int c = S.scan[r]; S.scan[r] = acc; acc += c; }
                S.ctrl[EC_QLEN] = acc;
            }
            TM::sync();
            int at = S.scan[rank];
            for (int v = lo; v < hi; v++) {
                if (S.mate[v] >= 0) continue;
                const int b = S.inb[v];
                // (no other single node shares b: a blossom's only single node is its base)
                S.lab[v] = S.lab[b] = 1;
                if (b >= V) at += S.nleaf[b - V];
                else S.queue[at++] = v;
            }
            TM::sync();
        }
        if (rank == 0) {                             // the leaves of single S-blossoms, DFS order, at their places
            int at = 0;
            for (int v = 0; v < V; v++) {
                if (S.mate[v] >= 0) continue;
                const int b = S.inb[v];
                if (b >= V) {
                    int k = at;
                    S.leaves(b, [&](int x) { S.queue[k++] = x; return false; });
                    at += S.nleaf[b - V];
                } else at++;
            }
        }
        TM::sync();
        for (;;) {                                   // substages
            if (rank == 0) S.scan_queue();
            TM::sync();
            if (S.ctrl[EC_ERR]) break;
            if (S.ctrl[EC_AUG]) break;
            // delta: the first minimum of delta1 (node duals), delta2 (node order), delta3 (nodes, then blossoms in
            // creation order), delta4 (blossoms in creation order)
            const int cl = S.ctrl[EC_CLEN];
            const HuKey k = TM::argmin([&](int lane, int W) {
                HuKey best = hu_none();
                for (int v = lane; v < V; v += W) {
                    best = hu_min(best, ed_key(S.dual[v], 0, v));
                    if (S.lab[S.inb[v]] == 0 && S.bedge[v] != -1) best = hu_min(best, ed_key(S.slack(S.bedge[v]), 1, v));
                    if (S.par[v] == -1 && S.lab[v] == 1 && S.bedge[v] != -1)
                        best = hu_min(best, ed_key(__ddiv_rn(S.slack(S.bedge[v]), 2.0), 2, v));
                }
                for (int p = lane; p < cl; p += W) {
                    const int s = S.clist[p];
                    if (s < 0) continue;
                    const int b = V + s;
                    if (S.par[b] != -1) continue;
                    if (S.lab[b] == 1 && S.bedge[b] != -1)
                        best = hu_min(best, ed_key(__ddiv_rn(S.slack(S.bedge[b]), 2.0), 2, V + p));
                    if (S.lab[b] == 2) best = hu_min(best, ed_key(S.bdual[s], 3, p));
                }
                return best;
            }, red);
            const int kind = (int)(k.s >> 30), idx = (int)(k.s & 0x3fffffff);
            double delta;
            int dedge = -1, dblossom = -1;
            if (kind == 0) delta = S.dual[idx];
            else if (kind == 1) { dedge = S.bedge[idx]; delta = S.slack(dedge); }
            else if (kind == 2) {
                const int b = idx < V ? idx : V + S.clist[idx - V];
                dedge = S.bedge[b];
                delta = __ddiv_rn(S.slack(dedge), 2.0);
            } else { dblossom = V + S.clist[idx]; delta = S.bdual[dblossom - V]; }
            TM::sync();
            for (int v = rank; v < V; v += T) {
                const int l = S.lab[S.inb[v]];
                if (l == 1) S.dual[v] = __dsub_rn(S.dual[v], delta);
                else if (l == 2) S.dual[v] = __dadd_rn(S.dual[v], delta);
            }
            for (int p = rank; p < cl; p += T) {
                const int s = S.clist[p];
                if (s < 0 || S.par[V + s] != -1) continue;
                if (S.lab[V + s] == 1) S.bdual[s] = __dadd_rn(S.bdual[s], delta);
                else if (S.lab[V + s] == 2) S.bdual[s] = __dsub_rn(S.bdual[s], delta);
            }
            TM::sync();
            if (kind == 0) break;                    // optimum reached
            if (rank == 0) {
                if (kind == 1 || kind == 2) {
                    S.allow[dedge >> 1] = stamp;
                    S.push(S.tail(dedge));
                } else S.expandBlossom(dblossom, false);
            }
            TM::sync();
        }
        if (S.ctrl[EC_ERR] || !S.ctrl[EC_AUG]) break;
        // end of a stage: expand the top-level S-blossoms with zero dual, in creation order
        if (rank == 0) {
            const int cl = S.ctrl[EC_CLEN];
            for (int p = 0; p < cl; p++) {
                const int s = S.clist[p];
                if (s < 0) continue;
                const int b = V + s;
                if (S.par[b] == -1 && S.lab[b] == 1 && S.bdual[s] == 0.0) S.expandBlossom(b, true);
            }
        }
        TM::sync();
    }
    if (rank == 0) {
        int n = 0;
        if (!S.ctrl[EC_ERR]) {
            const int32_t *pos = eb.pos + vb;
            int32_t *out = eb.out_pairs + 2 * eb.out_base[seq];
            for (int v = 0; v < V; v++) {
                if (S.mate[v] < 0) continue;
                const int a = pos[v], c = pos[S.head(S.mate[v])];
                if (a < c) { out[2 * n] = a; out[2 * n + 1] = c; n++; }
            }
        } else n = S.ctrl[EC_ERR];
        eb.out_n[seq] = n;
    }
    TM::sync();
}

// ---- host side: the graph of a sequence (shared by the library and the emulation build) ----

// Weights as hu_weights, and no weight above DBL_MAX / 4 (2 * wt and the dual sums stay finite).
inline bool ed_weights(const double *sc, int64_t ns, double power, std::vector<double> &w)
{
    if (!hu_weights(sc, ns, power, w)) return false;
    for (const double x : w)
        if (x > DBL_MAX / 4) return false;
    return true;
}

// The NetworkX graph of one sequence's stems: edges at the first occurrence of their pair (stems in order, t
// ascending) with the last stem's weight; nodes in order of first appearance (pos: node -> position); per node its
// edges in the order they were added, as oriented edge ids (rowptr [V+1], adj); ep [2E] the oriented endpoints.
// Returns NetworkX's maxweight (0 when no weight is > 0).
inline double ed_seq_graph(int N, const int32_t *st, const double *w, int64_t ns, std::vector<int32_t> &pos,
                           std::vector<int64_t> &rowptr, std::vector<int32_t> &adj, std::vector<int32_t> &ep,
                           std::vector<double> &wt)
{
    std::unordered_map<uint32_t, int32_t> edge_of;
    std::vector<int32_t> last;
    std::vector<int32_t> ends;                       // positions (v, w) per edge
    for (int64_t s = 0; s < ns; s++)
        for (int t = 0; t < st[3 * s + 2]; t++) {
            const uint32_t v = (uint32_t)(st[3 * s] + t), x = (uint32_t)(st[3 * s + 1] - t);
            auto it = edge_of.emplace(v << 16 | x, (int32_t)last.size());
            if (it.second) { last.push_back((int32_t)s); ends.push_back((int32_t)v); ends.push_back((int32_t)x); }
            else last[(size_t)it.first->second] = (int32_t)s;
        }
    const size_t E = last.size();
    std::vector<int32_t> node((size_t)N, -1);
    pos.clear();
    ep.resize(2 * E);
    for (size_t k = 0; k < 2 * E; k++) {
        int32_t &nd = node[(size_t)ends[k]];
        if (nd < 0) { nd = (int32_t)pos.size(); pos.push_back(ends[k]); }
        ep[k] = nd;
    }
    const size_t V = pos.size();
    rowptr.assign(V + 1, 0);
    for (size_t k = 0; k < 2 * E; k++) rowptr[(size_t)ep[k] + 1]++;
    for (size_t x = 0; x < V; x++) rowptr[x + 1] += rowptr[x];
    adj.resize(2 * E);
    std::vector<int64_t> at(rowptr.begin(), rowptr.end() - 1);
    for (size_t k = 0; k < 2 * E; k++) adj[(size_t)at[(size_t)ep[k]]++] = (int32_t)k;   // edge k/2, tail ep[k]
    wt.resize(E);
    double maxw = 0.0;
    for (size_t e = 0; e < E; e++) {
        wt[e] = w[last[e]];
        if (wt[e] > maxw) maxw = wt[e];
    }
    return maxw;
}

}  // namespace sqrn
