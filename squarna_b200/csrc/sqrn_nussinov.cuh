// sqrn_nussinov.cuh -- the Nussinov builder of SQRNalgos (squarna_b200/SQRNalgos.py: Nussinov, BackTrack) on the
// device: the stem-weighted dynamic program over the upper triangle and the backtrack, one CTA per sequence.
//
//   D[i][i] = 0;  D[i][j] (j > i) over the partners k of j with i <= k < j - 1, in increasing k:
//     tot(k) = (left + D[k+1][j-1]) + e(k, j),  left = D[i][k-1] if k > i else 0,  e(k, j) = -(score of its stem)
//     best   = the first strict minimum of tot, if it is < 1e9
//     best <= D[i][j-1] ?  D[i][j] = best, K[i][j] = its k  :  D[i][j] = D[i][j-1], no K entry
//
// Every cell is a pure function of cells of smaller span, so any order that respects the dependencies gives the
// same float64 values; the kernels sweep COLUMNS j = 1 .. N-1, all rows i < j of a column in parallel (column j
// only reads columns < j).  The triangle is stored column-major with its diagonal, so the reads D[i][k-1] of a warp
// (32 consecutive rows) are contiguous.  A warp walks the candidates of the column in step: the staged (k, e,
// D[k+1][j-1]) are broadcast reads, and a lane skips the k below its row.
//
// The same functions compile for the host with a team of one thread (SQRN_HOST_EMU, tests/emu/nussinov_emu.cpp).
#pragma once
#include <stdint.h>
#include <algorithm>
#include <string>
#include <vector>
#include "../../include/sqrn.h"
#include "sqrn_device.cuh"

namespace sqrn {

constexpr int NU_CHUNK = 1024;      // global tier: candidates of a column staged per pass (more take several passes)
constexpr int NU_SMEM_TW = 8;       // shared-memory tier: 256 threads (a column has fewer rows than that)
constexpr int NU_GLOB_TW = 16;      // global tier: 512 threads
constexpr double NU_NONE = 1e9;     // `best` before any candidate (SQRNalgos.Nussinov: 10 ** 9)

__host__ __device__ constexpr int64_t nu_cells(int n) { return (int64_t)n * (n + 1) / 2; }    // triangle with diagonal
__host__ __device__ __forceinline__ int64_t nu_col(int j) { return (int64_t)j * (j + 1) / 2; }   // D[i][j] at nu_col(j) + i
__host__ __device__ constexpr size_t nu_al(size_t x) { return (x + 15) & ~(size_t)15; }

// What the backtrack needs after the sweep, in the memory the sweep used: separator prefix counts [N+1], partner of
// every position [N], and the stack of open intervals (disjoint, each of at least two positions: at most N/2 + 1).
__host__ __device__ constexpr size_t nu_bt_bytes(int n)
{
    return nu_al(4 * (size_t)(n + 1)) + nu_al(4 * (size_t)n) + nu_al(8 * ((size_t)n / 2 + 2));
}

// Dynamic shared memory of one CTA.  Shared-memory tier: the triangle, then the staged candidates of a column (at
// most nmax of them, one pass).  Global tier: the previous column, then NU_CHUNK staged candidates; the triangle is in
// the CTA's workspace slot.  The backtrack scratch starts at byte 0 in both.  The last 16 bytes carry the item number.
struct NuLayout { int nmax, chunk; size_t prev_off, ca_off, ce_off, ck_off, item_off, total; };

__host__ __device__ constexpr size_t nu_max(size_t a, size_t b) { return a > b ? a : b; }

__host__ __device__ inline NuLayout nu_layout(int nmax, bool smem_tier, int chunk = NU_CHUNK)
{
    NuLayout L{};
    L.nmax = nmax;
    L.chunk = smem_tier ? (nmax > 1 ? nmax : 1) : chunk;
    size_t off = smem_tier ? nu_al(8 * (size_t)nu_cells(nmax)) : 0;
    L.prev_off = off;
    if (!smem_tier) off += nu_al(8 * (size_t)nmax);
    L.ca_off = off; off += nu_al(8 * (size_t)L.chunk);
    L.ce_off = off; off += nu_al(8 * (size_t)L.chunk);
    L.ck_off = off; off += nu_al(2 * (size_t)L.chunk);
    off = nu_max(off, nu_al(nu_bt_bytes(nmax)));
    L.item_off = off;
    L.total = off + 16;
    return L;
}

// Longest sequence the shared-memory tier takes within `budget` bytes of dynamic shared memory per CTA.
inline int nu_smem_max_n(size_t budget)
{
    int n = 0;
    while (n < SQRN_MAX_LEN && nu_layout(n + 1, true).total <= budget) n++;
    return n;
}

// A batch as the kernels see it.  Candidate lists P(j): sequence b's N + 1 column pointers start at colptr[off[b] + b];
// column j's partners are pk[colptr[..j] .. colptr[..j+1]) in increasing k (all k < j - 1), energies in pe.
struct NuBatch {
    int n_items; const int32_t *order;          // sequences of this launch, longest first
    const int64_t *off; const uint8_t *sym;     // symbols: the separators ';' '&' count for the backtrack
    const int64_t *colptr; const int16_t *pk; const double *pe;
    int minloop;
    const int64_t *out_base; int32_t *out_pairs; int32_t *out_n;   // sequence b: up to N/2 pairs at out_base[b]
    int *counter;
    // per-CTA workspace slots: global-tier triangle (slot_d doubles), K (slot_k int16, both tiers), the running best
    // of a row across candidate passes (slot_s each, global tier)
    double *wd; int16_t *wk; double *wbest; int16_t *wbk; int64_t slot_d, slot_k, slot_s;
};

// One sequence: the column sweep (whole team), then the backtrack (one thread).  tri: the triangle (shared memory or
// the workspace slot); prevbuf: NULL when the previous column is read in place (shared-memory tier), else a shared
// copy of it; smem: the layout's base (staged candidates, backtrack scratch); K: the slot's int16 triangle.
// pre[p] = separators ';' '&' among the first p symbols, p = 0 .. N
__host__ __device__ inline void sep_prefix(const uint8_t *sq, int N, int32_t *pre)
{
    pre[0] = 0;
    for (int p = 0; p < N; p++) pre[p + 1] = pre[p] + (sq[p] == ';' || sq[p] == '&');
}

template <int TW>
__device__ void nu_item(const NuBatch &nb, int seq, double *tri, double *prevbuf, const NuLayout &L, unsigned char *smem,
                        int16_t *K, double *sbest, int16_t *sbk)
{
    using TM = Team<TW>;
    constexpr int T = TM::T;
    const int rank = TM::rank(), lane = rank & 31;
    const int64_t o = nb.off[seq];
    const int N = (int)(nb.off[seq + 1] - o);
    const int64_t *cp = nb.colptr + o + seq;
    double *ca = (double *)(smem + L.ca_off), *ce = (double *)(smem + L.ce_off);
    int16_t *ck = (int16_t *)(smem + L.ck_off);
    if (rank == 0 && N > 0) { tri[0] = 0.0; if (prevbuf) prevbuf[0] = 0.0; }
    TM::sync();
    for (int j = 1; j < N; j++) {
        const double *prev = prevbuf ? prevbuf : tri + nu_col(j - 1);
        double *col = tri + nu_col(j);
        int16_t *kcol = K + nu_col(j);
        const int64_t c0 = cp[j], nc = cp[j + 1] - c0;
        for (int64_t s = 0; s == 0 || s < nc; s += L.chunk) {
            const int cn = (int)(nc - s < L.chunk ? nc - s : L.chunk);
            const bool first = s == 0, last = s + L.chunk >= nc;
            for (int q = rank; q < cn; q += T) {
                const int k = nb.pk[c0 + s + q];
                ck[q] = (int16_t)k; ce[q] = nb.pe[c0 + s + q]; ca[q] = prev[k + 1];
            }
            TM::sync();
            for (int ib = rank - lane; ib < j; ib += T) {        // ib: the warp's first row
                const int i = ib + lane;
                const bool row = i < j;
                int lo = 0, hi = cn;                              // first staged k >= ib
                while (lo < hi) { const int m = (lo + hi) >> 1; if (ck[m] < ib) lo = m + 1; else hi = m; }
                double best = NU_NONE; int bk = -1;
                if (!first && row) { best = sbest[i]; bk = sbk[i]; }
                for (int q = lo; q < cn; q++) {
                    const int k = ck[q];
                    if (row && k >= i) {
                        const double left = k > i ? tri[nu_col(k - 1) + i] : 0.0;
                        const double tot = __dadd_rn(__dadd_rn(left, ca[q]), ce[q]);
                        if (tot < best) { best = tot; bk = k; }
                    }
                }
                if (row) {
                    if (last) {
                        const double unp = prev[i];
                        if (best <= unp) { col[i] = best; kcol[i] = (int16_t)bk; }
                        else { col[i] = unp; kcol[i] = -1; }
                    } else { sbest[i] = best; sbk[i] = (int16_t)bk; }
                }
            }
            TM::sync();
        }
        if (rank == 0) col[j] = 0.0;
        if (prevbuf) {
            TM::sync();
            for (int i = rank; i <= j; i += T) prevbuf[i] = col[i];
        }
        TM::sync();
    }
    if (rank == 0) {
        // BackTrack from (0, N-1) (SQRNalgos.BackTrack, partial=False): the intervals on the stack are disjoint, so
        // every position is in at most one pair and emitting by position gives the pairs sorted by (v, w)
        const uint8_t *sq = nb.sym + o;
        int32_t *pre = (int32_t *)smem;
        int32_t *partner = (int32_t *)(smem + nu_al(4 * (size_t)(N + 1)));
        int32_t *stk = (int32_t *)(smem + nu_al(4 * (size_t)(N + 1)) + nu_al(4 * (size_t)N));
        sep_prefix(sq, N, pre);
        for (int p = 0; p < N; p++) partner[p] = -1;
        const int ml = nb.minloop;
        // a separator in [lo, hi)
        auto sep = [&](int lo_, int hi_) { return hi_ > lo_ && pre[hi_] - pre[lo_] > 0; };
        int sp = 0;
        if (N >= 2) { stk[0] = 0; stk[1] = N - 1; sp = 1; }
        while (sp > 0) {
            sp--;
            const int i = stk[2 * sp], j = stk[2 * sp + 1];
            const int k = K[nu_col(j) + i];
            if (k < 0) {                                            // j unpaired: shrink from the right
                const int gap = (j - 1) - i;
                if (gap > ml || (gap > 0 && sep(i + 1, j - 1))) { stk[2 * sp] = i; stk[2 * sp + 1] = j - 1; sp++; }
                continue;
            }
            partner[k] = j;
            const int left = (k - 1) - i;
            if (left > ml || (left > 0 && sep(i + 1, k - 1))) { stk[2 * sp] = i; stk[2 * sp + 1] = k - 1; sp++; }
            const int inner = (j - 1) - (k + 1);
            if (inner > ml || (inner > 0 && sep(k + 2, j - 1))) { stk[2 * sp] = k + 1; stk[2 * sp + 1] = j - 1; sp++; }
        }
        int32_t *out = nb.out_pairs + 2 * nb.out_base[seq];
        int n = 0;
        for (int v = 0; v < N; v++)
            if (partner[v] >= 0) { out[2 * n] = v; out[2 * n + 1] = partner[v]; n++; }
        nb.out_n[seq] = n;
    }
    TM::sync();
}

// ---- host side: checks and the candidate lists (shared by the library and the emulation build) ----

// Stems (i, j, len) of one sequence of N positions: every pair (i+t, j-t), t < len, inside [0, N), len >= 1.
inline bool nu_stems_ok(int N, const int32_t *st, int64_t ns)
{
    for (int64_t s = 0; s < ns; s++) {
        const int64_t i = st[3 * s], j = st[3 * s + 1], ln = st[3 * s + 2];
        if (ln < 1 || i < 0 || j >= N || i + ln - 1 >= N || j - ln + 1 < 0) return false;
    }
    return true;
}

// The pairs (k, j), k + min_span <= j, of the stems of one sequence, each once with the index of the LAST stem that
// holds it (what a dict filled in stem order keeps), sorted by (j, k).  A key is j (SP_J bits) | k | stem index: 15 bits
// each for positions up to SQRN_MAX_LEN, 34 for the stem.
constexpr int SP_J = 49, SP_K = 34;
constexpr uint64_t SP_POS = 0x7fff, SP_STEM = (1ull << SP_K) - 1;

inline void stem_pair_keys(const int32_t *st, int64_t ns, int min_span, std::vector<uint64_t> &out)
{
    std::vector<uint64_t> keys;
    for (int64_t s = 0; s < ns; s++)
        for (int t = 0; t < st[3 * s + 2]; t++) {
            const int64_t k = st[3 * s] + t, j = st[3 * s + 1] - t;
            if (k + min_span <= j) keys.push_back((uint64_t)j << SP_J | (uint64_t)k << SP_K | (uint64_t)s);
        }
    std::sort(keys.begin(), keys.end());
    out.clear();
    for (size_t q = 0; q < keys.size(); q++)
        if (q + 1 == keys.size() || keys[q + 1] >> SP_K != keys[q] >> SP_K) out.push_back(keys[q]);   // else a later stem holds it too
}

// P(j) of one sequence: counts[j] partners per column, then k ascending within each column, energies -score.  Pairs
// with k >= j - 1 can never be taken and are left out.
inline void nu_seq_lists(int N, const int32_t *st, const double *sc, int64_t ns, std::vector<int64_t> &counts,
                         std::vector<int16_t> &pk, std::vector<double> &pe)
{
    std::vector<uint64_t> keys;
    stem_pair_keys(st, ns, 2, keys);
    counts.assign((size_t)N, 0);
    pk.clear(); pe.clear();
    for (const uint64_t key : keys) {
        counts[(size_t)(key >> SP_J)]++;
        pk.push_back((int16_t)(key >> SP_K & SP_POS));
        pe.push_back(-sc[key & SP_STEM]);
    }
}

}  // namespace sqrn
