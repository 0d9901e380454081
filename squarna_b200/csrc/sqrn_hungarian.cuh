// sqrn_hungarian.cuh -- the Hungarian builder of SQRNalgos (squarna_b200/SQRNalgos.py: Hungarian) on the device:
// SciPy's linear_sum_assignment (rectangular_lsap.cpp: Crouse's shortest augmenting path) on the symmetric N x N
// cost matrix of the stem pairs, then the pair filter.  One team (a warp or a CTA) per sequence.
//
//   cost[v][w] = cost[w][v] = -(score ** power) for a pair (v, w), v < w, of a stem (the later stem's score when two
//   stems hold it); +0.0 everywhere else.
//
// No N x N matrix exists anywhere.  The adjacency (row CSR, both orientations, cost per entry) is read-only; before each
// step of the search the row of the current i is scattered into a dense row: cval[j] is cost[i][j] where cstamp[j] == i,
// and 0.0 is read where it is not, which is SciPy's arithmetic on its zero cells.  A row's scatter only overwrites
// entries of other rows, so nothing is ever cleared.
//
// For curRow = 0 .. N-1 the search repeats steps until it reaches an unassigned column.  A step scans the remaining
// columns: r = ((minVal + cost[i][j]) - u[i]) - v[j], spc[j] = r and path[j] = i where r < spc[j]; then it picks, among
// the minimum spc, the LAST unassigned position if there is one, else the FIRST position -- what SciPy's sequential
// `spc < lowest || (spc == lowest && row4col == -1)` keeps.  The lanes scan strided positions and the pick is a team
// minimum of the key (order-preserving image of spc with -0.0 read as +0.0, assigned, assigned ? it : N-1-it), which
// is unique per position and so independent of the order the partial keys meet in.  The picked column is swapped to
// the tail of `remaining` (SciPy drops it; the order of the live part is the same), so after the search the tail holds
// the columns SC of the search, and the rows SR are curRow and the rows assigned to SC other than the sink.  The duals
// and the augment follow SciPy operation for operation, without FMA.
//
// State per sequence: u v spc cval (f64), path row4col col4row remaining cstamp (int16): 42 bytes a position.  The
// same functions compile for the host (SQRN_HOST_EMU, tests/emu/hungarian_emu.cpp), where HuEmuTeam runs the scan of a
// simulated team lane after lane and combines the partial keys in the device's order.
#pragma once
#include <cmath>
#include "sqrn_nussinov.cuh"

namespace sqrn {

constexpr int HU_WARP_MAX_N = 256;  // warp tier: sequences of up to 8 positions a lane
constexpr int HU_WPC = 8;           // warp tier: warps (sequences) per CTA
constexpr int HU_CTA_TW = 8;        // CTA and global tiers: 256 threads a sequence
constexpr double HU_INF = __builtin_huge_val();

struct HuLayout { size_t u, v, spc, cval, path, r4c, c4r, rem, stamp, total; };

__host__ __device__ inline HuLayout hu_layout(int n)
{
    HuLayout L{};
    size_t off = 0;
    const size_t d = nu_al(8 * (size_t)n), h = nu_al(2 * (size_t)n);
    L.u = off; off += d;
    L.v = off; off += d;
    L.spc = off; off += d;
    L.cval = off; off += d;
    L.path = off; off += h;
    L.r4c = off; off += h;
    L.c4r = off; off += h;
    L.rem = off; off += h;
    L.stamp = off; off += h;
    L.total = off;
    return L;
}

struct HuKey { uint64_t v; uint32_t s; };

__host__ __device__ __forceinline__ HuKey hu_none() { return HuKey{~0ull, ~0u}; }
__host__ __device__ __forceinline__ HuKey hu_min(HuKey a, HuKey b) { return b.v < a.v || (b.v == a.v && b.s < a.s) ? b : a; }

// ascending doubles -> ascending integers; -0.0 and +0.0 (equal for SciPy's comparisons) get the same image
__device__ __forceinline__ uint64_t hu_image(double x)
{
    x = __dadd_rn(x, 0.0);
#ifndef SQRN_HOST_EMU
    uint64_t u = (uint64_t)__double_as_longlong(x);
#else
    uint64_t u; memcpy(&u, &x, 8);
#endif
    return (u >> 63) ? ~u : (u | 0x8000000000000000ull);
}

// the key of position `it` of `remaining` (column j): 1 bit assigned | 15 bits ordinal | 15 bits j
__device__ __forceinline__ HuKey hu_key(double spc, bool assigned, int it, int j, int N)
{
    return HuKey{hu_image(spc), (uint32_t)assigned << 30 | (uint32_t)(assigned ? it : N - 1 - it) << 15 | (uint32_t)j};
}

// Dynamic shared memory of a CTA: the CTA tier holds the state, the reduction scratch (one key a warp) and the item
// number; the global tier only the last two; the warp tier HU_WPC states.
__host__ __device__ inline size_t hu_cta_smem(int n, bool state) { return (state ? hu_layout(n).total : 0) + 16 * HU_CTA_TW + 16; }
__host__ __device__ inline size_t hu_warp_smem(int n) { return HU_WPC * hu_layout(n).total; }

// Longest sequence whose state fits `budget` bytes of dynamic shared memory per CTA (the CTA tier).
inline int hu_smem_max_n(size_t budget)
{
    int n = 0;
    while (n < SQRN_MAX_LEN && hu_cta_smem(n + 1, true) <= budget) n++;
    return n;
}

// A batch as the kernels see it.  Sequence b: row v of its adjacency is acol / acost [rowptr[off[b] + b + v] ..
// rowptr[off[b] + b + v + 1]).
struct HuBatch {
    int n_items; const int32_t *order;          // sequences of this launch, longest first
    const int64_t *off; const uint8_t *sym;
    const int64_t *rowptr; const int16_t *acol; const double *acost;
    int minloop;
    const int64_t *out_base; int32_t *out_pairs; int32_t *out_n;   // sequence b: up to N/2 pairs at out_base[b]; -1: infeasible
    int *counter;
    unsigned char *ws; int64_t slot_bytes;      // global tier: the state of CTA c at ws + c * slot_bytes
};

#ifndef SQRN_HOST_EMU
// TW == 1: a warp per sequence; TW > 1: a CTA.  argmin returns the team minimum of f(lane, T) to every thread; it is a
// barrier of the team.  red: TW keys of shared scratch (CTA teams).
template <int TW> struct HuTeam {
    static constexpr int T = TW * 32;
    __device__ static __forceinline__ int rank() { return Team<TW>::rank(); }
    __device__ static __forceinline__ void sync() { Team<TW>::sync(); }
    template <class F> __device__ static __forceinline__ HuKey argmin(F f, HuKey *red)
    {
        HuKey k = f(rank(), T);
        const uint32_t hi = (uint32_t)(k.v >> 32), lo = (uint32_t)k.v;
        const uint32_t mh = __reduce_min_sync(0xffffffffu, hi);
        bool in = hi == mh;
        const uint32_t ml = __reduce_min_sync(0xffffffffu, in ? lo : 0xffffffffu);
        in = in && lo == ml;
        const uint32_t ms = __reduce_min_sync(0xffffffffu, in ? k.s : 0xffffffffu);
        k.v = (uint64_t)mh << 32 | ml; k.s = ms;
        if (TW == 1) { __syncwarp(); return k; }
        if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = k;
        __syncthreads();
        k = red[0];
        #pragma unroll
        for (int w = 1; w < TW; w++) k = hu_min(k, red[w]);
        return k;
    }
};
#else
// A team of W lanes simulated on one thread: the parallel loops run with one thread, the scan lane after lane; the
// partial keys meet as on the device (a tree within each warp, then the warps in order).
template <int W> struct HuEmuTeam {
    static constexpr int T = 1;
    static inline int rank() { return 0; }
    static inline void sync() {}
    template <class F> static HuKey argmin(F f, HuKey *)
    {
        HuKey k[W];
        for (int l = 0; l < W; l++) k[l] = f(l, W);
        for (int g = 0; g < W; g += 32) {
            const int n = W - g < 32 ? W - g : 32;
            for (int d = 16; d > 0; d >>= 1)
                for (int l = 0; l < d && l + d < n; l++) k[g + l] = hu_min(k[g + l], k[g + l + d]);
        }
        HuKey r = k[0];
        for (int g = 32; g < W; g += 32) r = hu_min(r, k[g]);
        return r;
    }
};
#endif

// One sequence of N >= 1 positions: the assignment (whole team), the filter (whole team) and the output (rank 0).
// st: the state (HuLayout) in shared memory or in the CTA's slot.
template <class TM>
__device__ void hu_item(const HuBatch &hb, int seq, unsigned char *st, const HuLayout &L, HuKey *red)
{
    constexpr int T = TM::T;
    const int rank = TM::rank();
    const int64_t o = hb.off[seq];
    const int N = (int)(hb.off[seq + 1] - o);
    const int64_t *rp = hb.rowptr + o + seq;
    double *u = (double *)(st + L.u), *v = (double *)(st + L.v), *spc = (double *)(st + L.spc), *cval = (double *)(st + L.cval);
    int16_t *path = (int16_t *)(st + L.path), *r4c = (int16_t *)(st + L.r4c), *c4r = (int16_t *)(st + L.c4r);
    int16_t *rem = (int16_t *)(st + L.rem), *stamp = (int16_t *)(st + L.stamp);
    for (int p = rank; p < N; p += T) { u[p] = 0.0; v[p] = 0.0; r4c[p] = -1; c4r[p] = -1; stamp[p] = -1; }
    TM::sync();
    for (int cur = 0; cur < N; cur++) {
        int i = cur, nrem = N, sink = -1;
        double minVal = 0.0;
        for (bool first = true; sink < 0; first = false) {
            for (int64_t q = rp[i] + rank; q < rp[i + 1]; q += T) {
                const int c = hb.acol[q];
                cval[c] = hb.acost[q]; stamp[c] = (int16_t)i;
            }
            TM::sync();
            const double ui = u[i], mv = minVal;
            const int ci = i, nr = nrem;
            const HuKey k = TM::argmin([&](int lane, int W) {
                HuKey best = hu_none();
                for (int it = lane; it < nr; it += W) {
                    int j;
                    if (first) { j = N - 1 - it; rem[it] = (int16_t)j; }    // remaining = N-1 .. 0, spc = +inf
                    else j = rem[it];
                    const double c = stamp[j] == ci ? cval[j] : 0.0;
                    const double r = __dsub_rn(__dsub_rn(__dadd_rn(mv, c), ui), v[j]);
                    double s = first ? HU_INF : spc[j];
                    if (r < s) { path[j] = (int16_t)ci; spc[j] = r; s = r; }
                    best = hu_min(best, hu_key(s, r4c[j] >= 0, it, j, N));
                }
                return best;
            }, red);
            const int j = (int)(k.s & 0x7fff), ord = (int)(k.s >> 15 & 0x7fff);
            const int it = (k.s >> 30) ? ord : N - 1 - ord;
            minVal = spc[j];
            if (minVal == HU_INF) {                            // SciPy: "cost matrix is infeasible"
                if (rank == 0) hb.out_n[seq] = -1;
                return;
            }
            if (rank == 0) { rem[it] = rem[nrem - 1]; rem[nrem - 1] = (int16_t)j; }
            nrem--;
            if (r4c[j] < 0) sink = j; else i = r4c[j];
        }
        // duals over SC = remaining[nrem ..] (position nrem: the sink, swapped there by rank 0 just now)
        for (int q = nrem + rank; q < N; q += T) {
            const int j = q == nrem ? sink : rem[q];
            const double d = __dsub_rn(minVal, spc[j]);
            v[j] = __dsub_rn(v[j], d);
            if (j != sink) { const int r = r4c[j]; u[r] = __dadd_rn(u[r], d); }
        }
        if (rank == 0) u[cur] = __dadd_rn(u[cur], minVal);
        TM::sync();
        if (rank == 0)
            for (int j = sink;;) {
                const int r = path[j];
                r4c[j] = (int16_t)r;
                const int t = c4r[r];
                c4r[r] = (int16_t)j; j = t;
                if (r == cur) break;
            }
    }
    // the filter: (k, l) with k < l - minloop or a separator in seq[k+1 : l], mutual, on a non-zero cost cell.  spc
    // (8N bytes) takes the N + 1 separator counts, path the flags.
    TM::sync();
    int32_t *pre = (int32_t *)spc;
    if (rank == 0) sep_prefix(hb.sym + o, N, pre);
    TM::sync();
    for (int k = rank; k < N; k += T) {
        const int l = c4r[k];
        bool keep = false;
        if (l > k && c4r[l] == k && (k < l - hb.minloop || pre[l] - pre[k + 1] > 0))
            for (int64_t q = rp[k]; q < rp[k + 1]; q++)
                if (hb.acol[q] == l) { keep = hb.acost[q] != 0.0; break; }
        path[k] = keep;
    }
    TM::sync();
    if (rank == 0) {
        int32_t *out = hb.out_pairs + 2 * hb.out_base[seq];
        int n = 0;
        for (int k = 0; k < N; k++)
            if (path[k]) { out[2 * n] = k; out[2 * n + 1] = c4r[k]; n++; }
        hb.out_n[seq] = n;
    }
    TM::sync();
}

// ---- host side: checks and the adjacency (shared by the library and the emulation build) ----

// Stems of one sequence for this builder: those nu_stems_ok takes whose every pair (i+t, j-t) has i+t < j-t.
inline bool hu_stems_ok(int N, const int32_t *st, int64_t ns)
{
    if (!nu_stems_ok(N, st, ns)) return false;
    for (int64_t s = 0; s < ns; s++)
        if ((int64_t)st[3 * s] + st[3 * s + 2] - 1 >= (int64_t)st[3 * s + 1] - st[3 * s + 2] + 1) return false;
    return true;
}

// w[s] = pow(score, power) per stem (CPython's float ** for a finite base >= 0); false when a score is negative or NaN
// or a weight is not finite (the host builder then has complex numbers or an infeasible matrix).
inline bool hu_weights(const double *sc, int64_t ns, double power, std::vector<double> &w)
{
    w.resize((size_t)ns);
    for (int64_t s = 0; s < ns; s++) {
        if (!(sc[s] >= 0.0)) return false;
        w[(size_t)s] = pow(sc[s], power);
        if (!std::isfinite(w[(size_t)s])) return false;
    }
    return true;
}

// The adjacency of one sequence: rowptr [N+1], then per row its partners (either orientation) with cost -(weight).
inline void hu_seq_adjacency(int N, const int32_t *st, const double *w, int64_t ns, std::vector<int64_t> &rowptr,
                             std::vector<int16_t> &col, std::vector<double> &cost)
{
    std::vector<uint64_t> keys;
    stem_pair_keys(st, ns, 1, keys);
    rowptr.assign((size_t)N + 1, 0);
    for (const uint64_t key : keys) { rowptr[(key >> SP_K & SP_POS) + 1]++; rowptr[(key >> SP_J) + 1]++; }
    for (int p = 0; p < N; p++) rowptr[(size_t)p + 1] += rowptr[(size_t)p];
    col.resize(2 * keys.size()); cost.resize(2 * keys.size());
    std::vector<int64_t> at(rowptr.begin(), rowptr.end() - 1);
    for (const uint64_t key : keys) {
        const int k = (int)(key >> SP_K & SP_POS), j = (int)(key >> SP_J);
        const double c = -w[key & SP_STEM];
        col[(size_t)at[(size_t)k]] = (int16_t)j; cost[(size_t)at[(size_t)k]++] = c;
        col[(size_t)at[(size_t)j]] = (int16_t)k; cost[(size_t)at[(size_t)j]++] = c;
    }
}

}  // namespace sqrn
