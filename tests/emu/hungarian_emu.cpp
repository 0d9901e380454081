// hungarian_emu.cpp -- TEST INFRASTRUCTURE: host build of the assignment and the filter in
// squarna_b200/csrc/sqrn_hungarian.cuh (SQRN_HOST_EMU), so that `pytest -m "not gpu"` checks them against SciPy's
// linear_sum_assignment and squarna_b200/SQRNalgos.Hungarian on a box without a GPU.  The scan of each step runs for a
// simulated team of `width` lanes (1; 32: the warp tier; 256: the CTA and global tiers, which run the same item
// function with the state in shared memory or in a workspace slot) and the partial keys are combined in the device's
// order.  It is not linked into libsqrn_b200.so; barriers and concurrency are only covered by the `-m gpu` tests.
#define SQRN_HOST_EMU 1
#include <stdlib.h>
#include "../../squarna_b200/csrc/sqrn_params.h"
#include "../../squarna_b200/csrc/sqrn_hungarian.cuh"

using namespace sqrn;

extern "C" int emu_hu_smem_max_n(long long budget) { return hu_smem_max_n((size_t)budget); }

// One sequence through hu_item with a team of `width` lanes; col4row (N) receives the assignment when given.
static int run_item(int N, const uint8_t *sym, const int64_t *rowptr, const int16_t *acol, const double *acost,
                    int minloop, int width, int32_t *pairs, int32_t *col4row)
{
    const int64_t one_off[2] = {0, N}, base = 0;
    int32_t n_out = 0;
    HuBatch hb{};
    hb.n_items = 1; hb.off = one_off; hb.sym = sym;
    hb.rowptr = rowptr; hb.acol = acol; hb.acost = acost; hb.minloop = minloop;
    hb.out_base = &base; hb.out_pairs = pairs; hb.out_n = &n_out;
    const HuLayout L = hu_layout(N);
    std::vector<double> state(L.total / 8 + 2);
    unsigned char *st = (unsigned char *)state.data();
    if (width == 1) hu_item<HuEmuTeam<1>>(hb, 0, st, L, nullptr);
    else if (width == 32) hu_item<HuEmuTeam<32>>(hb, 0, st, L, nullptr);
    else if (width == 256) hu_item<HuEmuTeam<256>>(hb, 0, st, L, nullptr);
    else return -1;
    if (col4row)
        for (int p = 0; p < N; p++) col4row[p] = ((int16_t *)(st + L.c4r))[p];
    return n_out;
}

// The assignment alone on an adjacency (rowptr [N+1], acol / acost): col4row [N] out.
extern "C" int emu_lsap(int N, const int64_t *rowptr, const int16_t *acol, const double *acost, int width, int32_t *col4row)
{
    std::vector<uint8_t> sym((size_t)N + 1, 'A');
    std::vector<int32_t> pairs((size_t)N + 2);
    return run_item(N, sym.data(), rowptr, acol, acost, 0, width, pairs.data(), col4row) < 0 ? SQRN_E_BADARG : SQRN_OK;
}

// Same arguments as sqrn_hungarian_batch, plus the team width; the same checks.
extern "C" int emu_hungarian(int64_t n_seqs, const int64_t *off, const uint8_t *sym, const int64_t *so,
                             const int32_t *stems, const double *scores, int minloop, double power, int width,
                             int64_t *pair_offsets, int32_t *pairs)
{
    if (minloop < 0) return SQRN_E_BADARG;
    pair_offsets[0] = 0;
    for (int64_t b = 0; b < n_seqs; b++) {
        const int N = (int)(off[b + 1] - off[b]);
        const int64_t ns = so[b + 1] - so[b];
        if (N > SQRN_MAX_LEN || (ns > 0 && !hu_stems_ok(N, stems + 3 * so[b], ns))) return SQRN_E_BADARG;
        std::vector<double> w;
        if (ns > 0 && !hu_weights(scores + so[b], ns, power, w)) return SQRN_E_BADARG;
        std::vector<int64_t> rowptr;
        std::vector<int16_t> acol;
        std::vector<double> acost;
        hu_seq_adjacency(N, stems + 3 * so[b], w.data(), ns, rowptr, acol, acost);
        const int n = N > 0 ? run_item(N, sym + off[b], rowptr.data(), acol.data(), acost.data(), minloop, width,
                                       pairs + 2 * pair_offsets[b], nullptr) : 0;
        if (n < 0) return SQRN_E_BADARG;
        pair_offsets[b + 1] = pair_offsets[b] + n;
    }
    return SQRN_OK;
}
