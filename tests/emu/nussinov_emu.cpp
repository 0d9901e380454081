// nussinov_emu.cpp -- TEST INFRASTRUCTURE: single-thread host build of the Nussinov DP and backtrack in
// squarna_b200/csrc/sqrn_nussinov.cuh (SQRN_HOST_EMU, team size 1), so that `pytest -m "not gpu"` checks them against
// squarna_b200/SQRNalgos.Nussinov on a box without a GPU.  It is not linked into libsqrn_b200.so; the parallel
// behaviour (barriers between columns, warps walking the candidates in step) is only covered by the `-m gpu` tests.
#define SQRN_HOST_EMU 1
#include <stdlib.h>
#include "../../squarna_b200/csrc/sqrn_params.h"
#include "../../squarna_b200/csrc/sqrn_nussinov.cuh"

using namespace sqrn;

extern "C" int emu_nu_smem_max_n(long long budget) { return nu_smem_max_n((size_t)budget); }

// tier 0: the shared-memory tier (triangle read in place); tier 1: the global tier (a copy of the previous column,
// `chunk` staged candidates per pass, the row state kept across passes).  Same arguments as sqrn_nussinov_batch.
extern "C" int emu_nussinov(int64_t n_seqs, const int64_t *off, const uint8_t *sym, const int64_t *so,
                            const int32_t *stems, const double *scores, int minloop, int tier, int chunk,
                            int64_t *pair_offsets, int32_t *pairs)
{
    if (minloop < 0 || chunk < 1) return SQRN_E_BADARG;
    pair_offsets[0] = 0;
    for (int64_t b = 0; b < n_seqs; b++) {
        const int N = (int)(off[b + 1] - off[b]);
        const int64_t ns = so[b + 1] - so[b];
        if (N > SQRN_MAX_LEN || (ns > 0 && !nu_stems_ok(N, stems + 3 * so[b], ns))) return SQRN_E_BADARG;
        std::vector<int64_t> cnt, colptr((size_t)N + 1, 0);
        std::vector<int16_t> pk;
        std::vector<double> pe;
        nu_seq_lists(N, stems + 3 * so[b], scores + so[b], ns, cnt, pk, pe);
        for (int j = 0; j < N; j++) colptr[(size_t)j + 1] = colptr[(size_t)j] + cnt[(size_t)j];
        const int64_t one_off[2] = {0, N}, base = 0;
        int32_t n_out = 0;
        NuBatch nb{};
        nb.n_items = 1; nb.off = one_off; nb.sym = sym + off[b];
        nb.colptr = colptr.data(); nb.pk = pk.data(); nb.pe = pe.data(); nb.minloop = minloop;
        nb.out_base = &base; nb.out_pairs = pairs + 2 * pair_offsets[b]; nb.out_n = &n_out;
        const NuLayout L = nu_layout(N, tier == 0, chunk);
        std::vector<double> smem(L.total / 8 + 2), tri(tier == 0 ? 0 : (size_t)nu_cells(N) + 1), sbest((size_t)N + 1);
        std::vector<int16_t> K((size_t)nu_cells(N) + 1), sbk((size_t)N + 1);
        unsigned char *sm = (unsigned char *)smem.data();
        nu_item<0>(nb, 0, tier == 0 ? (double *)sm : tri.data(), tier == 0 ? nullptr : (double *)(sm + L.prev_off), L, sm,
                   K.data(), sbest.data(), sbk.data());
        pair_offsets[b + 1] = pair_offsets[b] + n_out;
    }
    return SQRN_OK;
}
