/*
 * sqrn.h -- C ABI of libsqrn_b200.so, the B200 (sm_100a) implementation of
 * SQUARNA's greedy single-sequence hot path.
 *
 * The reference (febos/SQUARNA) is pure Python and has no FFI of its own; the
 * seam this library replaces is
 *
 *   SQRNdbnseq.py:1076-1085  BPMatrix (+ alignment weighting)
 *   SQRNdbnseq.py:1102-1199  the "G" block: pool loop over OptimalStems
 *                            (AnnotateStems 427-495, ScoreStems 607-751,
 *                             ChooseStems 754-789)
 *   SQRNdbnseq.py:1201-1236  dedupe, ScoreStruct 861-899, RankStructs 902-955,
 *                            PairsToDBN 104-163, ConsensusStemSet 845-858
 *   SQRNdbnali.py:86-101     YieldStems (BPMatrix + AnnotateStems only)
 *
 * batched over sequences x parameter sets.  The Python drivers in
 * squarna_b200/ (SQRNdbnseq / RunSQRNdbnseq / SQRNdbnali / Predict / Main) call
 * these entry points through ctypes; INTEGRATION.md shows the binding a
 * maintainer of the reference would add.
 *
 * Conventions
 *   - plain C, no exceptions cross the boundary; every call returns 0 (SQRN_OK)
 *     or a negative error class, sqrn_last_error() gives the message;
 *   - the caller owns every buffer; the library never keeps caller pointers
 *     after a call returns;
 *   - a context belongs to one GPU and one host thread at a time (one process
 *     or thread per GPU; ctypes releases the GIL during calls);
 *   - there is NO CPU fallback: without a usable CUDA device every compute
 *     entry point fails with SQRN_E_CUDA.
 */
#ifndef SQRN_H
#define SQRN_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(__GNUC__)
#define SQRN_API __attribute__((visibility("default")))
#else
#define SQRN_API
#endif

#define SQRN_ABI_VERSION 3

#define SQRN_OK             0
#define SQRN_E_BADARG      -1
#define SQRN_E_CAPACITY    -2   /* an output buffer is too small; needed sizes are written back */
#define SQRN_E_CUDA        -3
#define SQRN_E_UNSUPPORTED -4
#define SQRN_E_NOMEM       -5   /* host allocation failed */

#define SQRN_MAX_BPKEYS 32
#define SQRN_MAX_LEN    16000    /* ungapped nucleotides per sequence */
#define SQRN_MAX_REACT_LUT 2048

typedef struct sqrn_ctx sqrn_ctx;

/* One parameter set of a .conf file (SQUARNA.py:15-77 ParseConfig; fields read
 * at SQRNdbnseq.py:1050-1062).  bpweights keeps the dict order because later
 * keys overwrite earlier ones in either orientation (SQRNdbnseq.py:282-284). */
typedef struct {
    int32_t n_bp;                          /* number of bpweights entries        */
    uint8_t bp_keys[2 * SQRN_MAX_BPKEYS];  /* two symbols per entry ("GC", ...)  */
    double  bp_vals[SQRN_MAX_BPKEYS];
    double  suboptmax, suboptmin, suboptsteps;
    double  minlen, minbpscore, minfinscorefactor;
    double  bracketweight, distcoef, orderpenalty, loopbonus, maxstemnum;
} sqrn_paramset;

/* restraint classes, one byte per position (ParseRestraints, SQRNdbnseq.py:370-376) */
#define SQRN_RC_UNPAIRED 1   /* '_' '+' */
#define SQRN_RC_NOLEFT   2   /* '/'  : may not be the 3' partner (j) */
#define SQRN_RC_NORIGHT  4   /* '\\' : may not be the 5' partner (i) */

/* A CSR batch of ungapped sequences (what SQRNdbnseq.py:1004-1037 produces per
 * sequence: upper-cased, T->U, gaps removed, restraints parsed).              */
typedef struct {
    int64_t        n_seqs;
    const int64_t *offsets;      /* [n_seqs+1] into symbols / react_code / restr_class / cols */
    const uint8_t *symbols;      /* raw ASCII; case and T/U are normalised by the library       */
    /* reactivities: NULL = all 0.5 ("default reacts", SQRNdbnseq.py:273).  Else one
     * code per position into react_values (the distinct processed reactivities of
     * the batch).  Up to SQRN_MAX_REACT_LUT distinct values the reactivity factors
     * ((1-(ri+rj)/2)*2)**0.5 come from a host libm table (bit-exact); above that the
     * device evaluates sqrt() (<= 1 ulp from libm pow on ~0.1 % of inputs).         */
    const uint16_t *react_code;
    const double  *react_values;
    int32_t        n_react_values;
    int32_t        react_sum_compensated; /* builtin sum() over exact Python floats (CPython >= 3.12) */
    /* restraints: both NULL = none */
    const uint8_t *restr_class;  /* SQRN_RC_* flags per position */
    const int64_t *rbp_offsets;  /* [n_seqs+1] into rbps (pairs) */
    const int32_t *rbps;         /* (v, w) per restraint pair, v < w, local coordinates */
    /* alignment weighting (SQRNdbnseq.py:1031-1034, 1084-1085): score *= smat[cols[i], cols[j]] */
    const double  *smat;         /* [smat_L x smat_L] row-major or NULL */
    int32_t        smat_L;
    const int32_t *cols;         /* aligned column of every ungapped position */
    /* flags of SQRNdbnseq (SQRNdbnseq.py:973-980) */
    int32_t interchainonly, hardrest, rankbydiff;
    int32_t poollim, conslim, max_structs;   /* max_structs: structures returned per sequence (<=0: all) */
    int32_t rankby[3];
    uint64_t priority_mask;      /* bit p: parameter set p has priority (RankStructs 912-913) */
    /* base-pair-probability weighting of the score matrix (BPMatrix, SQRNdbnseq.py:341-365), ABI >= 2.  The host
     * evaluates the probabilities (ViennaRNA in the reference) and hands over, per sequence b, one row-major
     * N_b x N_b float64 matrix term[i * N_b + j] = (bpp[i, j] / max bpp) ** |power| at element offset
     * bpp_offsets[b].  bpp_mode 1: scoremat += term (the reference's negative powers), 2: scoremat *= term
     * (positive powers), 0: no weighting.  The term belongs to ONE parameter set: sqrn_predict_batch accepts it
     * only with n_ps == 1 (parameter sets with different powers are separate calls). */
    const double  *bpp_term;
    const int64_t *bpp_offsets;  /* [n_seqs+1] */
    int32_t        bpp_mode;
} sqrn_batch;

/* Results, caller-allocated.  Sequence b owns structures
 * [struct_offsets[b], struct_offsets[b+1]) in final rank order; structure k owns
 * stems [stem_offsets[k], stem_offsets[k+1]) in selection order and N_b dbn
 * bytes at dbn + dbn_offsets[k].  On SQRN_E_CAPACITY need_* say what to allocate. */
typedef struct {
    int64_t  cap_structs, cap_stems, cap_dbn;
    int64_t *struct_offsets;     /* [n_seqs+1] */
    double  *scores;             /* [cap_structs*3] total, struct, react, each round(x,3) (ScoreStruct 899) */
    uint8_t *struct_is_int0;     /* [cap_structs] structscore is the int 0 (prints "0") */
    uint64_t*psmask;             /* [cap_structs] parameter sets that produced the structure */
    int32_t *n_total;            /* [n_seqs] structures found before truncation to max_structs */
    int64_t *stem_offsets;       /* [cap_structs+1] */
    int32_t *stems;              /* [cap_stems*3] i, j, len (outermost pair, length) */
    int64_t *dbn_offsets;        /* [cap_structs] */
    int8_t  *dbn;                /* [cap_dbn] 0 '.', +L opening bracket of level L, -L closing */
    int8_t  *cons;               /* [total symbols] consensus of the top conslim structures */
    int64_t  need_structs, need_stems, need_dbn;
} sqrn_result;

/* stems of one AnnotateStems pass per sequence (YieldStems, SQRNdbnali.py:60-108) */
typedef struct {
    int64_t  cap_stems;
    int64_t *stem_offsets;       /* [n_seqs+1] */
    int32_t *stems;              /* [cap_stems*3] i, j, len in UNGAPPED coordinates, reference order */
    double  *scores;             /* [cap_stems] bp score */
    int64_t  need_stems;
} sqrn_stems;

SQRN_API int  sqrn_abi_version(void);
SQRN_API int  sqrn_device_count(void);                 /* 0 when no CUDA device is usable */
SQRN_API int  sqrn_ctx_create(int device, sqrn_ctx **out);
SQRN_API void sqrn_ctx_destroy(sqrn_ctx *ctx);
SQRN_API const char *sqrn_last_error(const sqrn_ctx *ctx);   /* ctx may be NULL: last create error */

/* Use an externally owned CUDA stream (cudaStream_t as void*) for all work of
 * this context, e.g. torch.cuda.current_stream().cuda_stream.                 */
SQRN_API int  sqrn_ctx_set_stream(sqrn_ctx *ctx, void *cuda_stream);

/* Tuning / test knobs.  SQRN_TUNE_REGION selects how ScoreStems evaluates the region inside a
 * candidate (SQRNdbnseq.py:665-689): 0 automatic, 1 the reference's position scan, 2 the walk over
 * the selected stems.  All settings give identical results; tests force each one.             */
#define SQRN_TUNE_REGION 1
#define SQRN_TUNE_NO_FAST_KERNEL 2   /* 1: the fast lane uses the general kernel instead of the specialised one */
#define SQRN_TUNE_CLUSTER 3          /* long sequences (> 2048 nt, run to completion): 0 automatic (a thread-block
                                        cluster per sequence when there are too few to fill the SMs one CTA each),
                                        1 never, 2/4/8/16 always with this cluster size */
#define SQRN_TUNE_NO_GLIST 4         /* 1: CTA teams (> 320 nt) rescan the anti-diagonals every greedy step instead of keeping
                                        the persistent candidate list in global memory (k_long) */
#define SQRN_TUNE_GL_REBUILD 5       /* passes between two rebuilds (compaction + re-binning) of that list; 0: the default */
SQRN_API int  sqrn_ctx_set_tuning(sqrn_ctx *ctx, int what, int value);

/* The full "G" path for a batch: replaces SQRNdbnseq.py:1048-1246 (algos == {"G"},
 * bpp == 0).  Host buffers in, host buffers out.                              */
SQRN_API int  sqrn_predict_batch(sqrn_ctx *ctx, const sqrn_paramset *ps, int n_ps,
                        const sqrn_batch *in, sqrn_result *out);

/* Enumeration only: replaces SQRNdbnali.py:86-101 for a batch.                 */
SQRN_API int  sqrn_yield_stems_batch(sqrn_ctx *ctx, const sqrn_paramset *ps,
                            const sqrn_batch *in, sqrn_stems *out);

/* Alignment step 1 (SQRNdbnali.py:211-242, MatrixToDBNs 121-150) for a batch of ALIGNED sequences: the stems of every
 * sequence (as sqrn_yield_stems_batch) summed into the smat_L x smat_L stem-score matrix, per cell in SEQUENCE ORDER
 * (float64 addition order is observable), on the device; the stems never come back to the host.  in->cols maps every
 * ungapped position to its alignment column, in->smat_L is the alignment length, in->smat must be NULL.
 *   matrix     [smat_L * smat_L] row-major, symmetric (the reference adds every score to [v, w] and [w, v]);
 *   threshold  minbpscore * depth: cells >= threshold with w - v >= 4 are what MatrixToDBNs walks;
 *   cells      [cap_cells] their flat indices v * smat_L + w in MatrixToDBNs' order (value descending, index ascending);
 *              *n_cells = how many, or -1 when there are more than cap_cells (or than 65536): the caller then sorts the
 *              matrix itself.                                                                                          */
SQRN_API int  sqrn_stem_matrix_batch(sqrn_ctx *ctx, const sqrn_paramset *ps, const sqrn_batch *in, double *matrix,
                            double threshold, int64_t cap_cells, int64_t *n_cells, int32_t *cells);

/* The Nussinov builder (SQRNalgos.py: Nussinov + BackTrack, what RunAlgo runs for algorithm "N") for a batch, on the
 * device: per sequence the minimum-energy nested structure over the pairs of its stems, energy of a pair = -(score of
 * its stem), followed back from (0, N-1) with the hairpin rule `minloop` and the separators ';' '&' of `symbols`.
 * Host buffers in and out.
 *   offsets      [n_seqs+1], offsets[0] == 0; symbols [offsets[n_seqs]]: the ungapped sequences (N <= SQRN_MAX_LEN);
 *   stem_offsets [n_seqs+1], stems [3 * ...] (i, j, len), scores [...]: as sqrn_yield_stems_batch returns them; a stem
 *                holds the pairs (i+t, j-t), t < len; a pair two stems hold takes the later stem's score;
 *   minloop      >= 0 (RunAlgo passes 3);
 *   pair_offsets [n_seqs+1] out; pairs [2 * sum_b floor(N_b / 2)] int32 out: sequence b's pairs (v, w), sorted, at
 *                pairs + 2 * pair_offsets[b] (a sequence has at most N/2 pairs, so this size always suffices).
 * SQRN_E_BADARG: a stem outside [0, N) or with len < 1, a sequence longer than SQRN_MAX_LEN, minloop < 0.
 * Sequences of up to ~238 positions (the opt-in shared memory of a B200) keep their DP triangle in shared memory, longer
 * ones in a device workspace of at most 4 GiB (at least one 1.28 GB slot at 16 000 nt), which the context keeps at the
 * size of its largest call until sqrn_ctx_destroy; one CTA per sequence either way, longest first, the two tiers run
 * concurrently.                                                                                                      */
SQRN_API int  sqrn_nussinov_batch(sqrn_ctx *ctx, int64_t n_seqs, const int64_t *offsets, const uint8_t *symbols,
                                  const int64_t *stem_offsets, const int32_t *stems, const double *scores,
                                  int32_t minloop, int64_t *pair_offsets, int32_t *pairs);

/* The Hungarian builder (SQRNalgos.py: Hungarian, what RunAlgo runs for algorithm "H") for a batch, on the device: per
 * sequence SciPy's linear_sum_assignment (rectangular_lsap.cpp) on the symmetric N x N matrix with cost -(score **
 * power) at the pairs of its stems and 0 elsewhere, reproduced operation for operation (the same assignment, ties
 * included), then the pairs (k, l) kept by the host builder: mutual, on a non-zero cell, and k < l - minloop or a
 * separator ';' '&' of `symbols` between them.  No N x N matrix is formed.  Host buffers in and out.
 *   offsets, symbols, stem_offsets, stems, scores, pair_offsets, pairs: as sqrn_nussinov_batch (pairs sorted by v);
 *                a stem's pairs (i+t, j-t) must have i+t < j-t; a pair two stems hold takes the later stem's score;
 *   minloop      >= 0 (RunAlgo passes 3);  power: the exponent of the weights (RunAlgo passes 1.7).
 * SQRN_E_BADARG: a stem outside [0, N), with len < 1 or with a pair (v, w), v >= w; a sequence longer than
 * SQRN_MAX_LEN; minloop < 0; a negative or NaN score; a non-finite score ** power (C pow; the host builder has complex
 * numbers or an infeasible matrix there); a reduced cost that overflows (SciPy: infeasible).
 * Sequences of up to 256 positions run a warp each, longer ones a CTA each with the state (42 bytes a position) in
 * shared memory up to ~5 500 positions on a B200 (the opt-in limit), in a device workspace beyond (one slot per SM at
 * most, 1.4 MB at SQRN_MAX_LEN, kept by the context until sqrn_ctx_destroy).  Longest first within each tier; the warp
 * tier runs concurrently with the others.                                                                            */
SQRN_API int  sqrn_hungarian_batch(sqrn_ctx *ctx, int64_t n_seqs, const int64_t *offsets, const uint8_t *symbols,
                                   const int64_t *stem_offsets, const int32_t *stems, const double *scores,
                                   int32_t minloop, double power, int64_t *pair_offsets, int32_t *pairs);

/* The Edmonds builder (SQRNalgos.py: Edmonds, what RunAlgo runs for algorithm "E") for a batch, on the device: per
 * sequence NetworkX's max_weight_matching (networkx/algorithms/matching.py, maxcardinality False) on the graph whose
 * edges are the pairs of its stems, weight score ** power, reproduced statement for statement (the same matching, ties
 * included).  An edge sits at the first occurrence of its pair in stem order and takes the last stem's score; the nodes
 * and each node's adjacency keep NetworkX's insertion order.  No pair filter.  Host buffers in and out.
 *   offsets, stem_offsets, stems, scores, pair_offsets, pairs: as sqrn_hungarian_batch (no symbols); pairs (v, w),
 *                v < w, sorted by v;  power: the exponent of the weights (RunAlgo passes 1.7).
 * SQRN_E_BADARG: a stem outside [0, N), with len < 1 or with a pair (v, w), v >= w; a sequence longer than
 * SQRN_MAX_LEN; a negative or NaN score; a score ** power (C pow) that is not finite or above DBL_MAX / 4 (the host
 * builder has complex numbers or overflows there).
 * Sequences of up to 256 positions run a warp each, longer ones a CTA each with the node state (~124 bytes a node) in
 * shared memory up to 1 933 positions on a B200 (the opt-in limit), in a device workspace beyond.  Every team keeps
 * 16 bytes an edge in the workspace (at most 4 GiB, kept by the context until sqrn_ctx_destroy).  Longest first
 * within each tier; the warp tier runs concurrently with the others.                                                 */
SQRN_API int  sqrn_edmonds_batch(sqrn_ctx *ctx, int64_t n_seqs, const int64_t *offsets, const int64_t *stem_offsets,
                                 const int32_t *stems, const double *scores, double power, int64_t *pair_offsets,
                                 int32_t *pairs);

/* ---- single-path fast lane (poollim == 1: `byseq pl=1`, SQUARNA.py:887-935) --
 * One parameter set, default reactivities, no restraints: one structure per
 * sequence, written as ASCII dot-bracket.  `symbols`/`offsets`/outputs are HOST
 * pointers for sqrn_fast_predict_host and DEVICE pointers for
 * sqrn_fast_predict_device (inputs already resident in HBM; asynchronous on the
 * context's stream).  scores: 3 doubles per sequence (total, structscore,
 * reactscore; ScoreStruct, SQRNdbnseq.py:899), rounded as round(x,3) by the host
 * variant and unrounded by the device variant.  The host variant pipelines the
 * batch in chunks: host->device copy, kernel and device->host copy overlap; a
 * chunk that mixes sequences of <= 320 symbols with longer ones is dealt to two
 * launches (warp teams / CTA teams), so any mix of lengths may be passed in any
 * order.  The device variants run ONE kernel chosen from max_len: group
 * resident batches by length class (<= 128, 224, 320, longer).                 */
SQRN_API int  sqrn_fast_predict_host(sqrn_ctx *ctx, const sqrn_paramset *ps,
                            int64_t n_seqs, const int64_t *offsets, const uint8_t *symbols,
                            uint8_t *dbn_ascii, double *scores, int32_t *n_stems);
SQRN_API int  sqrn_fast_predict_device(sqrn_ctx *ctx, const sqrn_paramset *ps,
                              int64_t n_seqs, int64_t total_len, int32_t max_len,
                              const int64_t *d_offsets, const uint8_t *d_symbols,
                              uint8_t *d_dbn_ascii, double *d_scores, int32_t *d_n_stems);

/* The same lane over the PACKED boundary format (2-bit base codes in, 4-bit bracket codes out): 0.11 GB instead of
 * 0.30 GB over PCIe per million 130-nt sequences.  Plain A/C/G/U(T) sequences only (sqrn_pack_symbols reports anything
 * else; such batches use the byte lane).
 *   offsets  [n_seqs+1] uint32, in bases (the batch holds < 2^32 bases);
 *   packed   base k of the batch = bits 2 (k & 3) .. of byte k >> 2; A C G U = 0 1 2 3;
 *   dbn_nib  [total/2 + n_seqs + 1] bytes: sequence b starts at byte (offsets[b] >> 1) + b, two positions per byte
 *            (low nibble first): 0 '.', L = opening, 8 | L = closing bracket of level L (1..7);
 *   score_milli [2 n_seqs]: round(total, 3) and round(structscore, 3) (ScoreStruct, SQRNdbnseq.py:899) in thousandths;
 *            the reactscore of a plain sequence is 0.5;
 *   n_stems  [n_seqs] uint16 or NULL;  flags [n_seqs] or NULL: bit 0 = structscore is the int 0, bit 1 = MORE THAN 7
 *            pseudoknot levels -- that sequence's dbn_nib is not valid, redo it through the byte lane.
 * sqrn_pack_symbols / sqrn_unpack_dbn are the host-side converters (threaded); *n_other = symbols outside ACGUT.     */
SQRN_API int  sqrn_fast_predict_packed_host(sqrn_ctx *ctx, const sqrn_paramset *ps,
                            int64_t n_seqs, const uint32_t *offsets, const uint8_t *packed,
                            uint8_t *dbn_nib, int32_t *score_milli, uint16_t *n_stems, uint8_t *flags);
/* ... and with everything resident in HBM (asynchronous on the context's stream; d_offsets int64 as in
 * sqrn_fast_predict_device).  d_flags bit 3: the score sat next to a rounding tie and its thousandths are NOT set
 * (the host variant redoes those with CPython's round()).                                                            */
SQRN_API int  sqrn_fast_predict_packed_device(sqrn_ctx *ctx, const sqrn_paramset *ps,
                            int64_t n_seqs, int64_t total_len, int32_t max_len,
                            const int64_t *d_offsets, const uint8_t *d_packed,
                            uint8_t *d_dbn_nib, int32_t *d_score_milli, uint16_t *d_n_stems, uint8_t *d_flags);
SQRN_API int  sqrn_pack_symbols(int64_t n_total, const uint8_t *symbols, uint8_t *packed, int64_t *n_other);
SQRN_API int  sqrn_unpack_dbn(int64_t n_seqs, const uint32_t *offsets, const uint8_t *dbn_nib, uint8_t *dbn_ascii);
/* Level codes of sqrn_result::dbn / cons (+L opening, -L closing bracket of level L, 0 unpaired) -> the glyphs of
 * PairsToDBN (SQRNdbnseq.py:142-143), threaded.  Levels 31..49 (Cyrillic brackets) come out as byte 0: the caller
 * prints those structures itself; levels beyond the alphabet are '.', as in the reference.                            */
SQRN_API int  sqrn_codes_to_ascii(int64_t n, const int8_t *codes, uint8_t *ascii);
/* DBNToPairs (SQRNdbnseq.py:172-207) on one dot-bracket line given as n code points: one stack per bracket kind, closing
 * brackets without a partner ignored, pairs sorted by (i, j).  open_cp / close_cp: the n_kinds bracket glyphs (the
 * alphabet of PairsToDBN, passed by the Python mirror); pairs [2 * (n / 2)] int32; host only.                         */
SQRN_API int  sqrn_dbn_pairs(int64_t n, const uint32_t *text, int32_t n_kinds, const uint32_t *open_cp, const uint32_t *close_cp,
                             int32_t *pairs, int64_t *n_pairs);
/* Per-sequence flags of the last sqrn_fast_predict_host call (bit 1: more than 30 pseudoknot levels, the ASCII
 * glyphs ran out).  When that call returns SQRN_E_UNSUPPORTED for this reason every OTHER sequence's result is valid:
 * the flagged ones go through sqrn_predict_batch, whose level codes have no such limit.                              */
SQRN_API int  sqrn_fast_last_flags(const sqrn_ctx *ctx, int64_t n_seqs, uint8_t *flags);

/* TEST SEAM (tests/ only): one launch of the work kernel in a given mode
 * (0 run to completion, 1 one OptimalStems + ChooseStems, 2 AnnotateStems,
 * 3 ScoreStruct + dbn) on top of caller-supplied pre-selected stems.            */
SQRN_API int  sqrn_debug_run(sqrn_ctx *ctx, const sqrn_paramset *ps, const sqrn_batch *in, int mode, int n_items,
                    const int32_t *item_seq, const int64_t *init_off, const int32_t *init_stems,
                    const double *item_subopt, const int64_t *out_cap, int32_t *out_stems, int32_t *out_n,
                    double *out_fin, double *out_raw, uint8_t *out_flags, int8_t *dbn_code, int min_ccap);

/* counters of the last call: kernels launched, device milliseconds of the main kernel */
/* Bulk text lane of the CLI's single-sequence mode (host only): what SQUARNA.py:80-256 (input) and
 * SQRNdbnseq.py:1301-1406 (the printed block) do, for the plain shape of an input -- name line + sequence,
 * nothing else -- on whole buffers.  SQRN_E_UNSUPPORTED: the text has another shape (default lines, per-entry
 * reactivities / restraints / reference, non-ASCII, ...): use the per-entry path.  multiline: plain FASTA.
 * sqrn_text_parse writes the counts always and fills the arrays when the capacities suffice (else
 * SQRN_E_CAPACITY).  sqrn_text_format writes the blocks of entries [first, first + count); *written = bytes
 * needed / written. */
SQRN_API int  sqrn_text_parse(const char *text, int64_t len, int multiline, int64_t *n_entries, int64_t *total_seq,
                        int64_t cap_entries, int64_t cap_seq, int64_t *name_begin, int32_t *name_len,
                        int64_t *seq_offsets, uint8_t *seq);
SQRN_API int  sqrn_text_ungap(int64_t n, const int64_t *seq_offsets, const uint8_t *seq,      /* UnAlign, seq.py:236-255 */
                        int64_t *sym_offsets, uint8_t *sym);
SQRN_API int  sqrn_text_format(int64_t first, int64_t count, const char *text, const int64_t *name_begin,
                        const int32_t *name_len, const int64_t *seq_offsets, const uint8_t *seq,
                        const int64_t *sym_offsets, const uint8_t *dbn, const double *scores, int conslim,
                        const char *psname, char *out, int64_t cap, int64_t *written);

SQRN_API int  sqrn_ctx_last_stats(const sqrn_ctx *ctx, int64_t *n_launches, double *kernel_ms,
                         int64_t *n_optimal_calls);

#ifdef __cplusplus
}
#endif
#endif /* SQRN_H */
