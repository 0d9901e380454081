"""Loader and thin object wrapper for libsqrn_b200.so (include/sqrn.h).

There is no CPU fallback: if the shared object has not been built, or no CUDA
device is usable, every entry point raises.
"""
import ctypes as C
import os

import numpy as np

from ._abi import (Batch, ParamSet, Result, Stems, E_CAPACITY, OK, pack_sequences, paramset_array, ptr)

E_UNSUPPORTED = -4

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("SQRN_LIB_PATH") or os.path.join(_HERE, "libsqrn_b200.so")      # (override: kernel experiments)

MODE_TAIL, MODE_STEP, MODE_YIELD, MODE_FINAL = 0, 1, 2, 3

EXPORTS = ["sqrn_abi_version", "sqrn_device_count", "sqrn_ctx_create", "sqrn_ctx_destroy",
           "sqrn_last_error", "sqrn_ctx_set_stream", "sqrn_predict_batch", "sqrn_yield_stems_batch",
           "sqrn_fast_predict_host", "sqrn_fast_predict_device", "sqrn_ctx_last_stats", "sqrn_debug_run",
           "sqrn_ctx_set_tuning", "sqrn_text_parse", "sqrn_text_ungap", "sqrn_text_format",
           "sqrn_fast_predict_packed_host", "sqrn_pack_symbols", "sqrn_unpack_dbn", "sqrn_fast_last_flags",
           "sqrn_stem_matrix_batch", "sqrn_fast_predict_packed_device", "sqrn_codes_to_ascii", "sqrn_dbn_pairs",
           "sqrn_nussinov_batch", "sqrn_hungarian_batch", "sqrn_edmonds_batch"]

_lib = None


class SqrnError(RuntimeError):
    """a library call failed; `code` is its SQRN_E_* return code"""

    def __init__(self, msg, code=None):
        super().__init__(msg)
        self.code = code


def load():
    """dlopen libsqrn_b200.so and declare the prototypes of include/sqrn.h."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise SqrnError("libsqrn_b200.so is not built (run `python -c 'import __graft_entry__ as g; g.build()'` "
                        "or `make -C squarna_b200/csrc`); squarna_b200 has no CPU fallback")
    L = C.CDLL(LIB_PATH)
    vp, i32, i64 = C.c_void_p, C.c_int32, C.c_int64
    L.sqrn_abi_version.restype = C.c_int
    L.sqrn_device_count.restype = C.c_int
    L.sqrn_ctx_create.argtypes = [C.c_int, C.POINTER(vp)]
    L.sqrn_ctx_destroy.argtypes = [vp]
    L.sqrn_ctx_destroy.restype = None
    L.sqrn_last_error.argtypes = [vp]
    L.sqrn_last_error.restype = C.c_char_p
    L.sqrn_ctx_set_stream.argtypes = [vp, vp]
    L.sqrn_ctx_set_tuning.argtypes = [vp, C.c_int, C.c_int]
    L.sqrn_predict_batch.argtypes = [vp, C.POINTER(ParamSet), C.c_int, C.POINTER(Batch), C.POINTER(Result)]
    L.sqrn_yield_stems_batch.argtypes = [vp, C.POINTER(ParamSet), C.POINTER(Batch), C.POINTER(Stems)]
    L.sqrn_fast_predict_host.argtypes = [vp, C.POINTER(ParamSet), i64, vp, vp, vp, vp, vp]
    L.sqrn_fast_predict_device.argtypes = [vp, C.POINTER(ParamSet), i64, i64, i32, vp, vp, vp, vp, vp]
    L.sqrn_fast_predict_packed_host.argtypes = [vp, C.POINTER(ParamSet), i64, vp, vp, vp, vp, vp, vp]
    L.sqrn_fast_predict_packed_device.argtypes = [vp, C.POINTER(ParamSet), i64, i64, i32, vp, vp, vp, vp, vp, vp]
    L.sqrn_pack_symbols.argtypes = [i64, vp, vp, C.POINTER(i64)]
    L.sqrn_unpack_dbn.argtypes = [i64, vp, vp, vp]
    L.sqrn_codes_to_ascii.argtypes = [i64, vp, vp]
    L.sqrn_dbn_pairs.argtypes = [i64, vp, C.c_int32, vp, vp, vp, C.POINTER(C.c_int64)]
    L.sqrn_fast_last_flags.argtypes = [vp, i64, vp]
    L.sqrn_stem_matrix_batch.argtypes = [vp, C.POINTER(ParamSet), C.POINTER(Batch), vp, C.c_double, i64, C.POINTER(i64), vp]
    L.sqrn_nussinov_batch.argtypes = [vp, i64, vp, vp, vp, vp, vp, i32, vp, vp]
    L.sqrn_hungarian_batch.argtypes = [vp, i64, vp, vp, vp, vp, vp, i32, C.c_double, vp, vp]
    L.sqrn_edmonds_batch.argtypes = [vp, i64, vp, vp, vp, vp, C.c_double, vp, vp]
    L.sqrn_ctx_last_stats.argtypes = [vp, C.POINTER(i64), C.POINTER(C.c_double), C.POINTER(i64)]
    L.sqrn_debug_run.argtypes = [vp, C.POINTER(ParamSet), C.POINTER(Batch), C.c_int, C.c_int] + [vp] * 11 + [C.c_int]
    L.sqrn_text_parse.argtypes = [vp, i64, C.c_int, C.POINTER(i64), C.POINTER(i64), i64, i64, vp, vp, vp, vp]
    L.sqrn_text_ungap.argtypes = [i64, vp, vp, vp, vp]
    L.sqrn_text_format.argtypes = [i64, i64, vp, vp, vp, vp, vp, vp, vp, vp, C.c_int, C.c_char_p, vp, i64, C.POINTER(i64)]
    _lib = L
    return L


# ---- bulk text lane (host only; include/sqrn.h) -----------------------------
class ParsedText:
    """what sqrn_text_parse found: the text itself, name spans, and the sequence tokens as a CSR"""
    __slots__ = ("text", "n", "name_begin", "name_len", "seq_offsets", "seq")


def text_parse(text, multiline):
    """text: bytes of an input file.  Returns ParsedText, or None when the text is not of the plain shape
    (the caller then takes the per-entry path)."""
    L = load()
    n, tot = C.c_int64(0), C.c_int64(0)
    # entry capacity: a guess (counting the '>' of a 140 MB file in Python took longer than parsing it); the library
    # counts first and reports SQRN_E_CAPACITY with the exact number when the guess was too small
    cap_e, cap_s = len(text) // 24 + 16, len(text) + 1
    seq = np.empty(cap_s, np.uint8)
    while True:
        name_begin = np.empty(cap_e, np.int64)
        name_len = np.empty(cap_e, np.int32)
        seq_off = np.empty(cap_e + 1, np.int64)
        rc = L.sqrn_text_parse(text, len(text), int(bool(multiline)), C.byref(n), C.byref(tot), cap_e, cap_s,
                               ptr(name_begin), ptr(name_len), ptr(seq_off), ptr(seq))
        if rc == E_CAPACITY and n.value > cap_e and tot.value <= cap_s:
            cap_e = n.value
            continue
        break
    if rc != OK:
        return None
    out = ParsedText()
    out.text, out.n = text, n.value
    out.name_begin, out.name_len = name_begin[:n.value], name_len[:n.value]
    out.seq_offsets, out.seq = seq_off[:n.value + 1], seq[:tot.value]
    return out


def text_ungap(parsed):
    """(symbols without gap characters, their CSR offsets) of a ParsedText: UnAlign on the whole buffer"""
    L = load()
    sym = np.empty(max(len(parsed.seq), 1), np.uint8)
    off = np.empty(parsed.n + 1, np.int64)
    rc = L.sqrn_text_ungap(parsed.n, ptr(parsed.seq_offsets), ptr(parsed.seq), ptr(off), ptr(sym))
    if rc != OK:
        raise SqrnError("sqrn_text_ungap failed (%d)" % rc)
    return sym[:int(off[-1])], off


def text_format(parsed, first, count, sym_offsets, dbn, scores, conslim, psname, scratch=None):
    """the RunSQRNdbnseq text blocks of entries [first, first + count) as bytes; with `scratch` (a list holding a
    reusable uint8 array, or empty) a view into that array is returned instead (no copy, no fresh pages per call)"""
    L = load()
    need = C.c_int64(0)
    scores = np.ascontiguousarray(scores, dtype=np.float64)
    args = (first, count, parsed.text, ptr(parsed.name_begin), ptr(parsed.name_len), ptr(parsed.seq_offsets),
            ptr(parsed.seq), ptr(sym_offsets), ptr(dbn), ptr(scores), int(conslim), psname.encode("ascii"))
    # an upper bound of the text size (three numbers of at most 24 characters per entry), so that one call does it
    bound = int(parsed.name_len[first:first + count].sum()) + \
        5 * int(parsed.seq_offsets[first + count] - parsed.seq_offsets[first]) + count * (len(psname) + 128)
    if scratch is not None and scratch and len(scratch[0]) >= bound:
        buf = scratch[0]
    else:
        buf = np.empty(max(bound, 1), np.uint8)
        if scratch is not None:
            scratch[:] = [buf]
    rc = L.sqrn_text_format(*args, ptr(buf), len(buf), C.byref(need))
    if rc == E_CAPACITY:
        buf = np.empty(max(need.value, 1), np.uint8)
        if scratch is not None:
            scratch[:] = [buf]
        rc = L.sqrn_text_format(*args, ptr(buf), len(buf), C.byref(need))
    if rc != OK:
        raise SqrnError("sqrn_text_format failed (%d)" % rc)
    return buf[:need.value] if scratch is not None else buf[:need.value].tobytes()


def pack_symbols(symbols):
    """ASCII symbols (uint8 array) -> (2-bit packed uint8 array, number of symbols outside ACGUT); host only"""
    L = load()
    symbols = np.ascontiguousarray(symbols, dtype=np.uint8)
    packed = np.empty((len(symbols) + 3) // 4 + 1, np.uint8)
    bad = C.c_int64(0)
    rc = L.sqrn_pack_symbols(len(symbols), ptr(symbols), ptr(packed), C.byref(bad))
    if rc != OK:
        raise SqrnError("sqrn_pack_symbols failed (%d)" % rc)
    return packed, bad.value


def dbn_pairs(text, open_glyphs, close_glyphs):
    """DBNToPairs (include/sqrn.h: sqrn_dbn_pairs) of one dot-bracket line -> tuple of (i, j), sorted; host only"""
    L = load()
    cp = np.frombuffer(text.encode("utf-32-le", "surrogatepass"), dtype=np.uint32)
    pairs = np.empty(max(len(cp) // 2, 1) * 2, np.int32)
    m = C.c_int64(0)
    rc = L.sqrn_dbn_pairs(len(cp), ptr(cp), len(open_glyphs), ptr(open_glyphs), ptr(close_glyphs), ptr(pairs), C.byref(m))
    if rc != OK:
        raise SqrnError("sqrn_dbn_pairs failed (%d)" % rc)
    flat = pairs[:2 * m.value].tolist()
    return tuple(zip(flat[0::2], flat[1::2]))


def codes_to_ascii(codes):
    """int8 level codes (+L opening, -L closing bracket) -> glyph bytes (uint8, same shape); levels 31..49 -- the
    Cyrillic brackets -- come out as 0 (include/sqrn.h); host only, threaded"""
    L = load()
    codes = np.ascontiguousarray(codes, dtype=np.int8)
    out = np.empty(codes.shape, np.uint8)
    rc = L.sqrn_codes_to_ascii(codes.size, ptr(codes), ptr(out))
    if rc != OK:
        raise SqrnError("sqrn_codes_to_ascii failed (%d)" % rc)
    return out


def unpack_dbn(offsets32, dbn_nib):
    """4-bit bracket codes of the packed lane -> ASCII dot-bracket bytes (uint8 [total]); host only"""
    L = load()
    n = len(offsets32) - 1
    out = np.empty(max(int(offsets32[-1]), 1), np.uint8)
    rc = L.sqrn_unpack_dbn(n, ptr(offsets32), ptr(dbn_nib), ptr(out))
    if rc != OK:
        raise SqrnError("sqrn_unpack_dbn failed (%d)" % rc)
    return out[:int(offsets32[-1])]


class PackedBatch:
    """numpy arrays behind a sqrn_batch (kept alive as long as the object lives)."""

    def __init__(self, seqs, react_codes=None, react_values=None, react_comp=False, restr_class=None,
                 rbps=None, smat=None, cols=None, interchainonly=False, hardrest=False, rankbydiff=False,
                 poollim=1000, conslim=1, max_structs=0, rankby=(0, 2, 1), priority_mask=0,
                 bpp_terms=None, bpp_mode=0, ali_len=0, flat=False):
        """flat=True: the batch is already in CSR form -- seqs = (symbols uint8, offsets int64) and react_codes / restr_class /
        cols are single arrays over all positions, rbps = (rbp_offsets int64, pairs int32 (k, 2))"""
        self.seqs = seqs
        if flat:
            self.symbols, self.offsets = np.ascontiguousarray(seqs[0], np.uint8), np.ascontiguousarray(seqs[1], np.int64)
            if self.symbols.size == 0:
                self.symbols = np.zeros(1, np.uint8)
            n = len(self.offsets) - 1
        else:
            self.symbols, self.offsets = pack_sequences(seqs)
            n = len(seqs)

        def cat(lst, dt):
            if lst is None:
                return None
            if flat:
                a = np.ascontiguousarray(lst, dtype=dt).ravel()
                return a if a.size else np.zeros(1, dt)
            arrs = [np.asarray(x, dtype=dt).ravel() for x in lst]
            tot = sum(a.size for a in arrs)
            return np.concatenate(arrs) if tot else np.zeros(1, dt)

        self.react_code = cat(react_codes, np.uint16)
        self.react_values = None if react_values is None else np.ascontiguousarray(react_values, np.float64)
        self.restr_class = cat(restr_class, np.uint8)
        self.rbp_offsets = self.rbps = None
        if rbps is not None and flat:
            self.rbp_offsets = np.ascontiguousarray(rbps[0], np.int64)
            self.rbps = cat(rbps[1], np.int32)
        elif rbps is not None:
            self.rbp_offsets = np.zeros(n + 1, dtype=np.int64)
            np.cumsum([len(x) for x in rbps], out=self.rbp_offsets[1:])
            self.rbps = cat(rbps, np.int32)
        self.smat = None if smat is None else np.ascontiguousarray(smat, np.float64)
        self.cols = cat(cols, np.int32)
        self.ali_len = int(ali_len)
        b = Batch()
        b.n_seqs = n
        b.offsets = ptr(self.offsets)
        b.symbols = ptr(self.symbols)
        b.react_code = ptr(self.react_code)
        b.react_values = ptr(self.react_values)
        b.n_react_values = 0 if self.react_values is None else len(self.react_values)
        b.react_sum_compensated = int(bool(react_comp))
        b.restr_class = ptr(self.restr_class)
        b.rbp_offsets = ptr(self.rbp_offsets)
        b.rbps = ptr(self.rbps)
        b.smat = ptr(self.smat)
        b.smat_L = self.ali_len if self.smat is None else self.smat.shape[0]      # (without smat: the alignment length, for stem_matrix)
        b.cols = ptr(self.cols)
        b.interchainonly = int(bool(interchainonly))
        b.hardrest = int(bool(hardrest))
        b.rankbydiff = int(bool(rankbydiff))
        b.poollim = int(poollim)
        b.conslim = int(conslim)
        b.max_structs = int(max_structs)
        for k in range(3):
            b.rankby[k] = int(rankby[k])
        b.priority_mask = int(priority_mask)
        # base-pair-probability terms: one N x N float64 matrix per sequence (include/sqrn.h)
        self.bpp_term = self.bpp_offsets = None
        if bpp_terms is not None and bpp_mode:
            self.bpp_offsets = np.zeros(n + 1, dtype=np.int64)
            np.cumsum([int(t.size) for t in bpp_terms], out=self.bpp_offsets[1:])
            self.bpp_term = cat([np.ascontiguousarray(t, dtype=np.float64) for t in bpp_terms], np.float64)
            b.bpp_term = ptr(self.bpp_term)
            b.bpp_offsets = ptr(self.bpp_offsets)
            b.bpp_mode = int(bpp_mode)
        self.c = b


class FlatResult:
    """What one sqrn_predict_batch call returned (include/sqrn.h, sqrn_result), as the flat arrays it filled.
    Sequence b of the batch has N = offsets[b+1] - offsets[b] positions and the structures so[b] .. so[b+1]-1 in rank
    order; structure k has scores[k] = (total, structscore, reactscore), isint[k] (structscore is the int 0),
    mask[k] (bit q: parameter set q predicted it), stems[sto[k]:sto[k+1]] and N level codes at dbn[dbo[k]:].
    The offset / score columns are Python lists (one tolist() per array)."""

    def __init__(self, offsets, so, scores, isint, mask, ntot, sto, stems, dbo, dbn, cons):
        self.n = len(offsets) - 1
        self.off = np.asarray(offsets).tolist()
        self.so, self.sto, self.dbo = so.tolist(), sto.tolist(), dbo.tolist()
        nk = self.so[-1] if self.n else 0
        self.scores, self.isint, self.mask = scores[:nk].tolist(), isint[:nk].tolist(), mask[:nk].tolist()
        self.ntot = ntot.tolist()
        self.stems, self.dbn, self.cons = stems, dbn, cons
        self._glyphs = None

    def cons_codes(self, b):
        return self.cons[self.off[b]:self.off[b + 1]]

    def codes2d(self, b):
        """level codes of every structure of sequence b as one (n_structs, N) int8 array (a view when the rows lie
        back to back, which is how the library writes them)"""
        N = self.off[b + 1] - self.off[b]
        k0, k1 = self.so[b], self.so[b + 1]
        if k1 == k0:
            return np.zeros((0, N), np.int8)
        d0 = self.dbo[k0]
        if self.dbo[k1 - 1] - d0 == (k1 - k0 - 1) * N:
            return self.dbn[d0:d0 + (k1 - k0) * N].reshape(k1 - k0, N)
        return np.stack([self.dbn[self.dbo[k]:self.dbo[k] + N] for k in range(k0, k1)])

    def text(self, b):
        """the glyphs of every structure of sequence b, row after row in one str (n_structs * N characters), or None
        when its rows do not lie back to back.  Byte 0 in it: a bracket beyond the ASCII part of the alphabet."""
        N = self.off[b + 1] - self.off[b]
        k0, k1 = self.so[b], self.so[b + 1]
        if k1 == k0:
            return ""
        d0 = self.dbo[k0]
        if self.dbo[k1 - 1] - d0 != (k1 - k0 - 1) * N:
            return None
        if self._glyphs is None:                  # the whole call's codes in one threaded pass
            used = 0
            for q in range(self.n):
                if self.so[q + 1] > self.so[q]:
                    used = max(used, self.dbo[self.so[q + 1] - 1] + self.off[q + 1] - self.off[q])
            self._glyphs = codes_to_ascii(self.dbn[:used])
        return str(memoryview(self._glyphs[d0:d0 + (k1 - k0) * N]), "latin-1")

    def sequence(self, b):
        """(cons_codes, [(codes, (total, struct, react), struct_is_int0, psmask, stems (k,3))], n_total, codes2d)"""
        k0, k1 = self.so[b], self.so[b + 1]
        c2 = self.codes2d(b) if k1 > k0 else None
        sto, stems = self.sto, self.stems
        structs = [(c2[k - k0], tuple(self.scores[k]), bool(self.isint[k]), self.mask[k], stems[sto[k]:sto[k + 1]])
                   for k in range(k0, k1)]
        return (self.cons_codes(b), structs, self.ntot[b], c2)

    def per_sequence(self):
        return [self.sequence(b) for b in range(self.n)]

    @classmethod
    def from_sequences(cls, seqs):
        """the flat form of a per-sequence result list (what `per_sequence` returns; the 4th element may be missing)"""
        n = len(seqs)
        off = np.zeros(n + 1, np.int64)
        np.cumsum([len(q[0]) for q in seqs], out=off[1:])
        so = np.zeros(n + 1, np.int64)
        np.cumsum([len(q[1]) for q in seqs], out=so[1:])
        nk = int(so[-1])
        scores, isint, mask = np.zeros((max(nk, 1), 3)), np.zeros(max(nk, 1), np.uint8), np.zeros(max(nk, 1), np.uint64)
        sto, dbo = np.zeros(nk + 1, np.int64), np.zeros(max(nk, 1), np.int64)
        stems, dbn = [], []
        cons = np.concatenate([np.asarray(q[0], np.int8) for q in seqs]) if n else np.zeros(0, np.int8)
        k = at = 0
        for q in seqs:
            for codes, sc, ii, m, st in q[1]:
                scores[k], isint[k], mask[k] = sc, int(bool(ii)), m
                dbo[k] = at
                dbn.append(np.asarray(codes, np.int8))
                at += len(dbn[-1])
                st = np.asarray(st, np.int32).reshape(-1, 3)
                stems.append(st)
                sto[k + 1] = sto[k] + len(st)
                k += 1
        ntot = np.array([q[2] for q in seqs] if n else [0], np.int32)
        return cls(off, so, scores, isint, mask, ntot, sto,
                   np.concatenate(stems) if stems else np.zeros((0, 3), np.int32), dbo,
                   np.concatenate(dbn) if dbn else np.zeros(0, np.int8), cons)


class Context:
    """One GPU, one host thread at a time."""

    def __init__(self, device=0):
        self.L = load()
        h = C.c_void_p()
        rc = self.L.sqrn_ctx_create(int(device), C.byref(h))
        if rc != OK:
            raise SqrnError("sqrn_ctx_create failed (%d): %s" % (rc, self.L.sqrn_last_error(None).decode()))
        self.h = h
        self.device = device

    def close(self):
        if getattr(self, "h", None):
            self.L.sqrn_ctx_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc):
        if rc != OK:
            raise SqrnError("libsqrn_b200 error %d: %s" % (rc, self.L.sqrn_last_error(self.h).decode()), rc)

    def set_stream(self, cuda_stream):
        self._check(self.L.sqrn_ctx_set_stream(self.h, C.c_void_p(cuda_stream)))

    def set_region_mode(self, mode):
        """0 automatic, 1 position scan, 2 stem walk (identical results; see include/sqrn.h)"""
        self._check(self.L.sqrn_ctx_set_tuning(self.h, 1, int(mode)))

    def set_no_fast_kernel(self, flag):
        """route sqrn_fast_predict_* through the general kernel (tests compare both)"""
        self._check(self.L.sqrn_ctx_set_tuning(self.h, 2, int(bool(flag))))

    def set_cluster(self, mode):
        """long sequences: 0 automatic, 1 one CTA per sequence, 2/4/8/16 a cluster of that many CTAs per sequence"""
        self._check(self.L.sqrn_ctx_set_tuning(self.h, 3, int(mode)))

    def set_no_glist(self, flag):
        """CTA teams rescan every greedy step instead of keeping the global persistent list (tests compare both)"""
        self._check(self.L.sqrn_ctx_set_tuning(self.h, 4, int(bool(flag))))

    def stats(self):
        nl, ms, nc = C.c_int64(0), C.c_double(0), C.c_int64(0)
        self.L.sqrn_ctx_last_stats(self.h, C.byref(nl), C.byref(ms), C.byref(nc))
        return dict(launches=nl.value, kernel_ms=ms.value, optimal_calls=nc.value)

    # ---- fast lane -----------------------------------------------------
    def fast_predict(self, paramset, symbols, offsets):
        """host numpy in -> (dbn ascii uint8 [total], scores (n,3) rounded, n_stems (n,))"""
        n = len(offsets) - 1
        ps = paramset if isinstance(paramset, ParamSet) else ParamSet.from_dict(paramset)
        dbn = np.empty(max(int(offsets[-1]), 1), dtype=np.uint8)
        scores = np.empty((max(n, 1), 3), dtype=np.float64)
        nst = np.empty(max(n, 1), dtype=np.int32)
        rc = self.L.sqrn_fast_predict_host(self.h, C.byref(ps), n, ptr(offsets), ptr(symbols),
                                           ptr(dbn), ptr(scores), ptr(nst))
        if rc == E_UNSUPPORTED and n:
            # more than 30 pseudoknot levels somewhere: every other sequence is complete (include/sqrn.h); the
            # flagged ones are marked n_stems = -1 and left to the caller (predict_batch has no such limit)
            flags = self.fast_last_flags(n)
            deep = (flags & 2) != 0
            if deep.any():
                nst[:n][deep] = -1
                rc = OK
        self._check(rc)
        return dbn[:int(offsets[-1])], scores[:n], nst[:n]

    def fast_last_flags(self, n):
        """per-sequence flags of the last fast_predict call (bit 1: pseudoknot levels beyond the output format)"""
        fl = np.zeros(max(n, 1), np.uint8)
        self._check(self.L.sqrn_fast_last_flags(self.h, n, ptr(fl)))
        return fl[:n]

    def fast_predict_packed(self, paramset, packed, offsets32, dbn_nib=None, milli=None, nst=None, flags=None):
        """the fast lane over the packed boundary format (include/sqrn.h): 2-bit base codes + uint32 offsets in ->
        (4-bit bracket codes, scores in thousandths (n,2) int32, n_stems uint16, flags uint8).  Output arrays may be
        passed in (pinned memory of the caller)."""
        n = len(offsets32) - 1
        total = int(offsets32[-1])
        ps = paramset if isinstance(paramset, ParamSet) else ParamSet.from_dict(paramset)
        if dbn_nib is None:
            dbn_nib = np.empty(total // 2 + n + 1, np.uint8)
        if milli is None:
            milli = np.empty((max(n, 1), 2), np.int32)
        if nst is None:
            nst = np.empty(max(n, 1), np.uint16)
        if flags is None:
            flags = np.empty(max(n, 1), np.uint8)
        self._check(self.L.sqrn_fast_predict_packed_host(self.h, C.byref(ps), n, ptr(offsets32), ptr(packed),
                                                         ptr(dbn_nib), ptr(milli), ptr(nst), ptr(flags)))
        return dbn_nib, milli[:n], nst[:n], flags[:n]

    def fast_predict_device(self, paramset, n, total, max_len, d_off, d_sym, d_dbn, d_scores, d_nst):
        """device pointers (ints) in/out, asynchronous on the context's stream"""
        ps = paramset if isinstance(paramset, ParamSet) else ParamSet.from_dict(paramset)
        self._check(self.L.sqrn_fast_predict_device(self.h, C.byref(ps), n, total, max_len,
                                                    C.c_void_p(d_off), C.c_void_p(d_sym), C.c_void_p(d_dbn),
                                                    C.c_void_p(d_scores), C.c_void_p(d_nst)))

    # ---- general path ---------------------------------------------------
    def predict_batch(self, paramsets, batch):
        """paramsets: list of dicts; batch: PackedBatch.  Returns per sequence a tuple
        (cons_codes int8[N], [ (dbn_codes, (total, struct, react), struct_is_int0, psmask, stems (k,3)) ], n_total,
        codes of all its structures as one (n_structs, N) array)"""
        return self.predict_batch_flat(paramsets, batch).per_sequence()

    def predict_batch_flat(self, paramsets, batch):
        """the same call, the result left in the flat arrays the C ABI filled (FlatResult): callers that format many
        structures per sequence (predict_many with pl=100: ~40) read them without one Python object per structure"""
        arr = paramsets if not isinstance(paramsets, (list, tuple)) else paramset_array(list(paramsets))
        nps = len(paramsets)
        n = len(batch.offsets) - 1
        total = int(batch.offsets[-1])
        cap_s, cap_st, cap_d = max(8 * n, 8), max(16 * n, 64), max(4 * total, 64)
        first = True
        while True:
            so = np.zeros(n + 1, np.int64)
            scores = np.zeros((cap_s, 3))
            isint = np.zeros(cap_s, np.uint8)
            mask = np.zeros(cap_s, np.uint64)
            ntot = np.zeros(max(n, 1), np.int32)
            sto = np.zeros(cap_s + 1, np.int64)
            stems = np.zeros((cap_st, 3), np.int32)
            dbo = np.zeros(cap_s, np.int64)
            dbn = np.zeros(cap_d, np.int8)
            cons = np.zeros(max(total, 1), np.int8)
            r = Result()
            r.cap_structs, r.cap_stems, r.cap_dbn = cap_s, cap_st, cap_d
            r.struct_offsets, r.scores, r.struct_is_int0, r.psmask = ptr(so), ptr(scores), ptr(isint), ptr(mask)
            r.n_total, r.stem_offsets, r.stems, r.dbn_offsets = ptr(ntot), ptr(sto), ptr(stems), ptr(dbo)
            r.dbn, r.cons = ptr(dbn), ptr(cons)
            rc = self.L.sqrn_predict_batch(self.h, arr, nps, C.byref(batch.c) if first else None, C.byref(r))
            if rc == E_CAPACITY:
                cap_s, cap_st, cap_d = max(r.need_structs, 8), max(r.need_stems, 8), max(r.need_dbn, 8)
                first = False
                continue
            self._check(rc)
            break
        return FlatResult(batch.offsets, so, scores, isint, mask, ntot, sto, stems, dbo, dbn, cons)

    def yield_stems(self, paramset, batch):
        """AnnotateStems per sequence: list of (stems (k,3) int32, scores (k,) float64)"""
        ps = paramset if isinstance(paramset, ParamSet) else ParamSet.from_dict(paramset)
        n = len(batch.offsets) - 1
        cap = max(64 * n, 1024)
        first = True
        while True:
            off = np.zeros(n + 1, np.int64)
            st = np.zeros((cap, 3), np.int32)
            sc = np.zeros(cap)
            s = Stems()
            s.cap_stems, s.stem_offsets, s.stems, s.scores = cap, ptr(off), ptr(st), ptr(sc)
            rc = self.L.sqrn_yield_stems_batch(self.h, C.byref(ps), C.byref(batch.c) if first else None, C.byref(s))
            if rc == E_CAPACITY:
                cap = max(int(s.need_stems), 8)
                first = False
                continue
            self._check(rc)
            break
        return [(st[off[b]:off[b + 1]].copy(), sc[off[b]:off[b + 1]].copy()) for b in range(n)]

    @staticmethod
    def _builder_args(symbols, offsets, stems):
        """(n, offsets, symbols, stem_offsets, stems, scores, pair_offsets, pairs) of a builder call: the inputs flat,
        the outputs sized for N/2 pairs per sequence"""
        offsets = np.ascontiguousarray(offsets, np.int64)
        symbols = np.ascontiguousarray(symbols, np.uint8)
        n = len(offsets) - 1
        so = np.zeros(n + 1, np.int64)
        np.cumsum([len(sc) for _, sc in stems], out=so[1:])
        st = np.concatenate([np.asarray(x, np.int32).reshape(-1, 3) for x, _ in stems] + [np.zeros((1, 3), np.int32)])
        sc = np.concatenate([np.asarray(x, np.float64).ravel() for _, x in stems] + [np.zeros(1)])
        po = np.zeros(n + 1, np.int64)
        pairs = np.zeros((max(int((np.diff(offsets) // 2).sum()), 1), 2), np.int32)
        return n, offsets, symbols, so, st, sc, po, pairs

    def hungarian(self, symbols, offsets, stems, minloop=3, power=1.7):
        """the Hungarian builder (SQRNalgos.Hungarian: SciPy's linear_sum_assignment and the pair filter) on the
        device for a batch (include/sqrn.h: sqrn_hungarian_batch).  Arguments as `nussinov`; power: the exponent of
        the pair weights.  Returns per sequence its base pairs as an (n, 2) int32 array sorted by v.  Raises
        SqrnError with code E_BADARG for input the host builder cannot take either (negative or NaN scores,
        non-finite weights) as well as for malformed input."""
        n, offsets, symbols, so, st, sc, po, pairs = self._builder_args(symbols, offsets, stems)
        self._check(self.L.sqrn_hungarian_batch(self.h, n, ptr(offsets), ptr(symbols), ptr(so), ptr(st), ptr(sc),
                                                int(minloop), float(power), ptr(po), ptr(pairs)))
        return [pairs[po[b]:po[b + 1]] for b in range(n)]

    def edmonds(self, symbols, offsets, stems, power=1.7):
        """the Edmonds builder (SQRNalgos.Edmonds: NetworkX's max_weight_matching on the stem pairs) on the device for
        a batch (include/sqrn.h: sqrn_edmonds_batch).  Arguments as `hungarian` (the symbols only give the shape of
        the batch).  Returns per sequence the matched pairs as an (n, 2) int32 array of (v, w), v < w, sorted by v.
        Raises SqrnError with code E_BADARG for input the host builder cannot take either (negative or NaN scores,
        non-finite or huge weights) as well as for malformed input."""
        n, offsets, symbols, so, st, sc, po, pairs = self._builder_args(symbols, offsets, stems)
        self._check(self.L.sqrn_edmonds_batch(self.h, n, ptr(offsets), ptr(so), ptr(st), ptr(sc), float(power),
                                              ptr(po), ptr(pairs)))
        return [pairs[po[b]:po[b + 1]] for b in range(n)]

    def nussinov(self, symbols, offsets, stems, minloop=3):
        """the Nussinov builder (SQRNalgos.Nussinov + BackTrack) on the device for a batch (include/sqrn.h:
        sqrn_nussinov_batch).  symbols / offsets: the ungapped sequences as in PackedBatch; stems: per sequence
        (stems (k,3) int32, scores (k,) float64), as yield_stems returns them.  Returns per sequence its base pairs as
        an (n, 2) int32 array sorted by (v, w)."""
        n, offsets, symbols, so, st, sc, po, pairs = self._builder_args(symbols, offsets, stems)
        self._check(self.L.sqrn_nussinov_batch(self.h, n, ptr(offsets), ptr(symbols), ptr(so), ptr(st), ptr(sc),
                                               int(minloop), ptr(po), ptr(pairs)))
        return [pairs[po[b]:po[b + 1]] for b in range(n)]

    def stem_matrix(self, paramset, batch, threshold, cap_cells=65536):
        """alignment step 1 on the device (include/sqrn.h): batch carries cols and smat_L = alignment length (no smat).
        Returns (matrix (L, L) float64, flat indices of the cells MatrixToDBNs walks in its order, or None when there are
        too many for the device ranking)."""
        ps = paramset if isinstance(paramset, ParamSet) else ParamSet.from_dict(paramset)
        L_ = int(batch.c.smat_L)
        mat = np.empty((L_, L_), np.float64)
        cells = np.empty(max(cap_cells, 1), np.int32)
        m = C.c_int64(0)
        self._check(self.L.sqrn_stem_matrix_batch(self.h, C.byref(ps), C.byref(batch.c), ptr(mat), float(threshold),
                                                  int(cap_cells), C.byref(m), ptr(cells)))
        return mat, (cells[:m.value].copy() if m.value >= 0 else None)

    def debug_run(self, paramset, batch, mode, item_seq=None, init_stems=None, item_subopt=None,
                  out_cap=None, min_ccap=0, want_dbn=True):
        """test seam: one launch of the work kernel (see sqrn_debug_run in csrc/sqrn_abi.cu)"""
        ps = ParamSet.from_dict(paramset)
        nseq = len(batch.offsets) - 1
        n_items = len(item_seq) if item_seq is not None else nseq
        iseq = np.ascontiguousarray(item_seq if item_seq is not None else np.arange(nseq), dtype=np.int32)
        lens = np.diff(batch.offsets)[iseq]
        ioff = ist = None
        if init_stems is not None:
            ioff = np.zeros(n_items + 1, np.int64)
            np.cumsum([len(x) for x in init_stems], out=ioff[1:])
            flat = [t for x in init_stems for s in x for t in s]
            ist = np.array(flat if flat else [0], dtype=np.int32)
        isub = None if item_subopt is None else np.ascontiguousarray(item_subopt, np.float64)
        if out_cap is None:
            out_cap = (lens // 2 + 1) if mode != MODE_YIELD else (lens * lens // 4 + 8)
        ocap = np.ascontiguousarray(np.broadcast_to(out_cap, (n_items,)), dtype=np.int64)
        ooff = np.zeros(n_items + 1, np.int64)
        np.cumsum(ocap, out=ooff[1:])
        stems = np.zeros((max(int(ooff[-1]), 1), 3), np.int32)
        outn = np.zeros(max(n_items, 1), np.int32)
        fin = np.zeros(max(int(ooff[-1]), 1))
        raw = np.zeros((max(n_items, 1), 3))
        flags = np.zeros(max(n_items, 1), np.uint8)
        doff = np.zeros(n_items + 1, np.int64)
        np.cumsum(lens, out=doff[1:])
        dbn = np.zeros(max(int(doff[-1]), 1), np.int8)
        self._check(self.L.sqrn_debug_run(self.h, C.byref(ps), C.byref(batch.c), mode, n_items, ptr(iseq),
                                          ptr(ioff), ptr(ist), ptr(isub), ptr(ocap), ptr(stems), ptr(outn),
                                          ptr(fin), ptr(raw), ptr(flags), ptr(dbn) if want_dbn else None,
                                          int(min_ccap)))
        return dict(off=ooff, stems=stems, n=outn[:n_items], fin=fin, raw=raw[:n_items], flags=flags[:n_items],
                    dbn_off=doff, dbn_code=dbn)
