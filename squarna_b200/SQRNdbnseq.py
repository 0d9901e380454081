"""Single-sequence prediction: the Python surface of the reference's
SQRNdbnseq.py (same public names, argument order, defaults, return shapes and
printed text), with the greedy hot path running on the GPU through
libsqrn_b200.so.

What stays on the host here is string handling only: normalisation, un/re-
alignment, restraint parsing, reactivity pre-processing, bracket glyphs, metrics
against a known structure and text output.  BPMatrix, AnnotateStems, ScoreStems,
ChooseStems, the structure pool, ScoreStruct and the ranking are behind
``Context.predict_batch`` (csrc/sqrn_abi.cu, csrc/sqrn_device.cuh).

Reference lines cited as seq.py:N are /root/reference/src/SQUARNA/SQRNdbnseq.py.
"""
import math
import os
import sys
import threading

import functools
import re

import numpy as np

from . import _lib
from ._abi import E_BADARG
from ._lib import PackedBatch, SqrnError

GAPS = {'-', '.', '~'}          # seq.py:12
SEPS = {';', '&'}               # seq.py:14

# reactivity letters, seq.py:17-30
ReactDict = {"_": 0.00, "+": 0.50, "#": 1.00, "?": -999}
for _k, _v in zip("0123456789", (0.05, 0.15, 0.25, 0.35, 0.45, 0.55, 0.65, 0.75, 0.85, 0.95)):
    ReactDict[_k] = _v
for _k, _ch in enumerate("abcdefghijklmnopqrstuvwxyz"):
    ReactDict[_ch] = float("%.2f" % (0.04 * _k))

# bracket glyphs per pseudoknot level, seq.py:108-112
_OPEN = "([{<ABCDEFGHIJKLMNOPQRSTUVWXYZ" + "БГДЁЖЙЛПФЦЧШЩЬЫЪЭЮЯ"
_CLOSE = ")]}>abcdefghijklmnopqrstuvwxyz" + "бгдёжйлпфцчшщьыъэюя"
_OPEN_IDX = {c: k for k, c in enumerate(_OPEN)}
_CLOSE_IDX = {c: k for k, c in enumerate(_CLOSE)}
_BRACKET_RE = re.compile("[" + re.escape(_OPEN + _CLOSE) + "]")
_RESTR_RE = re.compile(r"[_+/\\]")

_ctx = {}
_ctx_lock = threading.Lock()


def get_context(device=0):
    """Process-wide GPU context (one per device; one host thread drives a context at a time)."""
    with _ctx_lock:
        if device not in _ctx:
            _ctx[device] = _lib.Context(device)
        return _ctx[device]


def visible_devices():
    """indices of the usable CUDA devices of this process (CUDA_VISIBLE_DEVICES applies)"""
    return list(range(_lib.load().sqrn_device_count()))


def _resolve_devices(devices, device=0):
    """devices=None: every visible GPU (the reference's Pool(threads) over sequences, SQUARNA.py:889, becomes one
    host thread per GPU); an int or a list picks them explicitly"""
    if devices is None:
        env = os.environ.get("SQRN_DEVICES")               # e.g. "0,2": the only knob the unchanged Predict() surface has
        devs = [int(x) for x in env.split(",") if x.strip()] if env else (visible_devices() or [device])
    elif isinstance(devices, int):
        devs = [devices]
    else:
        devs = list(devices)
    return devs or [device]


def run_sharded(fn, items, lengths, devices, exponent=3.0):
    """fn(sub_items, device) -> list, for the items dealt to each device by cost (length ** exponent), one host
    thread per GPU (ctypes releases the GIL during the library calls); results come back in input order.  No
    collective: sequences are independent (SURVEY 8e)."""
    from .sharding import shard_plan
    plan = shard_plan(lengths, len(devices), exponent)
    out = [None] * len(items)
    errors = []

    def work(dev, idx):
        try:
            if len(idx):
                res = fn([items[k] for k in idx.tolist()], dev)
                for k, r in zip(idx.tolist(), res):
                    out[k] = r
        except BaseException as e:                     # surfaced in the caller's thread
            errors.append(e)

    threads = [threading.Thread(target=work, args=(d, idx)) for d, idx in zip(devices, plan)]
    for t in threads:
        t.start()
    for t in threads:
        t.join()
    if errors:
        raise errors[0]
    return out


# ---- base-pair probabilities (bpp != 0 parameter sets, seq.py:341-365) --------------------------------
_RNA = None


def set_rna_module(module):
    """Use `module` in place of ViennaRNA's `RNA` for base-pair probabilities (anything with the same
    fold_compound / sc_add_SHAPE_deigan / pf / bpp / mfe / exp_params_rescale surface); None: import RNA."""
    global _RNA
    _RNA = module


def _rna():
    if _RNA is not None:
        return _RNA
    import RNA                                         # ViennaRNA, as in the reference (seq.py:342)
    return RNA


def BPPMatrix(shortseq, shortreacts, M=1.8, B=-0.6):
    """the base-pair probability matrix BPMatrix asks ViennaRNA for (seq.py:341-365): partition function with the
    SHAPE pseudo-energies when reactivities are given, redone with rescaled Boltzmann factors when every
    probability underflowed.  Returns the N x N float64 array (all zero if both attempts gave nothing)."""
    RNA = _rna()
    default = shortreacts is None or set(shortreacts) == {0.5, }
    fc = RNA.fold_compound(''.join(ch if ch not in SEPS and ord(ch) <= 127 else 'N' for ch in shortseq))
    if not default:
        fc.sc_add_SHAPE_deigan(ProcessReacts(shortreacts, reverse=True, M=M, B=B), m=M, b=B)
    fc.pf()
    bppm = np.array(fc.bpp())[1:, 1:]
    if np.max(bppm) > 0:
        return bppm
    (_ss, mfe) = fc.mfe()
    fc.exp_params_rescale(mfe)
    fc.pf()
    return np.array(fc.bpp())[1:, 1:]


def _bpp_terms(preps, idx, paramset, M, B):
    """None when the parameter set has bpp == 0; else (mode, [N x N term per entry of idx]) with
    term = (bppm / max bppm) ** |bpp|: mode 1 is added to the score matrix (bpp < 0), mode 2 multiplies it
    (bpp > 0) -- seq.py:350-364.  No probabilities at all: the neutral term (the reference leaves the matrix alone)."""
    power = paramset.get("bpp", 0)
    if not power:
        return None
    mode = 1 if power < 0 else 2
    terms = []
    for k in idx:
        p = preps[k]
        if p.bppm is None or p.bppm_key != (M, B):
            p.bppm = BPPMatrix(p.shortseq, p._sr if p._sr is None else list(p._sr), M, B)
            p.bppm_key = (M, B)
        mx = np.max(p.bppm) if p.bppm.size else 0
        if mx > 0:
            terms.append(np.ascontiguousarray((p.bppm / mx) ** abs(power), dtype=np.float64))
        else:
            terms.append(np.zeros_like(p.bppm) if mode == 1 else np.ones_like(p.bppm))
    return mode, terms


# --------------------------------------------------------------------- helpers
def ProcessReacts(reacts, missing_threshold=-10, middle=0.5, reverse=False, M=1.8, B=1.6):
    """Normalise raw reactivities into [0, 1] with the neutral value mapped to
    0.5 (seq.py:32-59).  Values are numpy float64 like the reference's."""
    neutral = np.exp(-B / M) - 1
    if reverse:
        neutral, middle = middle, neutral
    if not reacts:
        return []
    out = []
    for x in reacts:
        if x <= missing_threshold:
            x = neutral
        elif np.isnan(x):
            x = neutral
        else:
            x = min(max(0, x), 1)
        if x <= neutral:
            out.append((middle / neutral) * x)
        else:
            out.append(middle + ((x - neutral) / (1 - neutral)) * (1 - middle))
    return out


def EncodedReactivities(seq, reacts, reactformat):
    """list of floats -> reactivity line (seq.py:82-101)"""
    line = _reactivity_line(tuple(reacts), reactformat)       # (the default line of an alignment is shared by its rows)
    if len(line) == len(seq) and not any(ch in seq for ch in SEPS):
        return line
    return ''.join(seq[k] if seq[k] in SEPS else line[k] for k in range(len(seq)))


@functools.lru_cache(maxsize=256)
def _reactivity_line(reacts, reactformat):
    clipped = [min(max(x, 0), 1) if x == x else 1 for x in reacts]
    if reactformat == 3:
        line = ''.join("_+##"[int(x * 3)] for x in clipped)
    elif reactformat == 10:
        line = ''.join("01234567899"[int(x * 10)] for x in clipped)
    else:
        line = ''.join("abcdefghijklmnopqrstuvwxyz"[int(x * 25 + 0.5)] for x in clipped)
    return line


def DBNToPairs(dbn):
    """dbn string -> sorted list of (i, j); one stack per bracket type, closing
    brackets without a partner are ignored (seq.py:172-207).  (The same line is parsed again and again -- the reference
    structure and the restraint line of an alignment by every row: the pairs of the last few thousand distinct strings are
    kept; callers get their own list.)"""
    return list(_dbn_pairs(dbn))


_OPEN_CP = np.array([ord(c) for c in _OPEN], dtype=np.uint32)
_CLOSE_CP = np.array([ord(c) for c in _CLOSE], dtype=np.uint32)


@functools.lru_cache(maxsize=4096)
def _dbn_pairs(dbn):
    if len(dbn) >= 48:                  # long lines (alignment rows, rRNA restraints): the library's host-side parser
        return _lib.dbn_pairs(dbn, _OPEN_CP, _CLOSE_CP)
    return _dbn_pairs_py(dbn)


def _dbn_pairs_py(dbn):
    stacks = {}
    pairs = set()
    # only bracket characters matter: a regular expression finds them (restraint lines are mostly dots)
    for m in _BRACKET_RE.finditer(dbn):
        ch, pos = m.group(), m.start()
        k = _OPEN_IDX.get(ch)
        if k is not None:
            stacks.setdefault(k, []).append(pos)
            continue
        k = _CLOSE_IDX[ch]
        if stacks.get(k):
            pairs.add((stacks[k].pop(), pos))
    return tuple(sorted(pairs))


def _pair_levels(pairs):
    """levels of PairsToDBN (seq.py:119-139) for an arbitrary pair list.
    Returns (unique sorted pairs, insertion order, level per pair index)."""
    ps = sorted(set((min(v, w), max(v, w)) for v, w in pairs))
    n = len(ps)

    def crosses(p, q):
        return (p[0] < q[0] < p[1] < q[1]) or (q[0] < p[0] < q[1] < p[1])

    cc = [sum(1 for b in range(n) if b != a and crosses(ps[a], ps[b])) for a in range(n)]
    order = sorted(range(n), key=lambda a: (cc[a], ps[a][0]))
    groups = []
    for a in order:
        for g in groups:
            if not any(crosses(ps[a], ps[b]) for b in g):
                g.append(a)
                break
        else:
            groups.append([a])
    groups.sort(key=len, reverse=True)
    return ps, groups


def PairsToDBN(newpairs, length=0, returnlevels=False, levellimit=-1):
    """base pairs -> dbn string (seq.py:104-163)"""
    ps, groups = _pair_levels(newpairs)
    if returnlevels:
        return {ps[a]: lev + 1 for lev, g in enumerate(groups) for a in g}
    if levellimit >= 0:
        groups = groups[:levellimit]
    dbn = ['.'] * length
    for lev, g in enumerate(groups):
        op, cl = (_OPEN[lev], _CLOSE[lev]) if lev < len(_OPEN) else ('.', '.')
        for a in g:
            dbn[ps[a][0]] = op
            dbn[ps[a][1]] = cl
    return ''.join(dbn)


def StemsToDBN(stems, seq):
    return PairsToDBN([bp for stem in stems for bp in stem[0]], len(seq))


def ReAlign(shortdbn, longseq, seqmode=False):
    """put the gaps of longseq back into shortdbn (seq.py:210-233)"""
    ngaps = sum(1 for ch in longseq if ch in GAPS)
    assert len(shortdbn) + ngaps == len(longseq), \
        "Cannot ReAlign dbn string - wrong number of gaps:\n{}\n{}".format(longseq, shortdbn)
    it = iter(shortdbn)
    gap = '-' if seqmode else '.'
    return ''.join(gap if ch in GAPS else next(it) for ch in longseq)


def UnAlign(seq, dbn):
    """remove gap columns (and the pairs that touch them) (seq.py:236-255)"""
    if not any(g in seq for g in GAPS):                    # nothing to remove (the usual single-sequence input)
        return seq, dbn
    if len(seq) == len(dbn):
        # byte arrays instead of per-character joins (alignment rows: hundreds of columns, thousands of rows)
        try:
            sraw = np.frombuffer(seq.encode("latin-1"), dtype=np.uint8)
            draw = np.frombuffer(dbn.encode("latin-1"), dtype=np.uint8)
        except UnicodeEncodeError:
            sraw = None                                    # (Cyrillic brackets of deep pseudoknots, ...: the general path)
        if sraw is not None:
            gap = _GAP_BYTES[sraw]
            pairs = _dbn_pairs(dbn)
            if pairs:
                pr = np.array(pairs, dtype=np.int64)
                hit = gap[pr[:, 0]] | gap[pr[:, 1]]
                if hit.any():
                    draw = draw.copy()
                    draw[pr[hit].ravel()] = 46             # '.'
            keep = ~gap
            return sraw[keep].tobytes().decode("latin-1"), draw[keep].tobytes().decode("latin-1")
    clean = list(dbn)
    for v, w in DBNToPairs(dbn):
        if seq[v] in GAPS or seq[w] in GAPS:
            clean[v] = clean[w] = '.'
    keep = [k for k, ch in enumerate(seq) if ch not in GAPS]
    return ''.join(seq[k] for k in keep), ''.join(clean[k] for k in keep)


def ParseRestraints(restraints):
    """restraint string -> (rbps, rxs, rlefts, rrights) (seq.py:370-376)"""
    rbps = DBNToPairs(restraints)
    rxs, rlefts, rrights = set(), set(), set()
    for m in _RESTR_RE.finditer(restraints):
        ch = m.group()
        (rxs if ch in '_+' else rlefts if ch == '/' else rrights).add(m.start())
    return rbps, rxs, rlefts, rrights


def PairsToStems(sorted_pairs):
    """group sorted pairs into stacked runs (seq.py:498-517): [[pairs, len], ...]"""
    stems = []
    for k, bp in enumerate(sorted_pairs):
        prev = sorted_pairs[k - 1] if k else None
        if prev is None or not (prev[0] + 1 == bp[0] and prev[1] == bp[1] + 1):
            stems.append([[], 0])
        stems[-1][0].append(bp)
        stems[-1][1] += 1
    return stems


def ScoreStruct(seq, stemset, reacts):
    """The three structure scores of a stem list (seq.py:861-899).  Host copy
    used only for the printed `reference` line; predictions are scored on the
    GPU (team_finalize in csrc/sqrn_device.cuh)."""
    table = {"GU": -0.5, "UG": -0.5, "AU": 1.5, "UA": 1.5, "GC": 4.0, "CG": 4.0}
    thescore = 0
    paired = set()
    for stem in stemset:
        bpsum = 0
        for v, w in stem[0]:
            bpsum += table.get(seq[v] + seq[w], 0.0)
            paired.add(v)
            paired.add(w)
        if bpsum > 0:
            thescore += bpsum ** 1.7
    nonsep = [k for k in range(len(seq)) if seq[k] not in SEPS]
    reactscore = 1 - sum(reacts[k] if k in paired else 1 - reacts[k] for k in nonsep) / len(nonsep)
    return round(thescore * reactscore, 3), round(thescore, 3), round(reactscore, 3)


def ReferenceScores(seq, ref, reacts):
    """scores of the known structure (seq.py:958-970)"""
    if not reacts:
        reacts = [0.5] * len(seq)
    reacts = [reacts[k] for k in range(len(seq)) if seq[k] not in GAPS]
    seq, ref = UnAlign(seq, ref)
    return ScoreStruct(seq, PairsToStems(sorted(DBNToPairs(ref))), reacts)


# code point of every int8 level code (+L opening bracket of level L, -L closing one), indexed by
# the code reinterpreted as uint8; levels beyond the 49 bracket pairs print as '.' (seq.py:142-143)
_GLYPH32 = np.full(256, ord('.'), dtype=np.uint32)
for _lev in range(1, 128):
    if _lev <= len(_OPEN):
        _GLYPH32[_lev] = ord(_OPEN[_lev - 1])
        _GLYPH32[256 - _lev] = ord(_CLOSE[_lev - 1])


_GLYPH8 = np.where(_GLYPH32 < 128, _GLYPH32, 0).astype(np.uint8)      # 0: the glyph needs the wide table
_GLYPH_TABLE = _GLYPH8.tobytes()           # the same table for bytes.translate


def _codes_to_dbn(codes):
    """int8 level codes (+L open, -L close) -> glyph string"""
    return _GLYPH32[np.asarray(codes, dtype=np.int8).view(np.uint8)].tobytes().decode("utf-32-le")


def _metrics(pred, known):
    tp = len(pred & known)
    fp = len(pred - known)
    fn = len(known - pred)
    prc = round(tp / (tp + fp), 3) if (tp + fp) else 1
    rcl = round(tp / (tp + fn), 3) if (tp + fn) else 1
    fsc = round(2 * tp / (2 * tp + fp + fn), 3) if (2 * tp + fp + fn) else 1
    return tp, fp, fn, fsc, prc, rcl


# ------------------------------------------------------------ batch front-end
class _Prepared:
    """one sequence digested the way seq.py:1004-1037 does it"""
    __slots__ = ("seq", "shortseq", "shortrest", "_sr", "_rl", "rbps", "rclass", "_keep", "shortdbn",
                 "dbn", "compensated", "bppm", "bppm_key")

    @property
    def shortreacts(self):
        """processed reactivities of the ungapped sequence (all 0.5 when none were given)"""
        return [0.5] * len(self.shortseq) if self._sr is None else self._sr

    @property
    def keep(self):
        """ungapped position -> position in the input sequence"""
        return np.arange(len(self.seq)) if self._keep is None else self._keep


_REACT_LUT = {}


def _react_lut(M=1.8, B=1.6):
    """processed reactivity of every reactivity letter (seq.py:1019-1020 -> ProcessReacts defaults)"""
    key = (M, B)
    if key not in _REACT_LUT:
        chars = sorted(ReactDict)
        vals = ProcessReacts([ReactDict[ch] for ch in chars], M=M, B=B)
        lut = np.full(256, np.nan)
        for ch, v in zip(chars, vals):
            lut[ord(ch)] = v
        _REACT_LUT[key] = lut
    return _REACT_LUT[key]


_GAP_BYTES = np.zeros(256, dtype=bool)
for _ch in GAPS:
    _GAP_BYTES[ord(_ch)] = True
_GAP_DELETE = {ord(_ch): None for _ch in GAPS}      # str.translate: drop the gap symbols
_RC_BYTES = np.zeros(256, dtype=np.uint8)
_RC_BYTES[ord('_')] = _RC_BYTES[ord('+')] = 1
_RC_BYTES[ord('/')] = 2
_RC_BYTES[ord('\\')] = 4
_PLAIN_RESTR = np.zeros(256, dtype=bool)           # restraint symbols that are not brackets
for _ch in "._+/\\-~":
    _PLAIN_RESTR[ord(_ch)] = True


def _prepare(seq, reacts, restraints, dbn):
    """seq.py:1004-1037 for one entry.  The common shapes (no gaps, no restraints, encoded or absent
    reactivities) take vectorised paths; everything else goes through the reference's own steps."""
    p = _Prepared()
    p.bppm = p.bppm_key = p._rl = None
    seq = seq.upper().replace("T", "U")                               # seq.py:1004
    n = len(seq)
    if restraints:
        assert n == len(restraints), "Invalid restraints given"
    if reacts:
        assert len(reacts) == n, "Invalid reactivities given"
    p.seq = seq
    raw = np.frombuffer(seq.encode("latin-1", "replace"), dtype=np.uint8)
    gapmask = _GAP_BYTES[raw]
    has_gaps = bool(gapmask.any())
    p._keep = np.flatnonzero(~gapmask) if has_gaps else None         # None: identity
    # --- restraints -----------------------------------------------------------
    if not restraints:
        p.shortseq = seq.translate(_GAP_DELETE) if has_gaps else seq
        p.shortrest = '.' * len(p.shortseq)
        p.rbps = []
        p.rclass = np.zeros(len(p.shortseq), dtype=np.uint8)
    else:
        rraw = np.frombuffer(restraints.encode("latin-1", "replace"), dtype=np.uint8)
        if not has_gaps and bool(_PLAIN_RESTR[rraw].all()):
            p.shortseq, p.shortrest, p.rbps = seq, restraints, []    # no brackets: nothing for DBNToPairs
            p.rclass = _RC_BYTES[rraw]
        else:
            # the restraint classes of ParseRestraints (seq.py:370-376) are one table look-up per symbol; only the
            # brackets need its parser
            p.shortseq, p.shortrest = UnAlign(seq, restraints) if has_gaps else (seq, restraints)
            p.rbps = DBNToPairs(p.shortrest)
            p.rclass = _RC_BYTES[rraw[p._keep] if has_gaps else rraw]
    # --- reactivities ---------------------------------------------------------
    if not reacts:
        p._sr = None                                                  # all 0.5: "default reacts"
        p.compensated = True
    elif type(reacts) == str:
        letters = np.frombuffer(reacts.encode("latin-1", "replace"), dtype=np.uint8)
        vals = _react_lut()[letters]
        if np.isnan(vals).any():
            raise KeyError(next(ch for ch in reacts if ch not in ReactDict))
        p._sr = vals[p._keep] if has_gaps else vals                   # numpy floats, like ProcessReacts' output
        p._rl = letters[p._keep] if has_gaps else letters             # (their letters: _make_batch codes them without a sort)
        p.compensated = False
    else:
        if has_gaps:
            p._sr = [reacts[k] for k in p._keep.tolist()]
        else:
            p._sr = list(reacts) if n else []
        # builtin sum() in ScoreStruct compensates exact Python floats only (CPython >= 3.12)
        p.compensated = set(map(type, p._sr)) <= {float}
    p.dbn = dbn
    p.shortdbn = None
    if dbn:
        assert len(seq) == len(dbn)
        p.shortdbn = UnAlign(seq, dbn)[1]
    return p


def _encode_symbols(shortseq):
    """str -> bytes for the C ABI; non-latin-1 symbols can never pair and become '?'"""
    return shortseq.encode("latin-1", "replace")


def _make_batch(preps, idx, comp, stemmatrix, interchainonly, bpp=None, **opts):
    """PackedBatch of the prepared entries idx (all with the same reactivity-sum mode `comp`)"""
    # distinct processed reactivities of the batch -> codes + value table (host pow() table in the library)
    codes = values = None
    if idx and all(preps[k]._sr is None or preps[k]._rl is not None for k in idx):
        # letter-encoded (or absent) reactivities: the distinct values are those of the letters that occur -- the same
        # sorted table and codes as below, from a histogram of the letters instead of a sort of every value
        lens_ = [len(preps[k].shortseq) for k in idx]
        letters = np.concatenate([np.zeros(n_, np.uint8) if preps[k]._rl is None else preps[k]._rl for k, n_ in zip(idx, lens_)])
        seen = np.flatnonzero(np.bincount(letters, minlength=256))
        cand = np.where(seen == 0, 0.5, _react_lut()[seen])           # byte 0 stands for "no reactivities": 0.5
        if bool((cand != 0.5).any()):
            values_bits, inv = np.unique(cand.view(np.uint64), return_inverse=True)
            values = values_bits.view(np.float64)
            table = np.zeros(256, np.uint16)
            table[seen] = inv
            coded = table[letters]
            codes, o = [], 0
            for n_ in lens_:
                codes.append(coded[o:o + n_])
                o += n_
        arrs = []
    else:
        arrs = [None if preps[k]._sr is None else np.asarray(preps[k]._sr, dtype=np.float64) for k in idx]
    if any(a is not None and bool((a != 0.5).any()) for a in arrs):
        lens_ = [len(preps[k].shortseq) for k in idx]
        flat = np.concatenate([np.full(n_, 0.5) if a is None else a for a, n_ in zip(arrs, lens_)]) if idx else np.zeros(0)
        # bit patterns, not values: -0.0 / NaN payloads must stay distinct table entries
        values_bits, inverse = np.unique(flat.view(np.uint64), return_inverse=True)
        if len(values_bits) > 65535:
            raise NotImplementedError("more than 65535 distinct reactivity values in one batch")
        values = values_bits.view(np.float64)
        inverse = inverse.astype(np.uint16)
        codes, o = [], 0
        for n_ in lens_:
            codes.append(inverse[o:o + n_])
            o += n_
    any_restr = any(p.rbps or p.rclass.any() for p in (preps[k] for k in idx))
    smat = cols = None
    if stemmatrix is not None:
        smat = np.asarray(stemmatrix, dtype=np.float64)
        cols = [np.asarray(preps[k].keep, dtype=np.int32) for k in idx]
    return PackedBatch([_encode_symbols(preps[k].shortseq) for k in idx],
                       react_codes=codes, react_values=values, react_comp=comp,
                       restr_class=[preps[k].rclass for k in idx] if any_restr else None,
                       rbps=[np.array(preps[k].rbps, dtype=np.int32).reshape(-1, 2) for k in idx] if any_restr else None,
                       smat=smat, cols=cols, interchainonly=interchainonly, max_structs=0,
                       bpp_mode=bpp[0] if bpp else 0, bpp_terms=bpp[1] if bpp else None, **opts)


# ---------------------------------------------------------------- non-greedy algorithms (host)
def ConsensusStemSet(stemsets):
    """base pairs present in every stem list (seq.py:845-858)"""
    common = None
    for stemset in stemsets:
        bps = {bp for stem in stemset for bp in stem[0]}
        common = bps if common is None else common & bps
    return common or set()


def RankStructs(stemsets, rankbydiff=False, rankby=(0, 2, 1), priority=set()):
    """order of the predicted structures (seq.py:902-955): stable descending sort by the rankby score tuple,
    structures of priority parameter sets first, then -- with rankbydiff -- repeatedly the structure that adds
    most base pairs not seen so far.  stemsets: [stems, scores, paramset indices]"""
    def score_key(x):
        return [x[1][rb] for rb in rankby]

    ranked = sorted(stemsets, key=score_key, reverse=True)
    ranked = [x for x in ranked if priority & set(x[2])] + [x for x in ranked if not (priority & set(x[2]))]
    if not rankbydiff or len(ranked) < 3:
        return ranked
    bpsets = {id(x): {bp for stem in x[0] for bp in stem[0]} for x in ranked}
    everything = set().union(*bpsets.values())
    seen = set(bpsets[id(ranked[0])])
    cur = 1
    while seen != everything and cur < len(ranked) - 1:
        tail = sorted(ranked[cur:], key=lambda x: (len(bpsets[id(x)] - seen), score_key(x)), reverse=True)
        ranked = ranked[:cur] + tail
        seen |= bpsets[id(ranked[cur])]
        cur += 1
    return ranked[:cur] + sorted(ranked[cur:], key=score_key, reverse=True)


def _cell_scorer(p, paramset, smat, bpp_mode=0, bpp_term=None):
    """scoremat[v, w] of BPMatrix for one prepared entry (seq.py:258-339 and the bpp term 350-364, times the
    alignment weight 1084-1085)"""
    weights = {}
    for bp, w in paramset["bpweights"].items():
        weights[bp] = w
        weights[bp[1] + bp[0]] = w
    seq, reacts = p.shortseq, p.shortreacts
    default = p._sr is None or set(reacts) == {0.5}
    keep = p.keep

    def score(v, w):
        base = weights.get(seq[v] + seq[w], 0)
        rf = 1 if default else ((1 - (reacts[v] + reacts[w]) / 2) * 2) ** 0.5
        if base <= 0:
            rf = 1 / max(rf, 0.01)
        val = base * 1.0 * rf                        # bps * boolmat * reactfactor: the cell is a live pair here
        if bpp_mode == 1:
            val = val + bpp_term[v, w]
        elif bpp_mode == 2:
            val = val * bpp_term[v, w]
        if smat is not None:
            val = val * smat[keep[v], keep[w]]
        return val
    return score


def RunAlgo(seq, stems, cell_score, minlen, minscore, algo="E", levellimit=3, pairs=None):
    """one non-greedy prediction (seq.py:548-595).  stems: AnnotateStems output [[pairs, len, score], ...];
    cell_score(v, w) = bpscorematrix[v, w].  pairs: what the builder returned when it ran elsewhere (the device
    Nussinov, Hungarian or Edmonds builder); `stems` is then not read."""
    from . import SQRNalgos
    N = len(seq)
    if pairs is not None:
        pass                                         # the builder already ran
    elif algo == "E":
        pairs = SQRNalgos.Edmonds(stems)
    elif algo == "N":
        pairs = SQRNalgos.Nussinov(seq, stems, N, SEPS)
    elif algo == "H":
        pairs = SQRNalgos.Hungarian(seq, stems, N, SEPS)
    else:
        pairs = []

    def passing(pairlist):                           # partial stems below the thresholds go
        out = []
        for stem in PairsToStems(sorted((min(v, w), max(v, w)) for v, w in pairlist)):
            score = sum(cell_score(v, w) for v, w in stem[0])
            if score >= minscore and stem[1] >= minlen:
                out.append((stem, score))
        return out

    kept = [bp for stem, _ in passing(pairs) for bp in stem[0]]
    kept = DBNToPairs(PairsToDBN(kept, N, levellimit=levellimit))      # pseudoknots beyond the level limit go
    levels = PairsToDBN(kept, N, returnlevels=True)
    stemset = []
    for stem, score in passing(kept):
        if levels[stem[0][0]] > 1 and stem[1] < 4:                      # short pseudoknotted stems go
            continue
        stemset.append(stem + [score, score, ''])
    return stemset


def _predict_many_mixed(entries, paramsets, conslim, toplim, hardrest, rankbydiff, rankby, interchainonly,
                        stemmatrix, poollim, priority, algos, device, levellimit, M=1.8, B=-0.6):
    """SQRNdbnseq (seq.py:1039-1286) for parameter sets that name Nussinov / Hungarian / Edmonds or weight the
    score matrix with base-pair probabilities (bpp != 0): per parameter set the greedy structures come from
    sqrn_predict_batch and the stems for the other builders from sqrn_yield_stems_batch (both with that set's bpp
    term); de-duplication, ScoreStruct of the host-built structures, ranking and consensus follow the reference on
    the host."""
    preps = [_prepare(*e) for e in entries]
    ctx = get_context(device)
    n = len(entries)
    smat_np = None if stemmatrix is None else np.asarray(stemmatrix, dtype=np.float64)
    per_ps = [[None] * len(paramsets) for _ in range(n)]       # [entry][paramset] -> list of (stems, scores) in order
    for psi, ps in enumerate(paramsets):
        use = set(algos) if algos else set(ps["algorithms"])
        for k in range(n):
            per_ps[k][psi] = []
        for comp in (False, True):
            idx = [k for k in range(n) if preps[k].compensated == comp]
            if not idx:
                continue
            bpp = _bpp_terms(preps, idx, ps, M, B)
            others = [a for a in use if a != "G"]             # set order, as in the reference's `for algo in algos`
            if others:
                batch = _make_batch(preps, idx, comp, stemmatrix, interchainonly, bpp=bpp)
                found = ctx.yield_stems(ps, batch)
                # Nussinov, Hungarian and Edmonds on the device when the context has the builder (the host SQRNalgos
                # functions otherwise): one call each for the group, over the stems just enumerated; the stem lists are
                # built only for a builder that runs on the host
                nuss = getattr(ctx, "nussinov", None) if "N" in others else None
                dev_pairs = {"N": nuss(batch.symbols, batch.offsets, found, minloop=3)} if nuss is not None else {}
                for algo, name, kw in (("H", "hungarian", dict(minloop=3, power=1.7)), ("E", "edmonds", dict(power=1.7))):
                    build = getattr(ctx, name, None) if algo in others else None
                    if build is None:
                        continue
                    try:
                        dev_pairs[algo] = build(batch.symbols, batch.offsets, found, **kw)
                    except SqrnError as e:
                        # negative / NaN scores or non-finite / huge weights: the host builder gives what it gives today
                        if e.code != E_BADARG:
                            raise
                lists = any(a not in dev_pairs for a in others)
                for q, (k, (st, sc)) in enumerate(zip(idx, found)):
                    p = preps[k]
                    stems = [[[(i + t, j - t) for t in range(ln)], ln, float(s_)] for (i, j, ln), s_ in zip(st.tolist(), sc.tolist())] if lists else None
                    cell = _cell_scorer(p, ps, smat_np, bpp[0] if bpp else 0, bpp[1][q] if bpp else None)
                    ll = levellimit if levellimit is not None else 3 - int(len(p.shortseq) > 500)
                    for algo in others:
                        pairs = dev_pairs[algo][q].tolist() if algo in dev_pairs else None
                        stemset = RunAlgo(p.shortseq, stems, cell, ps["minlen"], ps["minbpscore"], algo, ll, pairs=pairs)
                        per_ps[k][psi].append((stemset, ScoreStruct(p.shortseq, stemset, p.shortreacts)))
            if "G" in use:
                batch = _make_batch(preps, idx, comp, stemmatrix, interchainonly, bpp=bpp, hardrest=False,
                                    rankbydiff=False, poollim=poollim, conslim=1, rankby=rankby, priority_mask=0)
                for k, (_cons, structs, *_rest) in zip(idx, ctx.predict_batch([ps], batch)):
                    for codes, sc, isint, _mask, stems in structs:
                        stemset = [[[(i + q, j - q) for q in range(ln)], ln] for i, j, ln in np.asarray(stems).tolist()]
                        total, struct, react = sc
                        per_ps[k][psi].append((stemset, (total, 0 if isint else struct, react)))
    final = []
    for k, p in enumerate(preps):
        fin, seen = [], {}
        for psi in range(len(paramsets)):
            for stemset, scores in per_ps[k][psi]:
                key = tuple(sorted(bp for stem in stemset for bp in stem[0]))
                if key not in seen:
                    fin.append([stemset, scores, psi])
                    seen[key] = {psi}
                else:
                    seen[key].add(psi)
        for item in fin:
            item[2] = sorted(seen[tuple(sorted(bp for stem in item[0] for bp in stem[0]))])
        ranked = RankStructs(fin, rankbydiff, rankby, priority=set(priority))
        sseq = p.shortseq
        bpw = paramsets[-1]["bpweights"]                               # the loop variable the reference leaves behind
        forced = {(v, w) for v, w in p.rbps if sseq[v] + sseq[w] in bpw or sseq[w] + sseq[v] in bpw} if hardrest else set()
        n_short = len(sseq)

        def expand(pairs, p=p, n_short=n_short):
            dbn = ReAlign(PairsToDBN(pairs, n_short), p.seq)
            return ''.join(p.seq[q] if p.seq[q] in SEPS else dbn[q] for q in range(len(p.seq)))

        dbns = [expand({bp for stem in x[0] for bp in stem[0]} | forced) for x in ranked]
        consbps = ConsensusStemSet([x[0] for x in ranked[:conslim]]) | forced
        cons = expand(consbps)
        preds = [(dbn, x[1], x[2]) for dbn, x in zip(dbns, ranked)]
        if p.dbn:
            known = set(DBNToPairs(p.shortdbn))
            consresult = list(_metrics(set(consbps), known))
            best, result = -1, []
            for rank, x in enumerate(ranked):
                bps = {bp for stem in x[0] for bp in stem[0]} | forced
                tp, fp, fn, fsc, prc, rcl = _metrics(bps, known)
                if fsc > best:
                    best = fsc
                    result = [tp, fp, fn, fsc, prc, rcl, rank + 1]
                if rank + 1 >= toplim:
                    break
            final.append((cons, preds, consresult, result))
        else:
            final.append((cons, preds, [np.nan] * 6, [np.nan] * 7))
    return final


def predict_many(entries, paramsets, conslim=1, toplim=5, hardrest=False, rankbydiff=False,
                 rankby=(0, 2, 1), interchainonly=False, stemmatrix=None, poollim=1000,
                 priority=frozenset(), algos=frozenset(), device=None, levellimit=None, M=1.8, B=-0.6, devices=None):
    """Batched SQRNdbnseq: entries = [(seq, reacts, restraints, dbn)], one GPU call for all of them per GPU.
    devices=None: every visible GPU -- the entries are dealt by length to one host thread per GPU (the
    reference's Pool(threads) over sequences, SQUARNA.py:889) and come back in input order; `device` (an int) or
    a list in `devices` names the GPUs explicitly.  Returns the reference's 4-tuple per entry."""
    assert set(rankby) == {0, 1, 2} and len(rankby) == 3, "Invalid ranking indices"
    devs = [device] if device is not None else _resolve_devices(devices)
    if len(devs) > 1 and len(entries) >= 2 * len(devs):
        return run_sharded(lambda sub, dev: predict_many(sub, paramsets, conslim, toplim, hardrest, rankbydiff,
                                                         rankby, interchainonly, stemmatrix, poollim, priority,
                                                         algos, dev, levellimit, M, B),
                           entries, [len(e[0]) for e in entries], devs)
    device = devs[0]
    # which parameter sets run the greedy algorithm (seq.py:1046-1102)
    gsets = []
    mixed = False
    for psi, ps in enumerate(paramsets):
        use = set(algos) if algos else set(ps["algorithms"])
        if use - {"G"} or ps.get("bpp", 0):
            # Nussinov / Hungarian / Edmonds sets: stems and the builders on the GPU (SURVEY 8f-2);
            # bpp sets: the probabilities come from the host (ViennaRNA or set_rna_module) as one term per
            # parameter set (SURVEY 8f-4), so the sets run one call each
            mixed = True
        if "G" in use:
            gsets.append(psi)
    if mixed:
        if any(ps.get("bpp", 0) for ps in paramsets):
            _rna()                                  # ModuleNotFoundError now, as the reference's `import RNA`, not after GPU work
            # N x N float64 per entry and bpp set on the device: bound the cells per call
            out, chunk, cells = [], [], 0
            for e in entries:
                c = len(e[0]) ** 2
                if chunk and cells + c > (1 << 25):
                    out += _predict_many_mixed(chunk, paramsets, conslim, toplim, hardrest, rankbydiff, rankby,
                                               interchainonly, stemmatrix, poollim, priority, algos, device, levellimit, M, B)
                    chunk, cells = [], 0
                chunk.append(e)
                cells += c
            if chunk:
                out += _predict_many_mixed(chunk, paramsets, conslim, toplim, hardrest, rankbydiff, rankby,
                                           interchainonly, stemmatrix, poollim, priority, algos, device, levellimit, M, B)
            return out
        return _predict_many_mixed(entries, paramsets, conslim, toplim, hardrest, rankbydiff, rankby,
                                   interchainonly, stemmatrix, poollim, priority, algos, device, levellimit, M, B)
    import time
    t_0 = time.perf_counter()
    preps = [_prepare(*e) for e in entries]
    t_1 = time.perf_counter()
    t_call = 0.0
    results = [None] * len(entries)
    if not gsets:
        todo = []
    else:
        todo = list(range(len(entries)))
    # sequences sharing the same reactivity-sum mode go into the same batch
    for comp in (False, True):
        idx = [k for k in todo if preps[k].compensated == comp]
        if not idx:
            continue
        batch = _make_batch(preps, idx, comp, stemmatrix, interchainonly, hardrest=hardrest, rankbydiff=rankbydiff,
                            poollim=poollim, conslim=conslim, rankby=rankby,
                            priority_mask=sum(1 << gsets.index(p) for p in priority if p in gsets))
        t_c = time.perf_counter()
        flat = get_context(device).predict_batch_flat([paramsets[g] for g in gsets], batch)
        t_call += time.perf_counter() - t_c
        for q, k in enumerate(idx):
            results[k] = (flat, q)

    # The reference's 4-tuple per entry.  With pl=100 a sequence has tens of structures: their texts come from one glyph
    # gather and one decode per sequence, their score tuples straight from the flat result's columns.
    t_2 = time.perf_counter()
    inds_of = {}
    final = []
    # (tens of thousands of small tuples and strings, none of them cyclic: the collector's generation scans over the
    #  growing result cost 40 % of this loop, so it rests while the loop runs)
    import gc
    gc_was_on = gc.isenabled()
    gc.disable()
    try:
        for k, p in enumerate(preps):
            seq = p.seq
            keep = p._keep
            seps = ';' in seq or '&' in seq
            width = len(seq)
            if seps or keep is not None:
                raw8 = np.frombuffer(seq.encode("latin-1", "replace"), dtype=np.uint8)
                seppos = np.flatnonzero((raw8 == 59) | (raw8 == 38)) if seps else ()        # ';' '&'

            def expand(codes2d):                       # glyphs + ReAlign + separators (seq.py:1239-1246), one row per structure
                if keep is None and not seps:
                    text = codes2d.tobytes().translate(_GLYPH_TABLE).decode("latin-1")
                    if "\x00" not in text:
                        return text
                for table, wide, encoding in ((_GLYPH8, np.uint8, "latin-1"), (_GLYPH32, np.uint32, "utf-32-le")):
                    g = np.take(table, codes2d.view(np.uint8))
                    if keep is not None:
                        long_ = np.full((len(g), width), 46, dtype=wide)
                        long_[:, keep] = g
                        g = long_
                    if seps:
                        g[:, seppos] = raw8[seppos]
                    if wide is np.uint32 or bool(g.all()):          # (0: a level of the Cyrillic part of the alphabet)
                        return g.tobytes().decode(encoding)

            if results[k] is None:
                cons_codes, c2, k0, k1, flat = np.zeros(len(p.shortseq), np.int8), None, 0, 0, None
            else:
                flat, q = results[k]
                cons_codes, k0, k1 = flat.cons_codes(q), flat.so[q], flat.so[q + 1]
                c2 = flat.codes2d(q) if k1 > k0 else None
            cons = expand(cons_codes.reshape(1, -1))
            preds = []
            if c2 is not None:
                whole = flat.text(q) if keep is None and not seps else None      # (the library's threaded glyph pass)
                if whole is None or "\x00" in whole:
                    whole = expand(c2)
                for j, sc, isint, mask in zip(range(0, (k1 - k0) * max(width, 1), max(width, 1)), flat.scores[k0:k1],
                                              flat.isint[k0:k1], flat.mask[k0:k1]):
                    inds = inds_of.get(mask)
                    if inds is None:
                        inds = inds_of[mask] = [gsets[b] for b in range(len(gsets)) if mask >> b & 1]
                    preds.append((whole[j:j + width], (sc[0], 0 if isint else sc[1], sc[2]), inds[:]))
            if p.dbn:                                # seq.py:1249-1285
                known = set(DBNToPairs(p.shortdbn))
                consresult = list(_metrics(set(DBNToPairs(_codes_to_dbn(cons_codes))), known))
                best, result = -1, []
                for rank in range(k1 - k0):
                    tp, fp, fn, fsc, prc, rcl = _metrics(set(DBNToPairs(_codes_to_dbn(c2[rank]))), known)
                    if fsc > best:
                        best = fsc
                        result = [tp, fp, fn, fsc, prc, rcl, rank + 1]
                    if rank + 1 >= toplim:
                        break
                final.append((cons, preds, consresult, result))
            else:
                final.append((cons, preds, [np.nan] * 6, [np.nan] * 7))
    finally:
        if gc_was_on:
            gc.enable()
    if os.environ.get("SQRN_TRACE") is not None:
        print("[sqrn] predict_many: prepare %.3f s, pack %.3f s, library call %.3f s, assemble %.3f s (%d entries)"
              % (t_1 - t_0, t_2 - t_1 - t_call, t_call, time.perf_counter() - t_2, len(entries)), file=sys.stderr)
    return final


def SQRNdbnseq(seq, reacts=None, restraints=None, dbn=None,
               paramsets=[], conslim=1, toplim=5,
               hardrest=False, rankbydiff=False,
               rankby=(0, 2, 1), interchainonly=False,
               threads=1, mp=True, stemmatrix=None, poollim=1000,
               entropy=False, algos=set(), levellimit=None,
               priority=set(),
               M=1.8, B=-0.6):
    """Predict alternative secondary structures of one sequence; same signature
    and return value as the reference (seq.py:973-1286):
    (consensus_dbn, [(dbn, (total, struct, react), [paramset indices]), ...],
     consensus_metrics[6], topN_metrics[7]).

    threads / mp only choose a multiprocessing layout in the reference and never
    change results; here the work is one batched GPU call.  Parameter sets that name Nussinov / Hungarian /
    Edmonds get their stems from the GPU, and those builders run there too (SQRNalgos.py is the reference); `entropy=True`
    returns the stem-matrix entropy string of the first parameter set."""
    if entropy:
        return Entropy(seq, reacts, restraints, paramsets[0], interchainonly, stemmatrix, M=M, B=B)
    return predict_many([(seq, reacts, restraints, dbn)], paramsets, conslim, toplim, hardrest,
                        rankbydiff, rankby, interchainonly, stemmatrix, poollim,
                        frozenset(priority), frozenset(algos), levellimit=levellimit, M=M, B=B)[0]


def _stem_matrix_entropy(n, stems, scores):
    """seq.py:520-545 from the (i, j, len) stems of one AnnotateStems pass and their scores"""
    mat = np.zeros((n, n))
    for (i, j, ln), score in zip(stems.tolist(), scores.tolist()):
        for q in range(ln):
            mat[i + q, j - q] = score
            mat[j - q, i + q] = score
    ent = 0
    for row in mat:
        tot = row.sum()
        if tot:
            probs = [x for x in row / tot if x]
            ent += sum(-(probs * np.log2(probs)))
    return str(round(ent / n, 3))


def entropy_many(entries, paramset, interchainonly=False, stemmatrix=None, device=0, M=1.8, B=-0.6):
    """Entropy for many entries [(seq, reacts, restraints)] with one sqrn_yield_stems_batch call per
    reactivity-sum mode; returns the strings in input order"""
    preps = [_prepare(seq, reacts, restraints, None) for seq, reacts, restraints in entries]
    out = [None] * len(preps)
    ctx = get_context(device)
    for comp in (False, True):
        idx = [k for k, p in enumerate(preps) if p.compensated == comp]
        if not idx:
            continue
        batch = _make_batch(preps, idx, comp, stemmatrix, interchainonly,
                            bpp=_bpp_terms(preps, idx, paramset, M, B))
        for k, (st, sc) in zip(idx, ctx.yield_stems(paramset, batch)):
            out[k] = _stem_matrix_entropy(len(preps[k].shortseq), st, sc)
    return out


def Entropy(seq, reacts, restraints, paramset, interchainonly=False, stemmatrix=None, device=0, M=1.8, B=-0.6):
    """mean row entropy of the stem-score matrix of the first parameter set, as the string the reference returns
    (seq.py:520-545, reached through SQRNdbnseq(entropy=True), seq.py:1087-1089): every stem AnnotateStems finds
    writes its score into the cells of its pairs (both triangles); a row's entropy is that of its non-zero cells
    normalised to 1.  The stems come from sqrn_yield_stems_batch."""
    return entropy_many([(seq, reacts, restraints)], paramset, interchainonly, stemmatrix, device, M, B)[0]


def _print_entry(name, sequence, reactivities, restraints, reference, reactformat, sink, rfam=None, entropy_val=None):
    """header block of RunSQRNdbnseq (seq.py:1301-1345); entropy_val: the string SQRNdbnseq(entropy=True) returned
    (seq.py:1313-1318 prints it next to the sequence)"""
    print(name, file=sink)
    if entropy_val is not None:
        print('\t'.join([sequence, "entropy:", entropy_val]), file=sink)
    else:
        print(sequence, file=sink)
    if reactivities:
        print(EncodedReactivities(sequence, reactivities, reactformat), "reactivities", sep='\t', file=sink)
    def with_separators(line):                   # the chain separators of the sequence shine through (seq.py:1326-1341)
        if len(line) == len(sequence) and ';' not in sequence and '&' not in sequence:
            return line
        return ''.join(sequence[k] if sequence[k] in SEPS else line[k] for k in range(len(sequence)))

    if restraints:
        print(with_separators(restraints), "restraints" + ("(" + rfam + ")" if rfam else ""), sep='\t', file=sink)
    if reference:
        print(with_separators(reference), "reference", *ReferenceScores(sequence, reference, reactivities), sep='\t', file=sink)
    print('_' * len(sequence), file=sink)


def _print_prediction(prediction, sequence, restraints, reference, paramsetnames, conslim, outplim, sink,
                      rfam=None):
    """result block of RunSQRNdbnseq (seq.py:1357-1406)"""
    consensus, predicted_structures, consensus_metrics, topN_metrics = prediction
    g4 = bool(rfam and restraints and '+' in restraints)
    if g4:
        consensus = ''.join('+' if restraints[k] == '+' else ch for k, ch in enumerate(consensus))
    if reference:
        print(consensus, "top-{}_consensus".format(conslim),
              "TP={},FP={},FN={},FS={},PR={},RC={}".format(*consensus_metrics), sep='\t', file=sink)
    else:
        print(consensus, "top-{}_consensus".format(conslim), sep='\t', file=sink)
    print('=' * len(sequence), file=sink)
    for k, (struct, scores, inds) in enumerate(predicted_structures[:outplim]):
        if g4:
            struct = ''.join('+' if restraints[q] == '+' else ch for q, ch in enumerate(struct))
        total, structscore, reactscore = scores
        fields = [struct, "#{}".format(k + 1), total, structscore, reactscore,
                  ','.join(paramsetnames[q] for q in inds)]
        if reference and k + 1 == topN_metrics[-1]:
            fields.append("TP={},FP={},FN={},FS={},PR={},RC={},RK={}".format(*topN_metrics))
        print(*fields, sep='\t', file=sink)
    return consensus, predicted_structures, consensus_metrics, topN_metrics


def _resolve_priority(priority, paramsetnames, rfam):
    if rfam and priority == {'bppN', 'bppH1', 'bppH2'}:          # seq.py:1304-1305
        priority = None
    if priority:
        return {k for k in range(len(paramsetnames)) if paramsetnames[k] in priority}
    return set()


def RunSQRNdbnseq(name, sequence, reactivities, restraints,
                  reference, paramsetnames,
                  paramsets, threads, rankbydiff, rankby,
                  hardrest, interchainonly, toplim, outplim,
                  conslim, reactformat, evalonly, poollim=1000,
                  mp=True, sink=sys.stdout, stemmatrix=None,
                  entropy=False, algos={'G', }, levellimit=None,
                  priority=None, rfam=None, M=1.8, B=-0.6):
    """Print the reference's text block for one entry and return the prediction
    4-tuple (seq.py:1289-1408)."""
    priority = _resolve_priority(priority, paramsetnames, rfam)
    entropy_val = None
    if entropy:                                                  # seq.py:1313-1318
        entropy_val = SQRNdbnseq(sequence, reactivities, restraints, reference, paramsets, conslim, toplim, hardrest,
                                 rankbydiff, rankby, interchainonly, threads, mp, stemmatrix, poollim,
                                 entropy=True, algos=algos, M=M, B=B)
    _print_entry(name, sequence, reactivities, restraints, reference, reactformat, sink, rfam, entropy_val)
    if evalonly:
        return None, None, None, None
    prediction = SQRNdbnseq(sequence, reactivities, restraints, reference,
                            paramsets, conslim, toplim, hardrest,
                            rankbydiff, rankby, interchainonly, threads, mp, stemmatrix,
                            poollim, algos=algos, levellimit=levellimit, priority=priority,
                            M=M, B=B)
    return _print_prediction(prediction, sequence, restraints, reference, paramsetnames, conslim, outplim,
                             sink, rfam)


def RunSQRNdbnseqBatch(entries, paramsetnames, paramsets, rankbydiff, rankby, hardrest, interchainonly,
                       toplim, outplim, conslim, reactformat, evalonly, poollim=1000, sink=sys.stdout,
                       stemmatrix=None, algos={'G', }, priority=None, rfam=None, levellimit=None,
                       entropy=False, M=1.8, B=-0.6, devices=None, header_on_error=True):
    """RunSQRNdbnseq for many entries [(name, seq, reacts, restraints, reference)]
    with ONE batched GPU call; text is written in input order (what the
    reference's ordered imap gives, SQUARNA.py:929-935)."""
    priority_in = priority
    priority = _resolve_priority(priority, paramsetnames, rfam)
    preds = [None] * len(entries)
    ents = [None] * len(entries)
    try:
        if entropy:                                              # seq.py:1313-1318, before evalonly returns
            ents = entropy_many([(e[1], e[2], e[3]) for e in entries], paramsets[0], interchainonly, stemmatrix, M=M, B=B)
        if not evalonly:
            preds = predict_many([(e[1], e[2], e[3], e[4]) for e in entries], paramsets, conslim, toplim,
                                 hardrest, rankbydiff, rankby, interchainonly, stemmatrix, poollim,
                                 frozenset(priority), frozenset(algos), levellimit=levellimit, M=M, B=B, devices=devices)
    except Exception:
        # An entry the prediction rejects.  The reference handles one entry at a time (SQUARNA.py:887-935), so it has
        # printed every entry before the bad one, and that entry's own header (seq.py:1300-1345), when it raises:
        # redo the batch entry by entry to fail at the same place.
        if len(entries) == 1:
            if not entropy and header_on_error:          # (byseq workers print into a buffer of their own, which is dropped)
                _print_entry(*entries[0], reactformat, sink, rfam, None)
            raise
        out = []
        for e in entries:
            out += RunSQRNdbnseqBatch([e], paramsetnames, paramsets, rankbydiff, rankby, hardrest, interchainonly, toplim,
                                      outplim, conslim, reactformat, evalonly, poollim, sink, stemmatrix, algos, priority_in,
                                      rfam, levellimit, entropy, M, B, devices, header_on_error)
        return out
    out = []
    for (name, seq, reacts, rests, ref), pred, ent in zip(entries, preds, ents):
        _print_entry(name, seq, reacts, rests, ref, reactformat, sink, rfam, ent)
        if evalonly:
            out.append((None, None, None, None))
        else:
            out.append(_print_prediction(pred, seq, rests, ref, paramsetnames, conslim, outplim, sink, rfam))
    return out
