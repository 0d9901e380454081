"""The Hungarian builder on the device (include/sqrn.h: sqrn_hungarian_batch, csrc/sqrn_hungarian.cuh) against SciPy's
linear_sum_assignment and the host restatement squarna_b200/SQRNalgos.Hungarian, pair for pair.

Without a GPU the assignment and the filter run through tests/emu/hungarian_emu.cpp, the host build of the same header,
with the scan of each step split over simulated teams of 1, 32 (the warp tier) and 256 lanes (the CTA and global
tiers) whose partial keys meet as on the device.  With -m gpu the C entry runs on the device: against the host builder
up to 5000 nt and across the tier thresholds, against the emulator at 12 000 nt, and end to end through predict_many /
the CLI against the same calls through a context without the builder."""
import contextlib
import ctypes as C
import io
import math
import os
import random
import subprocess

import numpy as np
import pytest
from scipy.optimize import linear_sum_assignment

from oracle import oracle as O
from squarna_b200 import SQRNalgos, SQRNdbnseq as S
from squarna_b200._abi import E_BADARG, OK, pack_sequences
from tests import common as T

_HERE = os.path.dirname(os.path.abspath(__file__))
_ROOT = os.path.dirname(_HERE)
_CSRC = os.path.join(_ROOT, "squarna_b200", "csrc")
_EMU_SRC = [os.path.join(_HERE, "emu", "hungarian_emu.cpp")] + \
    [os.path.join(_CSRC, f) for f in ("sqrn_hungarian.cuh", "sqrn_nussinov.cuh", "sqrn_device.cuh", "sqrn_params.h")]
_EMU_SO = os.path.join(_HERE, "emu", "_build", "libhungarian_emu.so")
SEPS = S.SEPS
WIDTHS = (1, 32, 256)
MAX_LEN = 32767
_emu_lib = None


def _emu():
    """the emulation build (g++ -ffp-contract=off, as tests/emu/emu.py), rebuilt when a source is newer"""
    global _emu_lib
    if _emu_lib is None:
        if not os.path.exists(_EMU_SO) or any(os.path.getmtime(s) > os.path.getmtime(_EMU_SO) for s in _EMU_SRC):
            os.makedirs(os.path.dirname(_EMU_SO), exist_ok=True)
            # parallel test workers may all build: each writes its own file and renames it into place
            tmp = "%s.%d.tmp" % (_EMU_SO, os.getpid())
            subprocess.check_call(["g++", "-O2", "-g", "-std=c++17", "-ffp-contract=off", "-fPIC", "-shared",
                                   "-Wno-unknown-pragmas", "-o", tmp, _EMU_SRC[0], "-lm"])
            os.replace(tmp, _EMU_SO)
        L = C.CDLL(_EMU_SO)
        L.emu_hu_smem_max_n.argtypes = [C.c_longlong]
        L.emu_lsap.argtypes = [C.c_int] + [C.c_void_p] * 3 + [C.c_int, C.c_void_p]
        L.emu_hungarian.argtypes = [C.c_int64] + [C.c_void_p] * 5 + [C.c_int, C.c_double, C.c_int] + [C.c_void_p] * 2
        _emu_lib = L
    return _emu_lib


def _ptr(a):
    return a.ctypes.data_as(C.c_void_p)


def _flat(seqs, stem_lists):
    """(symbols, offsets, stem_offsets, stems (k,3), scores) of sequences and their (i, j, len, score) stem lists"""
    sym, off = pack_sequences(seqs)
    so = np.zeros(len(seqs) + 1, np.int64)
    np.cumsum([len(x) for x in stem_lists], out=so[1:])
    rows = [s for x in stem_lists for s in x]
    st = np.array([s[:3] for s in rows] or [(0, 0, 0)], np.int32).reshape(-1, 3)
    sc = np.array([s[3] for s in rows] or [0.0], np.float64)
    return sym, off, so, st, sc


def emu_hungarian(seqs, stem_lists, width=256, minloop=3, power=1.7):
    """pairs per sequence from the emulated device code, as lists of (v, w); or the error code"""
    sym, off, so, st, sc = _flat(seqs, stem_lists)
    po = np.zeros(len(seqs) + 1, np.int64)
    pairs = np.zeros((max(int((np.diff(off) // 2).sum()), 1), 2), np.int32)
    rc = _emu().emu_hungarian(len(seqs), _ptr(off), _ptr(sym), _ptr(so), _ptr(st), _ptr(sc), minloop, power, width,
                              _ptr(po), _ptr(pairs))
    if rc != OK:
        return rc
    return [[tuple(p) for p in pairs[po[b]:po[b + 1]].tolist()] for b in range(len(seqs))]


def emu_lsap(n, entries, width):
    """col4row of the emulated assignment on the symmetric matrix with cost c at (v, w) and (w, v) for (v, w, c)"""
    rows = [[] for _ in range(n)]
    for v, w, c in entries:
        rows[v].append((w, c))
        rows[w].append((v, c))
    rp = np.zeros(n + 1, np.int64)
    np.cumsum([len(r) for r in rows], out=rp[1:])
    col = np.array([x[0] for r in rows for x in r] or [0], np.int16)
    cost = np.array([x[1] for r in rows for x in r] or [0.0], np.float64)
    out = np.zeros(max(n, 1), np.int32)
    assert _emu().emu_lsap(n, _ptr(rp), _ptr(col), _ptr(cost), width, _ptr(out)) == OK
    return out[:n].tolist()


def device_hungarian(ctx, seqs, stem_lists, minloop=3, power=1.7):
    sym, off, so, st, sc = _flat(seqs, stem_lists)
    per = [(st[so[b]:so[b + 1]], sc[so[b]:so[b + 1]]) for b in range(len(seqs))]
    return [[tuple(p) for p in x.tolist()] for x in ctx.hungarian(sym, off, per, minloop=minloop, power=power)]


def host_hungarian(seq, stems, minloop=3, power=1.7):
    lists = [[[(i + t, j - t) for t in range(ln)], ln, sc] for i, j, ln, sc in stems]
    return SQRNalgos.Hungarian(seq, lists, len(seq), SEPS, minloop=minloop, power=power)


# ---------------------------------------------------------------- generators
def _conf(name):
    from squarna_b200 import SQUARNA as CLI
    return CLI.ParseConfig(os.path.join(os.path.dirname(os.path.abspath(CLI.__file__)), name + ".conf"))[1]


def _conf_sets():
    """the H-running parameter sets of every shipped configuration"""
    from squarna_b200 import SQUARNA as CLI
    pkg = os.path.dirname(os.path.abspath(CLI.__file__))
    out = {}
    for f in sorted(os.listdir(pkg)):
        if f.endswith(".conf"):
            names, sets = CLI.ParseConfig(os.path.join(pkg, f))
            for nm, ps in zip(names, sets):
                if "H" in ps["algorithms"]:
                    out.setdefault((nm, tuple(sorted(ps["bpweights"].items())), ps["minlen"], ps["minbpscore"]), ps)
    return list(out.values())


def _rand_paramset(rng):
    w = {k: rng.choice([0.0, 0.5, 1.0, 1.25, 2.0, 3.25, 3.5]) for k in ("GC", "AU", "GU")}
    if rng.random() < 0.3:
        w["GA"] = rng.choice([0.5, 1.0])
    return T._ps(algorithms={"H"}, bpweights=w, minlen=float(rng.choice([1, 2, 3, 4])),
                 minbpscore=rng.choice([0.0, 0.0, 1.0, 2.75, 4.5, 6.0]))


def annotated_cases(seed, count, lo, hi, with_smat=None):
    """(shortseq, stems) of random SQRNdbnseq inputs (separators, restraints, reactivities, gaps) under the H-running
    sets of the shipped configurations and random parameter sets (minbpscore 0 among them), half with a stem matrix"""
    rng = random.Random(seed)
    sets = _conf_sets()
    out = []
    for _ in range(count):
        seq, reacts, rest, _kw = T.rand_case(rng, lo, hi)
        p = S._prepare(seq, reacts, rest, None)
        ps = rng.choice(sets) if rng.random() < 0.6 else _rand_paramset(rng)
        n = len(p.shortseq)
        smat = None
        if (rng.random() < 0.5) if with_smat is None else with_smat:
            m = np.array([[rng.choice([0.25, 0.5, 1.0, 1.5, 2.0]) for _ in range(n)] for _ in range(n)])
            smat = np.triu(m) + np.triu(m, 1).T
        stems = O.annotate(p.shortseq, ps, p.shortreacts, p.shortrest, smat=smat)
        out.append((p.shortseq, stems))
    return out


def synthetic_cases(seed, count, lo=0, hi=60):
    """hand-shaped stem lists: few distinct scores (zero among them), stems at position 0 and N-1, separators,
    overlapping stems that share pairs with other scores (the later stem wins), empty lists"""
    rng = random.Random(seed)
    out = []
    for c in range(count):
        n = rng.randint(lo, hi)
        sep_p = rng.choice([0.0, 0.05, 0.3])
        seq = "".join(";" if rng.random() < sep_p / 2 else "&" if rng.random() < sep_p / 2 else rng.choice("ACGU")
                      for _ in range(n))
        scores = rng.choice([[3.0], [0.0, 2.0], [0.25, 0.5, 0.75, 1.0], [1.0, 2.0, 3.25, 6.5], [0.0]])
        stems = []
        for _ in range(0 if n < 2 or c % 11 == 0 else rng.randint(1, 3 * n)):
            i = rng.choice([0, rng.randrange(n - 1)])
            j = rng.choice([n - 1, rng.randrange(i + 1, n)])
            if j <= i:
                continue
            ln = rng.randint(1, max(1, min(6, (j - i + 1) // 2)))
            stems.append((i, j, ln, rng.choice(scores)))
            if rng.random() < 0.3:                         # the same pairs again, shifted by one, another score
                stems.append((i, j, ln, rng.choice(scores)))
        out.append((seq, stems))
    return out


def lsap_matrices(seed, count, lo=0, hi=300):
    """symmetric sparse cost matrices with heavy ties: (n, [(v, w, cost)]), cost -(0.25 k) ** 1.7 for a few small k
    (k = 0 gives -0.0), duplicated weights everywhere"""
    rng = random.Random(seed)
    out = []
    for _ in range(count):
        n = rng.randint(lo, hi) if rng.random() < 0.7 else rng.randint(lo, min(hi, 20))
        ks = rng.sample(range(0, 12), rng.randint(1, 4))
        dens = rng.choice([0.02, 0.1, 0.3, 0.8])
        ent = {}
        for v in range(n):
            for w in range(v + 1, n):
                if rng.random() < dens:
                    ent[(v, w)] = -((0.25 * rng.choice(ks)) ** 1.7)
        out.append((n, [(v, w, c) for (v, w), c in ent.items()]))
    return out


def _check(cases, got, label, want=None, **kw):
    want = want if want is not None else [host_hungarian(seq, stems, **kw) for seq, stems in cases]
    bad = [(seq, stems, g) for (seq, stems), g, w in zip(cases, got, want) if g != w]
    assert not bad, "%s: %d of %d differ; first: %r" % (label, len(bad), len(cases), bad[0][:1])


# ---------------------------------------------------------------- CPU: the emulated device code
def test_emulated_assignment_matches_scipy():
    for n, ent in lsap_matrices(1, 300) + [(0, []), (1, []), (2, []), (2, [(0, 1, -1.0)]), (2, [(0, 1, -0.0)])]:
        cost = np.zeros((n, n))
        for v, w, c in ent:
            cost[v, w] = cost[w, v] = c
        want = linear_sum_assignment(cost)[1].tolist()
        for width in WIDTHS:
            assert emu_lsap(n, ent, width) == want, (n, width, ent)


def _emu_all_widths(cases, label, **kw):
    seqs, stems = [c[0] for c in cases], [c[1] for c in cases]
    want = [host_hungarian(seq, st, **kw) for seq, st in cases]
    for width in WIDTHS:
        _check(cases, emu_hungarian(seqs, stems, width, **kw), "%s width %d" % (label, width), want)


def test_emulated_builder_on_annotated_stems():
    _emu_all_widths(annotated_cases(2, 120, 1, 150), "1-150 nt")
    _emu_all_widths(annotated_cases(3, 8, 150, 400), "150-400 nt")


def test_emulated_builder_on_synthetic_stems():
    _emu_all_widths(synthetic_cases(4, 400) + [("", []), ("A", []), ("AC", []), ("AC", [(0, 1, 1, 2.0)]),
                                               ("AC", [(0, 1, 1, 0.0)])], "synthetic")


def test_emulated_builder_other_minloop_and_power():
    cases = synthetic_cases(5, 150, 2, 40) + annotated_cases(6, 20, 10, 80)
    for ml in (0, 1, 2, 4, 5):
        _emu_all_widths(cases, "minloop %d" % ml, minloop=ml)
    _emu_all_widths(cases, "power 1", power=1.0)


def test_emulated_builder_rejects_bad_input():
    for stem in ((0, 5, 1, 1.0), (-1, 3, 1, 1.0), (0, 4, 0, 1.0), (3, 4, 3, 1.0), (2, 4, 4, 1.0), (3, 3, 1, 1.0),
                 (4, 2, 1, 1.0), (1, 4, 3, 1.0)):
        assert emu_hungarian(["ACGUA"], [[stem]]) == E_BADARG, stem
    assert emu_hungarian(["ACGUACGU"], [[(0, 7, 1, 1.0)]], minloop=-1) == E_BADARG
    assert emu_hungarian(["A" * (MAX_LEN + 1)], [[]]) == E_BADARG
    for score, power in ((-1.0, 1.7), (math.nan, 1.7), (math.inf, 1.7), (1e300, 1.7), (0.0, -1.0), (2.0, math.nan)):
        assert emu_hungarian(["ACGUACGU"], [[(0, 7, 1, score)]], power=power) == E_BADARG, (score, power)
    # what is allowed: a zero score (cost -0.0, never kept), score 1 with a NaN power (1 ** nan == 1)
    assert emu_hungarian(["ACGUACGU"], [[(0, 7, 1, 0.0)]]) == [[]]
    assert emu_hungarian(["ACGUACGU"], [[(0, 7, 1, 1.0)]], power=math.nan) == [[(0, 7)]]


def test_smem_tier_limit_follows_the_layout():
    L = _emu()
    assert L.emu_hu_smem_max_n(227 * 1024) == 5528            # a B200's opt-in shared memory per block
    assert L.emu_hu_smem_max_n(48 * 1024) < L.emu_hu_smem_max_n(227 * 1024)


# ---------------------------------------------------------------- GPU: the C entry
def _threshold():
    import torch
    return _emu().emu_hu_smem_max_n(torch.cuda.get_device_properties(0).shared_memory_per_block_optin)


def _device_stems(ctx, seqs, ps):
    from squarna_b200._lib import PackedBatch
    return [[(i, j, ln, s_) for (i, j, ln), s_ in zip(st.tolist(), sc.tolist())]
            for st, sc in ctx.yield_stems(ps, PackedBatch([s.encode() for s in seqs]))]


@pytest.mark.gpu
def test_device_builder_matches_the_host_builder(gpu_ctx):
    for label, cases in (("annotated 1-150", annotated_cases(11, 500, 1, 150)),
                         ("annotated 150-700", annotated_cases(12, 40, 150, 700)),
                         ("synthetic", synthetic_cases(13, 500, 0, 300))):
        got = device_hungarian(gpu_ctx, [c[0] for c in cases], [c[1] for c in cases])
        _check(cases, got, label)
    cases = synthetic_cases(14, 100, 2, 60)
    for ml in (0, 5):
        _check(cases, device_hungarian(gpu_ctx, [c[0] for c in cases], [c[1] for c in cases], minloop=ml),
               "minloop %d" % ml, minloop=ml)


@pytest.mark.gpu
def test_device_builder_across_the_tier_thresholds(gpu_ctx):
    thr = _threshold()
    rng = random.Random(15)
    ps = _conf("hungariannobpp")[0]
    for ls, launches in (([255, 256], 1), ([256, 257], 2), ([257, 300], 1), ([thr - 1, thr], 1), ([thr, thr + 1], 2),
                         ([thr + 1], 1), ([100, 700, thr + 1], 3)):
        sq = [T.rand_seq(rng, n) for n in ls]
        st = _device_stems(gpu_ctx, sq, ps)
        got = device_hungarian(gpu_ctx, sq, st)
        assert gpu_ctx.stats()["launches"] == launches, ls
        assert got == [host_hungarian(a, b) for a, b in zip(sq, st)], ls


@pytest.mark.gpu
def test_device_builder_on_long_sequences(gpu_ctx):
    rng = random.Random(16)
    ps = _conf("hungariannobpp")[0]
    seqs = [T.rand_seq(rng, n) for n in (3000, 5000)]
    stems = _device_stems(gpu_ctx, seqs, ps)
    got = device_hungarian(gpu_ctx, seqs, stems)
    _check(list(zip(seqs, stems)), got, "3000 / 5000 nt")
    assert all(len(g) > 100 for g in got)
    # 12 000 nt: 1.1 GB as a dense host matrix; against the emulator.  The stems come from the oracle's AnnotateStems:
    # the device's stem enumeration keeps a sequence in one CTA's shared memory, which does not hold 12 000 nt
    seqs = [T.rand_seq(rng, 12000)]
    stems = [O.annotate(seqs[0], ps)]
    got = device_hungarian(gpu_ctx, seqs, stems)
    assert got == emu_hungarian(seqs, stems, 256) and len(got[0]) > 500


@pytest.mark.gpu
def test_device_builder_rejects_bad_input(gpu_ctx):
    from squarna_b200._lib import SqrnError
    for stem in ((0, 5, 1, 1.0), (-1, 3, 1, 1.0), (0, 4, 0, 1.0), (3, 4, 3, 1.0), (2, 2, 1, 1.0), (1, 4, 3, 1.0),
                 (0, 4, 1, -1.0), (0, 4, 1, math.nan), (0, 4, 1, 1e300)):
        with pytest.raises(SqrnError) as e:
            device_hungarian(gpu_ctx, ["ACGUA"], [[stem]])
        assert e.value.code == E_BADARG, stem
    with pytest.raises(SqrnError):
        device_hungarian(gpu_ctx, ["ACGUACGU"], [[(0, 7, 1, 1.0)]], minloop=-1)
    with pytest.raises(SqrnError):
        device_hungarian(gpu_ctx, ["A" * (MAX_LEN + 1)], [[]])
    assert device_hungarian(gpu_ctx, ["", "A", "AC", "ACGUACGU"], [[], [], [], []]) == [[], [], [], []]


class _HostBuilderContext:
    """the library context without `hungarian`: _predict_many_mixed then runs SQRNalgos.Hungarian on the host
    (Nussinov stays on the device)"""

    def __init__(self, ctx):
        self._ctx = ctx

    def yield_stems(self, *a, **k):
        return self._ctx.yield_stems(*a, **k)

    def predict_batch(self, *a, **k):
        return self._ctx.predict_batch(*a, **k)

    def predict_batch_flat(self, *a, **k):
        return self._ctx.predict_batch_flat(*a, **k)

    def nussinov(self, *a, **k):
        return self._ctx.nussinov(*a, **k)


@pytest.mark.gpu
@pytest.mark.parametrize("conf,lens", [("hungariannobpp", (120, 300, 640, 1000, 1500)), ("nobpp", (90, 300, 420))])
def test_predict_many_with_the_device_builder(gpu_ctx, monkeypatch, conf, lens):
    rng = random.Random(17)
    entries = []
    for n in lens:
        seq, reacts, rest, _kw = T.rand_case(rng, n, n, p_gap=0.0)
        entries.append((seq, reacts, rest, None))
    dev = S.predict_many(entries, _conf(conf), device=0)
    host_ctx = _HostBuilderContext(S.get_context(0))
    monkeypatch.setattr(S, "get_context", lambda device=0: host_ctx)
    host = S.predict_many(entries, _conf(conf), device=0)
    assert len(dev) == len(host)
    for a, b in zip(dev, host):
        assert T.same_prediction(a[:2], b[:2])


@pytest.mark.gpu
def test_cli_hungarian_text_with_the_device_builder(gpu_ctx, monkeypatch, tmp_path):
    from squarna_b200 import SQUARNA as CLI
    rng = random.Random(18)
    lines = []
    for k in range(12):
        lines += [">e%d" % k, T.rand_seq(rng, rng.randint(40, 400))]
    path = tmp_path / "multi.fas"
    path.write_text("\n".join(lines) + "\n")
    out = []
    for host in (False, True):
        if host:
            host_ctx = _HostBuilderContext(S.get_context(0))
            monkeypatch.setattr(S, "get_context", lambda device=0: host_ctx)
        buf = io.StringIO()
        with contextlib.redirect_stdout(buf):
            CLI.Main(["i=" + str(path), "c=hungariannobpp", "t=1"])
        out.append(buf.getvalue())
    assert out[0] == out[1] and out[0].count(">e") == 12
