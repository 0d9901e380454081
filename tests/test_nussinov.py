"""The Nussinov builder on the device (include/sqrn.h: sqrn_nussinov_batch, csrc/sqrn_nussinov.cuh) against the host
restatement squarna_b200/SQRNalgos.Nussinov, pair for pair.

Without a GPU the DP step and the backtrack run through tests/emu/nussinov_emu.cpp, the single-thread host build of
the same header, for both tiers (the global tier also with a few candidates per pass, so a column takes several).
With -m gpu the C entry runs on the device: against the host builder up to 1500 nt, against the emulator at 3000 -
8000 nt, and end to end through predict_many / the CLI against the same calls through a context without the builder."""
import contextlib
import ctypes as C
import io
import os
import random
import subprocess

import numpy as np
import pytest

from oracle import oracle as O
from squarna_b200 import SQRNalgos, SQRNdbnseq as S
from squarna_b200._abi import E_BADARG, OK, pack_sequences
from tests import common as T

_HERE = os.path.dirname(os.path.abspath(__file__))
_ROOT = os.path.dirname(_HERE)
_CSRC = os.path.join(_ROOT, "squarna_b200", "csrc")
_EMU_SRC = [os.path.join(_HERE, "emu", "nussinov_emu.cpp")] + \
    [os.path.join(_CSRC, f) for f in ("sqrn_nussinov.cuh", "sqrn_device.cuh", "sqrn_params.h")]
_EMU_SO = os.path.join(_HERE, "emu", "_build", "libnussinov_emu.so")
SEPS = S.SEPS
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
        L.emu_nu_smem_max_n.argtypes = [C.c_longlong]
        L.emu_nussinov.argtypes = [C.c_int64] + [C.c_void_p] * 5 + [C.c_int] * 3 + [C.c_void_p] * 2
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


def emu_nussinov(seqs, stem_lists, tier=0, chunk=1024, minloop=3):
    """pairs per sequence from the emulated device code, as lists of (v, w); or the error code"""
    sym, off, so, st, sc = _flat(seqs, stem_lists)
    po = np.zeros(len(seqs) + 1, np.int64)
    pairs = np.zeros((max(int((np.diff(off) // 2).sum()), 1), 2), np.int32)
    rc = _emu().emu_nussinov(len(seqs), _ptr(off), _ptr(sym), _ptr(so), _ptr(st), _ptr(sc), minloop, tier, chunk,
                             _ptr(po), _ptr(pairs))
    if rc != OK:
        return rc
    return [[tuple(p) for p in pairs[po[b]:po[b + 1]].tolist()] for b in range(len(seqs))]


def device_nussinov(ctx, seqs, stem_lists, minloop=3):
    sym, off, so, st, sc = _flat(seqs, stem_lists)
    per = [(st[so[b]:so[b + 1]], sc[so[b]:so[b + 1]]) for b in range(len(seqs))]
    return [[tuple(p) for p in x.tolist()] for x in ctx.nussinov(sym, off, per, minloop=minloop)]


def host_nussinov(seq, stems, minloop=3):
    lists = [[[(i + t, j - t) for t in range(ln)], ln, sc] for i, j, ln, sc in stems]
    return SQRNalgos.Nussinov(seq, lists, len(seq), SEPS, minloop=minloop)


# ---------------------------------------------------------------- generators
def _conf_sets():
    """the N-running parameter sets (defN, bppN, ...) of every shipped configuration, by name"""
    from squarna_b200 import SQUARNA as CLI
    pkg = os.path.dirname(os.path.abspath(CLI.__file__))
    out = {}
    for f in sorted(os.listdir(pkg)):
        if f.endswith(".conf"):
            names, sets = CLI.ParseConfig(os.path.join(pkg, f))
            for nm, ps in zip(names, sets):
                if "N" in ps["algorithms"]:
                    out.setdefault((nm, tuple(sorted(ps["bpweights"].items())), ps["minlen"], ps["minbpscore"]), ps)
    return list(out.values())


def _rand_paramset(rng):
    w = {k: rng.choice([-1.5, -1.0, 0.0, 0.5, 1.0, 1.25, 2.0, 3.25, 3.5]) for k in ("GC", "AU", "GU")}
    if rng.random() < 0.3:
        w["GA"] = rng.choice([0.5, 1.0])
    return T._ps(algorithms={"N"}, bpweights=w, minlen=float(rng.choice([1, 2, 3, 4])),
                 minbpscore=rng.choice([0.0, 1.0, 2.75, 4.5, 6.0]))


def annotated_cases(seed, count, lo, hi, with_smat=None):
    """(shortseq, stems) of random SQRNdbnseq inputs (separators, restraints, reactivities, gaps) under the N-running
    sets of the shipped configurations and random parameter sets, half of them with a stem matrix"""
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
    """hand-shaped stem lists: equal / zero / negative scores, stems at position 0 and N-1, separators next to the
    hairpin boundary, pairs two stems share, degenerate stems whose pairs cross, empty lists"""
    rng = random.Random(seed)
    out = []
    for c in range(count):
        n = rng.randint(lo, hi)
        sep_p = rng.choice([0.0, 0.05, 0.3])
        seq = "".join(";" if rng.random() < sep_p / 2 else "&" if rng.random() < sep_p / 2 else rng.choice("ACGU")
                      for _ in range(n))
        scores = rng.choice([[3.0], [0.0, -1.0, 2.0], [-2.0, -0.5], [0.25, 0.5, 0.75, 1.0], [1.0, 2.0, 3.25, 6.5]])
        stems = []
        for _ in range(0 if n < 2 or c % 11 == 0 else rng.randint(1, 3 * n)):
            i = rng.choice([0, rng.randrange(n)])
            j = rng.choice([n - 1, rng.randrange(n)])
            if i > j:
                i, j = j, i
            ln = rng.randint(1, max(1, min(n - i, j + 1, 6)))
            stems.append((i, j, ln, rng.choice(scores)))
        out.append((seq, stems))
    return out


def all_pairs_cases():
    """every pair of a short sequence possible, all with the same score (ties everywhere), one separator anywhere"""
    out = []
    for n in range(2, 14):
        for sep_at in range(n):
            seq = "".join("&" if k == sep_at else "G" if k < n // 2 else "C" for k in range(n))
            stems = [(i, j, 1, 3.0) for i in range(n) for j in range(i + 1, n)]
            out.append((seq, stems))
    return out


def boundary_cases(seed=7, count=4000):
    """separators next to BackTrack's hairpin boundary: 4-12 positions, 40 % of them separators, 1-8 single-pair stems
    with scores in {-1, 0, 1, 2}, so the walk reaches short unpaired intervals (left of a pair, inside it, and j left
    unpaired) that begin or end next to a separator, where `gap > minloop or (gap > 0 and a separator in ...)` flips"""
    rng = random.Random(seed)
    out = []
    for _ in range(count):
        n = rng.randint(4, 12)
        seq = "".join(rng.choice(";&") if rng.random() < 0.4 else rng.choice("ACGU") for _ in range(n))
        stems = []
        for _ in range(rng.randint(1, 8)):
            i, j = sorted(rng.sample(range(n), 2))
            stems.append((i, j, 1, float(rng.choice([-1, 0, 1, 2]))))
        out.append((seq, stems))
    return out


def _check(cases, got, label, want=None):
    want = want if want is not None else [host_nussinov(seq, stems) for seq, stems in cases]
    bad = [(seq, stems, g) for (seq, stems), g, w in zip(cases, got, want) if g != w]
    assert not bad, "%s: %d of %d differ; first: %r" % (label, len(bad), len(cases), bad[0][:1])


# ---------------------------------------------------------------- CPU: the emulated device code
def _emu_all_tiers(cases, label):
    seqs, stems = [c[0] for c in cases], [c[1] for c in cases]
    want = [host_nussinov(seq, st) for seq, st in cases]
    for tier, chunk in ((0, 1024), (1, 1024), (1, 3)):
        _check(cases, emu_nussinov(seqs, stems, tier, chunk), "%s tier %d chunk %d" % (label, tier, chunk), want)


def test_emulated_builder_on_annotated_stems():
    _emu_all_tiers(annotated_cases(1, 160, 1, 120), "1-120 nt")
    _emu_all_tiers(annotated_cases(2, 14, 120, 320), "120-320 nt")
    _emu_all_tiers(annotated_cases(3, 2, 600, 700, with_smat=False) + annotated_cases(4, 1, 600, 700, with_smat=True),
                   "600-700 nt")


def test_emulated_builder_on_synthetic_stems():
    _emu_all_tiers(synthetic_cases(5, 400) + all_pairs_cases() + boundary_cases() + [("", []), ("A", []), ("AC", [(0, 1, 1, 2.0)])],
                   "synthetic")


def test_emulated_builder_other_minloop():
    cases = synthetic_cases(6, 150, 2, 40) + boundary_cases(9, 1000)
    for ml in (0, 1, 5):
        got = emu_nussinov([c[0] for c in cases], [c[1] for c in cases], 1, 2, minloop=ml)
        assert got == [host_nussinov(s, st, minloop=ml) for s, st in cases], ml


def test_emulated_builder_rejects_malformed_stems():
    for stem in ((0, 5, 1, 1.0), (-1, 3, 1, 1.0), (0, 4, 0, 1.0), (3, 4, 3, 1.0), (2, 4, 4, 1.0)):
        assert emu_nussinov(["ACGUA"], [[stem]]) == E_BADARG, stem
    assert emu_nussinov(["ACGUACGU"], [[(0, 7, 1, 1.0)]], minloop=-1) == E_BADARG


def test_smem_tier_limit_follows_the_layout():
    L = _emu()
    assert L.emu_nu_smem_max_n(227 * 1024) == 238            # a B200's opt-in shared memory per block
    assert L.emu_nu_smem_max_n(48 * 1024) < L.emu_nu_smem_max_n(227 * 1024)


# ---------------------------------------------------------------- GPU: the C entry
def _threshold():
    import torch
    return _emu().emu_nu_smem_max_n(torch.cuda.get_device_properties(0).shared_memory_per_block_optin)


@pytest.mark.gpu
def test_device_builder_matches_the_host_builder(gpu_ctx):
    for label, cases in (("annotated 1-120", annotated_cases(11, 300, 1, 120)),
                         ("annotated 120-700", annotated_cases(12, 24, 120, 700)),
                         ("synthetic", synthetic_cases(13, 600) + all_pairs_cases() + boundary_cases(8))):
        got = device_nussinov(gpu_ctx, [c[0] for c in cases], [c[1] for c in cases])
        _check(cases, got, label)


def _device_stems(ctx, seqs, ps):
    from squarna_b200._lib import PackedBatch
    return [[(i, j, ln, s_) for (i, j, ln), s_ in zip(st.tolist(), sc.tolist())]
            for st, sc in ctx.yield_stems(ps, PackedBatch([s.encode() for s in seqs]))]


@pytest.mark.gpu
def test_device_builder_across_the_tier_threshold(gpu_ctx):
    thr = _threshold()
    rng = random.Random(14)
    ps = _conf_sets()[0]
    lens = [thr - 1, thr, thr + 1] * 2 + [rng.randint(30, thr) for _ in range(20)] + [900, 1500]
    seqs = [T.rand_seq(rng, n) for n in lens]
    stems = _device_stems(gpu_ctx, seqs, ps)
    got = device_nussinov(gpu_ctx, seqs, stems)
    assert gpu_ctx.stats()["launches"] == 2
    _check(list(zip(seqs, stems)), got, "mixed lengths")
    # the split is at the threshold: one launch for each side of it, two when the batch straddles it
    for ls, launches in (([thr - 1, thr], 1), ([thr, thr + 1], 2), ([thr + 1, thr + 2], 1)):
        sq = [T.rand_seq(rng, n) for n in ls]
        st = _device_stems(gpu_ctx, sq, ps)
        assert device_nussinov(gpu_ctx, sq, st) == [host_nussinov(a, b) for a, b in zip(sq, st)]
        assert gpu_ctx.stats()["launches"] == launches, ls


@pytest.mark.gpu
def test_device_builder_matches_the_emulator_on_long_sequences(gpu_ctx):
    rng = random.Random(15)
    ps = _conf_sets()[0]
    seqs = [T.rand_seq(rng, n) for n in (3000, 5000, 8000)]
    stems = _device_stems(gpu_ctx, seqs, ps)
    got = device_nussinov(gpu_ctx, seqs, stems)
    assert got == emu_nussinov(seqs, stems, 1)
    assert all(len(g) > 100 for g in got)


@pytest.mark.gpu
def test_device_builder_rejects_malformed_stems(gpu_ctx):
    from squarna_b200._lib import SqrnError
    for stem in ((0, 5, 1, 1.0), (-1, 3, 1, 1.0), (0, 4, 0, 1.0), (3, 4, 3, 1.0)):
        with pytest.raises(SqrnError):
            device_nussinov(gpu_ctx, ["ACGUA"], [[stem]])
    assert device_nussinov(gpu_ctx, ["", "A", "ACGUACGU"], [[], [], []]) == [[], [], []]


class _HostBuilderContext:
    """the library context without `nussinov`: _predict_many_mixed then runs SQRNalgos.Nussinov on the host"""

    def __init__(self, ctx):
        self._ctx = ctx

    def yield_stems(self, *a, **k):
        return self._ctx.yield_stems(*a, **k)

    def predict_batch(self, *a, **k):
        return self._ctx.predict_batch(*a, **k)

    def predict_batch_flat(self, *a, **k):
        return self._ctx.predict_batch_flat(*a, **k)


def _conf(name):
    from squarna_b200 import SQUARNA as CLI
    return CLI.ParseConfig(os.path.join(os.path.dirname(os.path.abspath(CLI.__file__)), name + ".conf"))[1]


@pytest.mark.gpu
@pytest.mark.parametrize("conf,lens", [("nussinovnobpp", (300, 640, 1000, 1500)), ("nobpp", (300, 420))])
def test_predict_many_with_the_device_builder(gpu_ctx, monkeypatch, conf, lens):
    rng = random.Random(16)
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
def test_cli_nussinov_text_with_the_device_builder(gpu_ctx, monkeypatch, tmp_path):
    from squarna_b200 import SQUARNA as CLI
    rng = random.Random(17)
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
            CLI.Main(["i=" + str(path), "c=nussinovnobpp", "t=1"])
        out.append(buf.getvalue())
    assert out[0] == out[1] and out[0].count(">e") == 12
