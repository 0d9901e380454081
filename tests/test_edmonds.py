"""The Edmonds builder on the device (include/sqrn.h: sqrn_edmonds_batch, csrc/sqrn_edmonds.cuh) against NetworkX's
max_weight_matching and the host restatement squarna_b200/SQRNalgos.Edmonds, pair for pair.

Without a GPU the matching runs through tests/emu/edmonds_emu.cpp, the host build of the same header, with the delta
minima split over simulated teams of 1, 32 (the warp tier) and 256 lanes (the CTA and global tiers) whose partial keys
meet as on the device.  With -m gpu the C entry runs on the device: against the host builder up to 1 000 nt, across the
tier thresholds, against the emulator at 3 000 and 5 000 nt (stems of a strict parameter set), and end to end through predict_many / the CLI against
the same calls through a context without the builder."""
import contextlib
import ctypes as C
import io
import math
import os
import random
import subprocess

import networkx as nx
import numpy as np
import pytest

from oracle import oracle as O
from squarna_b200 import SQRNalgos, SQRNdbnseq as S
from squarna_b200._abi import E_BADARG, OK
from tests import common as T
from tests.test_hungarian import _conf, _flat, _ptr, synthetic_cases

_HERE = os.path.dirname(os.path.abspath(__file__))
_CSRC = os.path.join(os.path.dirname(_HERE), "squarna_b200", "csrc")
_EMU_SRC = [os.path.join(_HERE, "emu", "edmonds_emu.cpp")] + \
    [os.path.join(_CSRC, f) for f in ("sqrn_edmonds.cuh", "sqrn_hungarian.cuh", "sqrn_nussinov.cuh", "sqrn_device.cuh",
                                      "sqrn_params.h")]
_EMU_SO = os.path.join(_HERE, "emu", "_build", "libedmonds_emu.so")
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
        L.emu_ed_smem_max_n.argtypes = [C.c_longlong]
        L.emu_matching.argtypes = [C.c_int, C.c_int64, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p]
        L.emu_edmonds.argtypes = [C.c_int64] + [C.c_void_p] * 4 + [C.c_double, C.c_int] + [C.c_void_p] * 2
        _emu_lib = L
    return _emu_lib


def emu_matching(edges, weights, width):
    """the emulated matching of the graph with `edges` (any hashable labels) added in this order, as sorted pairs"""
    ids = {}
    for e in edges:
        for x in e:
            ids.setdefault(x, len(ids))
    nodes = list(ids)
    ends = np.array([ids[x] for e in edges for x in e] or [0], np.int32)
    wt = np.array(list(weights) or [0.0], np.float64)
    out = np.zeros((len(ids) // 2 + 1, 2), np.int32)
    n = _emu().emu_matching(len(ids), len(edges), _ptr(ends), _ptr(wt), width, _ptr(out))
    assert n >= 0, n
    return sorted(tuple(sorted((nodes[a], nodes[b]))) for a, b in out[:n].tolist())


def nx_matching(edges, weights):
    g = nx.Graph()
    g.add_weighted_edges_from([(v, w, x) for (v, w), x in zip(edges, weights)])
    return sorted(tuple(sorted(p)) for p in nx.max_weight_matching(g))


def emu_edmonds(seqs, stem_lists, width=256, power=1.7):
    """pairs per sequence from the emulated device code, as lists of (v, w); or the error code"""
    _sym, off, so, st, sc = _flat(seqs, stem_lists)
    po = np.zeros(len(seqs) + 1, np.int64)
    pairs = np.zeros((max(int((np.diff(off) // 2).sum()), 1), 2), np.int32)
    rc = _emu().emu_edmonds(len(seqs), _ptr(off), _ptr(so), _ptr(st), _ptr(sc), power, width, _ptr(po), _ptr(pairs))
    if rc != OK:
        return rc
    return [[tuple(p) for p in pairs[po[b]:po[b + 1]].tolist()] for b in range(len(seqs))]


def device_edmonds(ctx, seqs, stem_lists, power=1.7):
    sym, off, so, st, sc = _flat(seqs, stem_lists)
    per = [(st[so[b]:so[b + 1]], sc[so[b]:so[b + 1]]) for b in range(len(seqs))]
    return [[tuple(p) for p in x.tolist()] for x in ctx.edmonds(sym, off, per, power=power)]


def host_edmonds(stems, power=1.7):
    """SQRNalgos.Edmonds, normalised as RunAlgo reads it"""
    lists = [[[(i + t, j - t) for t in range(ln)], ln, sc] for i, j, ln, sc in stems]
    return sorted((min(v, w), max(v, w)) for v, w in SQRNalgos.Edmonds(lists, power=power))


# ---------------------------------------------------------------- generators
def _conf_sets():
    """the E-running parameter sets of every shipped configuration"""
    from squarna_b200 import SQUARNA as CLI
    pkg = os.path.dirname(os.path.abspath(CLI.__file__))
    out = {}
    for f in sorted(os.listdir(pkg)):
        if f.endswith(".conf"):
            names, sets = CLI.ParseConfig(os.path.join(pkg, f))
            for nm, ps in zip(names, sets):
                if "E" in ps["algorithms"]:
                    out.setdefault((nm, tuple(sorted(ps["bpweights"].items())), ps["minlen"], ps["minbpscore"]), ps)
    return list(out.values())


def _rand_paramset(rng):
    w = {k: rng.choice([0.0, 0.5, 1.0, 1.25, 2.0, 3.25, 3.5]) for k in ("GC", "AU", "GU")}
    if rng.random() < 0.3:
        w["GA"] = rng.choice([0.5, 1.0])
    return T._ps(algorithms={"E"}, bpweights=w, minlen=float(rng.choice([1, 2, 3, 4])),
                 minbpscore=rng.choice([0.0, 0.0, 1.0, 2.75, 4.5, 6.0]))


def annotated_cases(seed, count, lo, hi):
    """(shortseq, stems) of random SQRNdbnseq inputs (separators, restraints, reactivities, gaps) under the E-running
    sets of the shipped configurations and random parameter sets (minbpscore 0 among them)"""
    rng = random.Random(seed)
    sets = _conf_sets()
    out = []
    for _ in range(count):
        seq, reacts, rest, _kw = T.rand_case(rng, lo, hi)
        p = S._prepare(seq, reacts, rest, None)
        ps = rng.choice(sets) if rng.random() < 0.6 else _rand_paramset(rng)
        out.append((p.shortseq, O.annotate(p.shortseq, ps, p.shortreacts, p.shortrest)))
    return out


def tie_graphs(seed, count, hi=80):
    """(edges in insertion order, weights): weights (0.25 k) ** 1.7 from a few k (0 among them), dense, sparse and
    disconnected graphs, node labels inserted out of numeric order, some graphs of zero weights only"""
    rng = random.Random(seed)
    out = []
    for c in range(count):
        n = rng.randint(2, hi)
        dens = rng.choice([0.03, 0.1, 0.3, 0.8])
        ks = rng.sample(range(0, 12), rng.randint(1, 4))
        perm = list(range(n))
        rng.shuffle(perm)
        parts = rng.choice([1, 1, 2, 3])                 # disconnected: no edge across parts
        part = {v: rng.randrange(parts) for v in range(n)}
        ent = {}
        for v in range(n):
            for w in range(v + 1, n):
                if part[v] == part[w] and rng.random() < dens:
                    ent[(perm[v], perm[w])] = (0.25 * rng.choice(ks)) ** 1.7
        edges = list(ent)
        rng.shuffle(edges)
        weights = [0.0] * len(edges) if c % 13 == 0 else [ent[e] for e in edges]
        out.append((edges, weights))
    return out + [([(5, 3)], [2.0]), ([(1, 0)], [0.0]), ([], [])]


def overlapping_cases(seed, count, hi=60):
    """stem lists whose stems hold the same pairs again with other scores: the edge keeps its first place and takes
    the last score"""
    rng = random.Random(seed)
    out = []
    for _ in range(count):
        n = rng.randint(4, hi)
        seq = "".join(rng.choice("ACGU") for _ in range(n))
        stems = []
        for _ in range(rng.randint(1, 2 * n)):
            i = rng.randrange(n - 3)
            j = rng.randrange(i + 3, n)
            ln = rng.randint(1, max(1, (j - i + 1) // 2))
            stems.append((i, j, ln, rng.choice([0.0, 0.25, 1.0, 2.0, 3.25])))
            if rng.random() < 0.5:                       # a later stem inside it: same pairs, another score
                t = rng.randrange(ln)
                stems.append((i + t, j - t, rng.randint(1, ln - t), rng.choice([0.0, 0.25, 1.0, 2.0, 3.25])))
        out.append((seq, stems))
    return out


def _check(cases, got, label, want=None, **kw):
    want = want if want is not None else [host_edmonds(stems, **kw) for _seq, stems in cases]
    bad = [(seq, stems, g) for (seq, stems), g, w in zip(cases, got, want) if g != w]
    assert not bad, "%s: %d of %d differ; first: %r" % (label, len(bad), len(cases), bad[0][:1])


# ---------------------------------------------------------------- CPU: the emulated device code
def test_emulated_matching_matches_networkx():
    for edges, weights in tie_graphs(1, 300):
        want = nx_matching(edges, weights)
        for width in WIDTHS:
            assert emu_matching(edges, weights, width) == want, (width, edges, weights)


def _emu_all_widths(cases, label, **kw):
    seqs, stems = [c[0] for c in cases], [c[1] for c in cases]
    want = [host_edmonds(st, **kw) for _seq, st in cases]
    for width in WIDTHS:
        _check(cases, emu_edmonds(seqs, stems, width, **kw), "%s width %d" % (label, width), want)


def test_emulated_builder_on_annotated_stems():
    _emu_all_widths(annotated_cases(2, 120, 1, 150), "1-150 nt")
    _emu_all_widths(annotated_cases(3, 4, 150, 300), "150-300 nt")


def test_emulated_builder_on_synthetic_stems():
    _emu_all_widths(synthetic_cases(4, 300) + overlapping_cases(5, 150) +
                    [("", []), ("A", []), ("AC", []), ("AC", [(0, 1, 1, 2.0)]), ("AC", [(0, 1, 1, 0.0)])], "synthetic")


def test_emulated_builder_power_one():
    _emu_all_widths(overlapping_cases(6, 60) + annotated_cases(7, 20, 10, 80), "power 1", power=1.0)


def test_emulated_builder_rejects_bad_input():
    for stem in ((0, 5, 1, 1.0), (-1, 3, 1, 1.0), (0, 4, 0, 1.0), (3, 4, 3, 1.0), (2, 4, 4, 1.0), (3, 3, 1, 1.0),
                 (4, 2, 1, 1.0), (1, 4, 3, 1.0)):
        assert emu_edmonds(["ACGUA"], [[stem]]) == E_BADARG, stem
    assert emu_edmonds(["A" * (MAX_LEN + 1)], [[]]) == E_BADARG
    for score, power in ((-1.0, 1.7), (math.nan, 1.7), (math.inf, 1.7), (1e300, 1.7), (0.0, -1.0), (2.0, math.nan),
                         (1e308, 1.0)):
        assert emu_edmonds(["ACGUACGU"], [[(0, 7, 1, score)]], power=power) == E_BADARG, (score, power)
    # what is allowed: a zero score (a zero-weight edge, matched), score 1 with a NaN power (1 ** nan == 1)
    assert emu_edmonds(["ACGUACGU"], [[(0, 7, 1, 0.0)]]) == [[(0, 7)]] == [host_edmonds([(0, 7, 1, 0.0)])]
    assert emu_edmonds(["ACGUACGU"], [[(0, 7, 1, 1.0)]], power=math.nan) == [[(0, 7)]]


def test_smem_tier_limit_follows_the_layout():
    L = _emu()
    assert L.emu_ed_smem_max_n(227 * 1024) == 1933            # a B200's opt-in shared memory per block
    assert L.emu_ed_smem_max_n(48 * 1024) < L.emu_ed_smem_max_n(227 * 1024)


# ---------------------------------------------------------------- GPU: the C entry
def _threshold():
    import torch
    return _emu().emu_ed_smem_max_n(torch.cuda.get_device_properties(0).shared_memory_per_block_optin)


def _device_stems(ctx, seqs, ps):
    from squarna_b200._lib import PackedBatch
    return [[(i, j, ln, s_) for (i, j, ln), s_ in zip(st.tolist(), sc.tolist())]
            for st, sc in ctx.yield_stems(ps, PackedBatch([s.encode() for s in seqs]))]


@pytest.mark.gpu
def test_device_builder_matches_the_host_builder(gpu_ctx):
    for label, cases in (("annotated 1-150", annotated_cases(11, 500, 1, 150)),
                         ("annotated 150-500", annotated_cases(12, 30, 150, 500)),
                         ("synthetic", synthetic_cases(13, 400, 0, 300) + overlapping_cases(14, 100))):
        got = device_edmonds(gpu_ctx, [c[0] for c in cases], [c[1] for c in cases])
        _check(cases, got, label)
    cases = annotated_cases(15, 3, 700, 1000)
    _check(cases, device_edmonds(gpu_ctx, [c[0] for c in cases], [c[1] for c in cases]), "annotated 700-1000")
    cases = overlapping_cases(16, 60)
    _check(cases, device_edmonds(gpu_ctx, [c[0] for c in cases], [c[1] for c in cases], power=1.0), "power 1",
           power=1.0)


def sparse_stems(rng, n, count=60):
    """a few random stems over a sequence of n positions: the tier follows n, the work follows the stems"""
    out = []
    for _ in range(count):
        i = rng.randrange(n - 3)
        j = rng.randrange(i + 3, min(n, i + 400))
        out.append((i, j, rng.randint(1, max(1, min(6, (j - i + 1) // 2))), rng.choice([0.25, 1.0, 2.0, 3.25])))
    return out


@pytest.mark.gpu
def test_device_builder_across_the_tier_thresholds(gpu_ctx):
    thr = _threshold()
    rng = random.Random(17)
    for ls, launches in (([255, 256], 1), ([256, 257], 2), ([257, 300], 1), ([thr - 1, thr], 1), ([thr, thr + 1], 2),
                         ([thr + 1], 1), ([100, 700, thr + 1], 3)):
        sq = [T.rand_seq(rng, n) for n in ls]
        st = [sparse_stems(rng, n) for n in ls]
        got = device_edmonds(gpu_ctx, sq, st)
        assert gpu_ctx.stats()["launches"] == launches, ls
        assert got == [host_edmonds(b) for b in st], ls


@pytest.mark.gpu
def test_device_builder_on_long_sequences(gpu_ctx):
    # device-enumerated stems under a strict set (minlen 4, minbpscore 16), against the emulator: the search is
    # sequential, so a sequence takes seconds to minutes here (DESIGN 3.10), and NetworkX longer still
    rng = random.Random(18)
    ps = T._ps(algorithms={"E"}, bpweights={"GC": 3.25, "AU": 1.25, "GU": 0.5}, minlen=4.0, minbpscore=16.0)
    seqs = [T.rand_seq(rng, n) for n in (3000, 5000)]
    stems = _device_stems(gpu_ctx, seqs, ps)
    got = device_edmonds(gpu_ctx, seqs, stems)
    assert got == emu_edmonds(seqs, stems, 256) and all(len(g) > 100 for g in got)


@pytest.mark.gpu
def test_device_builder_rejects_bad_input(gpu_ctx):
    from squarna_b200._lib import SqrnError
    for stem in ((0, 5, 1, 1.0), (-1, 3, 1, 1.0), (0, 4, 0, 1.0), (3, 4, 3, 1.0), (2, 2, 1, 1.0), (1, 4, 3, 1.0),
                 (0, 4, 1, -1.0), (0, 4, 1, math.nan), (0, 4, 1, 1e300), (0, 4, 1, math.inf)):
        with pytest.raises(SqrnError) as e:
            device_edmonds(gpu_ctx, ["ACGUA"], [[stem]])
        assert e.value.code == E_BADARG, stem
    with pytest.raises(SqrnError) as e:
        device_edmonds(gpu_ctx, ["A" * (MAX_LEN + 1)], [[]])
    assert e.value.code == E_BADARG
    assert device_edmonds(gpu_ctx, ["", "A", "AC", "ACGUACGU"], [[], [], [], []]) == [[], [], [], []]
    # zero-weight edges are tight from the start and get matched, as in NetworkX
    assert device_edmonds(gpu_ctx, ["ACGUACGU", ""], [[(0, 7, 2, 0.0)], []]) == [host_edmonds([(0, 7, 2, 0.0)]), []]


class _HostBuilderContext:
    """the library context without `edmonds`: _predict_many_mixed then runs SQRNalgos.Edmonds on the host (Nussinov
    and Hungarian stay on the device)"""

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

    def hungarian(self, *a, **k):
        return self._ctx.hungarian(*a, **k)


@pytest.mark.gpu
@pytest.mark.parametrize("conf,lens", [("edmondsnobpp", (120, 300, 640)), ("nobpp", (90, 300, 420))])
def test_predict_many_with_the_device_builder(gpu_ctx, monkeypatch, conf, lens):
    rng = random.Random(19)
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
def test_cli_edmonds_text_with_the_device_builder(gpu_ctx, monkeypatch, tmp_path):
    from squarna_b200 import SQUARNA as CLI
    rng = random.Random(20)
    lines = []
    for k in range(12):
        lines += [">e%d" % k, T.rand_seq(rng, rng.randint(40, 300))]
    path = tmp_path / "multi.fas"
    path.write_text("\n".join(lines) + "\n")
    out = []
    for host in (False, True):
        if host:
            host_ctx = _HostBuilderContext(S.get_context(0))
            monkeypatch.setattr(S, "get_context", lambda device=0: host_ctx)
        buf = io.StringIO()
        with contextlib.redirect_stdout(buf):
            CLI.Main(["i=" + str(path), "c=edmondsnobpp", "t=1"])
        out.append(buf.getvalue())
    assert out[0] == out[1] and out[0].count(">e") == 12
