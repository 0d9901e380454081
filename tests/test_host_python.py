"""Host-side Python of squarna_b200 (parsers, config, dbn helpers, reactivity handling,
text output) against golden vectors produced by the real reference.  No GPU needed."""
import contextlib
import io
import json
import math
import os

import pytest

from squarna_b200 import SQRNdbnseq as S
from squarna_b200 import SQUARNA as CLI

G = os.path.join(os.path.dirname(__file__), "golden")
PKG = os.path.dirname(os.path.abspath(CLI.__file__))


def load(name):
    with open(os.path.join(G, name)) as f:
        return json.load(f)


def test_shipped_configs_parse_like_the_reference():
    """every .conf shipped in the package gives the names and values the reference's files give"""
    gold = load("configs.json")
    assert len(gold) == 17
    for conf, g in gold.items():
        names, psets = CLI.ParseConfig(os.path.join(PKG, conf + ".conf"))
        assert names == g["names"], conf
        assert len(psets) == len(g["paramsets"])
        for ps, gp in zip(psets, g["paramsets"]):
            ps = dict(ps)
            ps["algorithms"] = sorted(ps["algorithms"])
            assert ps == gp, (conf, ps, gp)
            assert list(ps["bpweights"]) == list(gp["bpweights"])      # dict order matters (seq.py:282-284)


def test_config_errors(tmp_path):
    p = tmp_path / "bad.conf"
    p.write_text(">x\nalgorithms G\nbpweights GC=1\n")
    with pytest.raises(ValueError, match="Missing some of the parameters"):
        CLI.ParseConfig(str(p))


def test_reactivity_helpers():
    for c in load("reacts.json"):
        vals = [float("nan") if v is None else v for v in c["vals"]]
        out = S.ProcessReacts(vals, M=c["M"], B=c["B"])
        assert [float(x) for x in out] == c["out"]
        for f, enc in c["enc"].items():
            assert S.EncodedReactivities(c["seq"], out, int(f)) == enc
    assert S.ProcessReacts([]) == []
    assert S.ReactDict["z"] == 1.0 and S.ReactDict["d"] == 0.12 and S.ReactDict["?"] == -999


def test_pairs_to_dbn_and_levels():
    for c in load("levels.json"):
        pairs = [tuple(p) for p in c["pairs"]]
        assert S.PairsToDBN(pairs, c["n"]) == c["dbn"]
        lev = S.PairsToDBN(pairs, returnlevels=True)
        assert sorted([k[0], k[1], v] for k, v in lev.items()) == c["levels"]
        assert set(S.DBNToPairs(c["dbn"])) == set(pairs) or max(v for _, _, v in c["levels"]) > 49


def test_dbn_helpers():
    assert S.DBNToPairs("((..[[..))..]]") == [(0, 9), (1, 8), (4, 13), (5, 12)]
    assert S.DBNToPairs("))((") == []                       # closers without openers are ignored
    assert S.DBNToPairs("Бб") == [(0, 1)]
    assert S.UnAlign("AC-GU", "(.(.)") == ("ACGU", "(...")   # the pair (2,4) touches a gap column and vanishes
    assert S.UnAlign("A-CGU", "(..).") == ("ACGU", "(.).")
    assert S.ReAlign("(.).", "A-CGU") == "(..)."
    assert S.ReAlign("ACGU", "A-CGU", seqmode=True) == "A-CGU"
    with pytest.raises(AssertionError, match="Cannot ReAlign"):
        S.ReAlign("(.)", "A-CGU")
    assert S.PairsToStems([(0, 9), (1, 8), (4, 13)]) == [[[(0, 9), (1, 8)], 2], [[(4, 13)], 1]]
    assert S.ParseRestraints("(_/\\+)") == ([(0, 5)], {1, 4}, {2}, {3})


def test_default_format_parser():
    path = os.path.join(G, "inputs", "seq_input.fas")
    entries = list(CLI.ParseDefaultInput(path, "qtrf"))
    assert len(entries) == 17
    by_name = {e[0]: e for e in entries}
    name, seq, reacts, rest, ref = by_name[">External loop 1"]
    assert seq == "CCCAAAAGGG;CCCAAAAGGG" and reacts is None       # the trailing comment is dropped
    assert len(by_name[">testcase with reactivities"][2]) == 16
    assert by_name[">multiple chains with bp-to-the-right restraints"][3] == "........./////....................."
    assert CLI.GuessFormat(path) == ("default", False)
    assert CLI.GuessFormat(os.path.join(G, "inputs", "ali_input.afa"))[0] == "default"
    d = next(CLI.ParseDefaultInput(os.path.join(G, "inputs", "ali_input.afa"), "qtrf", returndefaults=True))
    assert d[0] is not None and d[2] is not None and len(d[0]) == len(d[2]) == 115


def test_other_parsers(tmp_path):
    fa = tmp_path / "x.fa"
    fa.write_text(">a\nACGU\nACGU\n\n>b\nGGGG\n")
    assert list(CLI.ParseFasta(str(fa))) == [(">a", "ACGUACGU", None, None, None), (">b", "GGGG", None, None, None)]
    assert CLI.GuessFormat(str(fa)) == ("fasta", False)
    stk = tmp_path / "x.stk"
    stk.write_text("# STOCKHOLM 1.0\n#=GF ID test\ns1 ACGU\ns2 AC-U\n#=GC SS_cons (..)\n\ns1 GG\ns2 GG\n#=GC SS_cons ..\n//\n")
    objs, single = CLI.ParseStockholm(str(stk))
    assert objs == [(">s1", "ACGUGG", None, None, "(..)..",), (">s2", "AC-UGG", None, None, "(..)..")] and not single
    assert CLI.ParseStockholm(str(stk), True) == (None, None, "(..)..")
    aln = tmp_path / "x.aln"
    aln.write_text("CLUSTAL W\n\ns1 ACGU\ns2 AC-U\n   **\n\ns1 GG\ns2 GG\n")
    assert CLI.ParseClustal(str(aln)) == ([(">s1", "ACGUGG", None, None, None), (">s2", "AC-UGG", None, None, None)], False)
    assert CLI.GuessFormat(str(aln)) == ("clustal", 0) and CLI.GuessFormat(str(stk)) == ("stockholm", 0)


def test_predict_argument_errors():
    with pytest.raises(AssertionError, match="Input file does not exist"):
        CLI.Predict(inputfile="/nonexistent")
    with pytest.raises(AssertionError, match="Config file does not exist"):
        CLI.Predict(inputseq="ACGU", configfile="nope")
    with pytest.raises(ValueError, match="Inappropriate toplim"):
        CLI.Predict(inputseq="ACGU", configfile="fastest", toplim="x")
    with pytest.raises(AssertionError, match="Inappropriate rankby"):
        CLI.Predict(inputseq="ACGU", configfile="fastest", rankby="q")
    with pytest.raises(ValueError, match="Inappropriate algorithm"):
        CLI.Predict(inputseq="ACGU", configfile="fastest", algorithms="x")
    with pytest.raises(NotImplementedError):          # rfam / g4 / rbp restraint discovery: external binaries + network
        CLI.Predict(inputseq="ACGU", configfile="fastest", rfam=True)


def test_evalonly_cli_text_matches_reference():
    """`eo` needs no prediction: parser + ReferenceScores + text are host code (byte-equal output)"""
    argv = load("cli_manifest.json")["seq_evalonly"]
    buf = io.StringIO()
    cwd = os.getcwd()
    os.chdir(G)
    try:
        with contextlib.redirect_stdout(buf):
            CLI.Main(argv)
    finally:
        os.chdir(cwd)
    with open(os.path.join(G, "cli", "seq_evalonly.txt")) as f:
        assert buf.getvalue() == f.read()


# ---- bulk text lane (csrc/sqrn_textio.cpp): the same entries and the same text as the per-entry Python path
def _rand_text(rng, n, fasta, gaps=True):
    lines = []
    for k in range(n):
        name = ">seq%d" % k + rng.choice(["", " some description", "\tx=1  "])
        alphabet = "ACGUTacgun" + ("-.~" if gaps else "")
        seq = "".join(rng.choice(alphabet) for _ in range(rng.randint(1, 90)))
        if seq[0] in "-.~":
            seq = "A" + seq[1:]
        lines.append(name)
        if fasta:
            while seq:
                cut = rng.randint(1, 60)
                lines.append(rng.choice(["", " "]) + seq[:cut])
                seq = seq[cut:]
                if rng.random() < 0.1:
                    lines.append("")
        else:
            lines.append(seq + rng.choice(["", " a comment", "\t# x"]))
            if rng.random() < 0.2:
                lines.append("")
    return "\n".join(lines) + rng.choice(["", "\n", "\r\n"])


@pytest.mark.parametrize("fasta", [False, True], ids=["default", "fasta"])
def test_bulk_text_parse_matches_the_entry_parsers(tmp_path, fasta):
    import random
    from squarna_b200 import _lib
    rng = random.Random(5)
    for trial in range(20):
        text = _rand_text(rng, rng.randint(1, 40), fasta)
        if trial % 4 == 3:
            text = text.replace("\r\n", "\n").replace("\n", "\r\n")
        path = tmp_path / ("t%d.fa" % trial)
        path.write_bytes(text.encode())
        want = list(CLI.ParseFasta(str(path)) if fasta else CLI.ParseDefaultInput(str(path), "qtrf"))
        got = _lib.text_parse(text.encode(), fasta)
        assert got is not None and got.n == len(want)
        for k, (name, seq, reacts, rests, ref) in enumerate(want):
            assert reacts is None and rests is None and ref is None
            b = int(got.name_begin[k])
            assert text.encode()[b:b + int(got.name_len[k])].decode() == name
            assert bytes(got.seq[got.seq_offsets[k]:got.seq_offsets[k + 1]]).decode() == seq


def test_bulk_text_parse_declines_other_shapes():
    from squarna_b200 import _lib
    for text in (b"....\n>s\nACGU\n",                       # default restraints line
                 b">s\nACGU\n0.1 0.2 0.3 0.4\n",            # reactivities of the entry
                 b">s\nACGU\n\n((.))\n",                   # restraints after a blank reactivity line
                 b">s\n\nACGU\n",                           # blank sequence line (an error in the reference)
                 b">s\n", b"", b"ACGU\n",                    # no sequence / no entry
                 b">s\nAC\xc3\xa9GU\n", b">s\nAC\rGU\n"):   # not ASCII / lone CR
        assert _lib.text_parse(text, False) is None, text
    assert _lib.text_parse(b"junk\n>s\nAC\nGU\n", True).n == 1          # FASTA drops text before the first '>'


def test_bulk_text_format_matches_the_entry_printer():
    import random
    import numpy as np
    from squarna_b200 import _lib
    rng = random.Random(6)
    text = _rand_text(rng, 60, False).encode()
    parsed = _lib.text_parse(text, False)
    seqs = [bytes(parsed.seq[parsed.seq_offsets[k]:parsed.seq_offsets[k + 1]]).decode() for k in range(parsed.n)]
    short = ["".join(ch for ch in s if ch not in S.GAPS) for s in seqs]
    dbns = ["".join(rng.choice("..(([)]).") for _ in s) for s in short]
    sym_off = np.zeros(parsed.n + 1, np.int64)
    np.cumsum([len(s) for s in short], out=sym_off[1:])
    dbn = np.frombuffer("".join(dbns).encode(), np.uint8)
    vals = [0.0, 0.5, 12.0, 187.935, 3.1, 1234567.891, 0.001, 45.67, 100.0, 0.125]
    scores = np.array([[rng.choice(vals), rng.choice(vals), rng.choice(vals)] for _ in seqs])
    got = _lib.text_format(parsed, 0, parsed.n, sym_off, dbn, scores, 2, "fastestG").decode()
    want = io.StringIO()
    for k, s in enumerate(seqs):
        name = text[int(parsed.name_begin[k]):int(parsed.name_begin[k]) + int(parsed.name_len[k])].decode()
        long_dbn = S.ReAlign(dbns[k], s)
        total, struct, react = (float(x) for x in scores[k])
        pred = (long_dbn, [(long_dbn, (total, 0 if struct == 0 else struct, react), [0])], [math.nan] * 6, [math.nan] * 7)
        S._print_entry(name, s, None, None, None, 3, want)
        S._print_prediction(pred, s, None, None, ["fastestG"], 2, 1, want)
    assert got == want.getvalue()
    part = _lib.text_format(parsed, 7, 5, sym_off, dbn, scores, 2, "fastestG").decode()
    assert part in got and part.startswith(">seq7")


def test_bulk_text_numbers_print_like_python():
    """scores are round(x, 3) values; the bulk formatter must print them as Python's print() does
    (shortest repr): integer-arithmetic digits in csrc/sqrn_textio.cpp against repr() on many magnitudes"""
    import random
    import numpy as np
    from squarna_b200 import _lib
    rng = random.Random(7)
    vals = [0.0, -0.0, 0.001, -0.001, 0.5, 1.0, 12.0, 100.0, 187.935, 999.999, 1000.0, 123456.789, 1e9 + 0.125, 4.0e12 - 1, 5e12,
            0.1, 0.01, 0.07, 2.675, 1.005, 99999999.999]
    for _ in range(30000):
        mag = rng.choice([1, 10, 1000, 1e5, 1e8])
        vals.append(round(rng.uniform(-mag, mag), 3))
    vals = [round(v, 3) for v in vals]
    n = len(vals)
    text = ("".join(">s\nA\n" for _ in range(n))).encode()
    parsed = _lib.text_parse(text, False)
    sym, sym_off = _lib.text_ungap(parsed)
    assert bytes(sym) == b"A" * n and sym_off[-1] == n
    scores = np.zeros((n, 3))
    scores[:, 0] = vals
    scores[:, 1] = 1.0
    scores[:, 2] = vals[::-1]
    out = _lib.text_format(parsed, 0, n, sym_off, np.full(n, ord("."), np.uint8), scores, 1, "x").decode().split("\n")
    lines = [ln for ln in out if "\t#1\t" in ln]
    assert len(lines) == n
    for k, ln in enumerate(lines):
        f = ln.split("\t")
        assert f[2] == repr(float(vals[k])) and f[4] == repr(float(vals[n - 1 - k])), (vals[k], f)


def test_bulk_text_ungap_matches_unalign():
    from squarna_b200 import _lib
    text = b">a\nAC-G.U~A\n>b\n---\n>c\nacgu\n"
    parsed = _lib.text_parse(text, False)
    sym, off = _lib.text_ungap(parsed)
    want = [S.UnAlign(s, "." * len(s))[0] for s in ("AC-G.U~A", "---", "acgu")]
    assert [bytes(sym[off[k]:off[k + 1]]).decode() for k in range(3)] == want


def test_bulk_lane_glue_without_a_gpu(tmp_path, monkeypatch):
    """the Python glue of the CLI bulk lane (parse -> ungap -> predict -> format) with the GPU call stubbed out:
    the text must be what the per-entry printer writes for the same (stub) prediction"""
    import numpy as np

    class Stub:
        def fast_predict(self, ps, sym, off):
            n = len(off) - 1
            dbn = np.full(len(sym), ord("."), np.uint8)
            for k in range(n):                       # a hairpin where there is room, so that gaps get re-inserted into brackets
                if off[k + 1] - off[k] >= 8:
                    dbn[off[k]] = ord("(")
                    dbn[off[k + 1] - 1] = ord(")")
            return dbn, np.tile([1.5, 3.0, 0.5], (n, 1)), np.ones(n, np.int32)

    monkeypatch.setattr(S, "get_context", lambda device=0: Stub())
    path = tmp_path / "in.fa"
    path.write_text(">a x\nACG-UACGU.A\n>b\nGGGG comment\n>c\nacgu~acguacgu\n")
    buf = io.StringIO()
    assert CLI._bulk_lane(str(path), False, "fastestG", {"dummy": 1}, 1, buf)
    want = io.StringIO()
    for name, seq in ((">a x", "ACG-UACGU.A"), (">b", "GGGG"), (">c", "acgu~acguacgu")):
        short = "".join(ch for ch in seq if ch not in S.GAPS)
        d = "." * len(short) if len(short) < 8 else "(" + "." * (len(short) - 2) + ")"
        long_dbn = S.ReAlign(d, seq)
        S._print_entry(name, seq, None, None, None, 3, want)
        S._print_prediction((long_dbn, [(long_dbn, (1.5, 3.0, 0.5), [0])], [math.nan] * 6, [math.nan] * 7),
                            seq, None, None, ["fastestG"], 1, 1, want)
    assert buf.getvalue() == want.getvalue()
    (tmp_path / "other.fa").write_text(">a\nACGU\n((..))\n")
    assert CLI._bulk_lane(str(tmp_path / "other.fa"), False, "fastestG", {"dummy": 1}, 1, io.StringIO()) is False


def test_bulk_lane_hands_deep_pseudoknots_to_the_entry_path(tmp_path, monkeypatch):
    """a sequence the fast lane marks n_stems = -1 (more than 30 pseudoknot levels: no one-byte glyph left) is
    printed by the per-entry path IN ITS PLACE; the entries around it stay on the bulk formatter"""
    import numpy as np

    class Stub:
        def fast_predict(self, ps, sym, off):
            n = len(off) - 1
            nst = np.ones(n, np.int32)
            nst[1] = -1
            nst[3] = -1
            return np.full(len(sym), ord("."), np.uint8), np.tile([0.0, 0.0, 0.5], (n, 1)), nst

    monkeypatch.setattr(S, "get_context", lambda device=0: Stub())
    path = tmp_path / "in.fa"
    path.write_text(">a\nACGU\n>b deep\nGG-GG\n>c\nACGUACGU\n>d\nCCCC\n")
    seen = []

    def per_entry(entries):
        seen.extend(entries)
        buf.write("<%s|%s>\n" % entries[0][:2])

    buf = io.StringIO()
    assert CLI._bulk_lane(str(path), False, "fastestG", {"dummy": 1}, 1, buf, per_entry=per_entry)
    assert seen == [(">b deep", "GG-GG", None, None, None), (">d", "CCCC", None, None, None)]
    parts = buf.getvalue().split("<>b deep|GG-GG>\n")
    assert len(parts) == 2 and parts[0].startswith(">a\nACGU\n") and parts[1].startswith(">c\nACGUACGU\n")
    assert parts[1].endswith("<>d|CCCC>\n")
    # without a per-entry printer the lane declines (the caller then prints everything per entry)
    assert CLI._bulk_lane(str(path), False, "fastestG", {"dummy": 1}, 1, io.StringIO()) is False


class _OracleContext:
    """stands in for the GPU context in CPU tests of the host logic: AnnotateStems and the greedy structures come
    from the oracle (which the -m gpu tests prove bit-identical to the kernels)"""

    @staticmethod
    def _extras(b, q, k):
        """(alignment weights, bpp term, bpp mode) of entry k = the q-th of the batch"""
        import numpy as np
        p = b["preps"][k]
        smat = None
        if b["stemmatrix"] is not None:
            keep = p.keep
            smat = np.asarray(b["stemmatrix"], dtype=np.float64)[np.ix_(keep, keep)]
        bpp = b["opts"].get("bpp")
        return smat, (bpp[1][q] if bpp else None), (bpp[0] if bpp else 0)

    def yield_stems(self, ps, b):
        import numpy as np
        from oracle import oracle as O
        out = []
        for q, k in enumerate(b["idx"]):
            p = b["preps"][k]
            smat, term, mode = self._extras(b, q, k)
            st = O.annotate(p.shortseq, ps, p.shortreacts, p.shortrest, (), b["interchainonly"], smat, term, mode)
            out.append((np.array([s[:3] for s in st], dtype=np.int32).reshape(-1, 3), np.array([s[3] for s in st])))
        return out

    def predict_batch(self, paramsets, b):
        import numpy as np
        from oracle import oracle as O
        out = []
        for q, k in enumerate(b["idx"]):
            p = b["preps"][k]
            smat, term, mode = self._extras(b, q, k)
            o = b["opts"]
            prio = [q_ for q_ in range(len(paramsets)) if o.get("priority_mask", 0) >> q_ & 1]
            cons, structs, _ = O.predict_short(p.shortseq, p.shortreacts, p.shortrest, list(paramsets), b["interchainonly"],
                                               o.get("poollim", 1000), smat, o.get("rankby", (0, 2, 1)), prio,
                                               o.get("rankbydiff", False), o.get("conslim", 1), o.get("hardrest", False),
                                               b["comp"], raw_codes=True, bpp_term=term, bpp_mode=mode)
            out.append((cons, [(codes, sc, isint, sum(1 << q_ for q_ in psl), np.array(stems, dtype=np.int32).reshape(-1, 3))
                               for codes, sc, isint, psl, stems, *_ in structs], len(structs)))
        return out

    def predict_batch_flat(self, paramsets, b):
        from squarna_b200._lib import FlatResult
        return FlatResult.from_sequences(self.predict_batch(paramsets, b))


def _stand_in(monkeypatch):
    monkeypatch.setattr(S, "get_context", lambda device=0: _OracleContext())
    monkeypatch.setattr(S, "_make_batch", lambda preps, idx, comp, stemmatrix, interchainonly, **opts:
                        dict(preps=preps, idx=idx, comp=comp, stemmatrix=stemmatrix, interchainonly=interchainonly, opts=opts))


def test_bpp_parameter_sets_on_the_host(monkeypatch):
    """def.conf / greedy.conf / 500.conf / edmonds / hungarian / nussinov.conf -- the configs with bpp != 0 sets, which
    the CLI uses by default -- against the REAL reference driven by tests/fake_rna.py in place of ViennaRNA
    (tests/golden/seq_api_bpp.json, entropy_bpp.json): BPPMatrix's calls, the additive / multiplicative terms, one
    device call per parameter set, host de-duplication and ranking.  Without an RNA module the call raises what the
    reference raises."""
    from tests import common as T, fake_rna
    _stand_in(monkeypatch)
    S.set_rna_module(None)
    psets = CLI.ParseConfig(os.path.join(PKG, "def.conf"))[1]
    for conf in ("def", "500", "1000", "greedy"):                # every default config asks for ViennaRNA
        with pytest.raises(ModuleNotFoundError):
            S.SQRNdbnseq("GGGGAAAACCCC", paramsets=CLI.ParseConfig(os.path.join(PKG, conf + ".conf"))[1])
    S.set_rna_module(fake_rna)
    try:
        confs, bad = {}, []
        cases = load("seq_api_bpp.json")
        for c in cases:
            if c["conf"] not in confs:
                confs[c["conf"]] = CLI.ParseConfig(os.path.join(PKG, c["conf"] + ".conf"))[1]
            kw = dict(c["kw"])
            if "priority" in kw:
                kw["priority"] = set(kw["priority"])
            kw["rankby"] = tuple(kw["rankby"])
            got = S.SQRNdbnseq(c["seq"], c["reacts"], c["restraints"], None, confs[c["conf"]], poollim=c["poollim"],
                               M=c["M"], B=c["B"], **kw)
            want = (c["cons"], [(d, tuple(sc), ps) for d, sc, ps in c["structs"]])
            if not T.same_prediction((got[0], got[1]), want):
                bad.append((c["conf"], c["seq"], c["kw"]))
        assert len(cases) >= 90 and not bad, "%d of %d differ; first: %r" % (len(bad), len(cases), bad[0])
        for c in load("entropy_bpp.json"):
            psets = CLI.ParseConfig(os.path.join(PKG, c["conf"] + ".conf"))[1]
            got = S.SQRNdbnseq(c["seq"], c["reacts"], c["restraints"], None, psets, entropy=True,
                               interchainonly=c["interchainonly"])
            assert got == c["entropy"], (c["seq"], got, c["entropy"])
    finally:
        S.set_rna_module(None)


def test_non_greedy_parameter_sets_on_the_host(monkeypatch):
    """_predict_many_mixed (Nussinov / Hungarian / Edmonds builders, RunAlgo, de-duplication across parameter sets,
    RankStructs, consensus, hardrest, level limit, alignment weighting) against the 160 cases of tests/golden/algos.json
    and algos_smat.json made by the real reference, with the oracle supplying what the GPU supplies in the -m gpu version of this test"""
    _stand_in(monkeypatch)
    from tests import common as T
    import numpy as np
    confs, bad = {}, []
    cases = load("algos.json") + load("algos_smat.json")        # the second file: with an alignment-derived stem matrix
    for c in cases:
        if c["conf"] not in confs:
            confs[c["conf"]] = CLI.ParseConfig(os.path.join(PKG, c["conf"] + ".conf"))[1]
        kw = dict(c["kw"])
        if "priority" in kw:
            kw["priority"] = set(kw["priority"])
        kw["rankby"] = tuple(kw["rankby"])
        if c.get("smat") is not None:
            kw["stemmatrix"] = np.array(c["smat"])
        got = S.SQRNdbnseq(c["seq"], c["reacts"], c["restraints"], None, confs[c["conf"]], poollim=c["poollim"], **kw)
        want = (c["cons"], [(d, tuple(sc), ps) for d, sc, ps in c["structs"]])
        if not T.same_prediction((got[0], got[1]), want):
            bad.append((c["conf"], c["seq"], c["kw"]))
    assert not bad, "%d of %d differ; first: %r" % (len(bad), len(cases), bad[0])


def test_bench_helpers_without_a_gpu(monkeypatch):
    """bench.py pieces that do not need a device: workload generator, algorithmic bytes (SURVEY 8d), and the
    best-effort CPU binding of multi-GPU ranks, which must leave the affinity alone when NVML is not usable"""
    import bench
    sym, off, lens = bench.make_batch(1000, bench.SEED)
    assert off[0] == 0 and off[-1] == len(sym) == lens.sum() and lens.min() >= 60 and lens.max() <= 200
    assert set(bytes(sym[:200])) <= set(b"ACGU")
    assert bench.algorithmic_bytes(lens) == int(sum((n + 3) // 4 + 8 + (n + 32) + n for n in lens.tolist()))
    before = os.sched_getaffinity(0)
    assert bench.bind_near_gpu(0) is None or os.sched_getaffinity(0) <= before
    monkeypatch.setenv("SQRN_BENCH_NO_BIND", "1")
    assert bench.bind_near_gpu(0) is None


def test_bench_dump_outputs_format_budget_and_sample(tmp_path, monkeypatch):
    """bench.py --dump-outputs: float32 / float64 .npy files within the byte budget, a sample of whole items that is
    the same from run to run, and each kept item's values equal to the input arrays'"""
    import numpy as np
    import bench
    rng = np.random.default_rng(1)
    n = 3000
    off = np.zeros(n + 1, np.int64)
    np.cumsum(rng.integers(60, 201, n), out=off[1:])
    dbn = rng.choice(np.frombuffer(b".()[]", np.uint8), int(off[-1]))
    sc, ns = rng.random((n, 3)), rng.integers(0, 40, n).astype(np.int32)
    kw = dict(rows={"scores": sc, "n_stems": ns}, ragged={"dbn": (off, dbn)})
    assert bench.dump_outputs(str(tmp_path / "all"), n, **kw) == n
    monkeypatch.setattr(bench, "DUMP_BYTES", 100_000)
    k = bench.dump_outputs(str(tmp_path / "a"), n, **kw)
    assert 0 < k < n and bench.dump_outputs(str(tmp_path / "b"), n, **kw) == k
    files = sorted(os.listdir(tmp_path / "a"))
    assert files == ["dbn.npy", "dbn_offsets.npy", "item_index.npy", "n_stems.npy", "scores.npy"]
    assert sum(os.path.getsize(tmp_path / "a" / f) for f in files) <= 100_000
    got = {f[:-4]: np.load(tmp_path / "a" / f) for f in files}
    for f in files:
        assert got[f[:-4]].dtype in (np.float32, np.float64)
        assert np.array_equal(got[f[:-4]], np.load(tmp_path / "b" / f))
    idx = got["item_index"].astype(np.int64)
    assert len(idx) == k and (np.diff(idx) > 0).all()
    assert np.array_equal(got["scores"], sc[idx]) and np.array_equal(got["n_stems"], ns[idx])
    o = got["dbn_offsets"].astype(np.int64)
    for j, b in enumerate(idx.tolist()):
        assert np.array_equal(got["dbn"][o[j]:o[j + 1]], dbn[off[b]:off[b + 1]])


def test_sqrndbnseq_host_python_on_the_reference_cases(monkeypatch):
    """squarna_b200.SQRNdbnseq.SQRNdbnseq -- _prepare (gaps, separators, restraints, reactivity decoding), the result
    assembly (level codes -> glyphs, ReAlign, separators, paramset lists, int-0 score) -- on the end-to-end cases of
    tests/golden/seq_api.json made by the real reference, with the oracle standing in for the GPU call"""
    import numpy as np
    from tests import common as T
    _stand_in(monkeypatch)
    confs, bad = {}, []
    cases = load("seq_api.json") + load("seq_api_long.json") + load("seq_api_c3.json") + load("seq_api_c3b.json")
    for c in cases:
        if c["conf"] not in confs:
            psets = CLI.ParseConfig(os.path.join(PKG, c["conf"] + ".conf"))[1]
            confs[c["conf"]] = [p for p in psets if p["algorithms"] == {"G"} and not p["bpp"]]
        kw = dict(c["kw"])
        if "priority" in kw:
            kw["priority"] = set(kw["priority"])
        kw["rankby"] = tuple(kw["rankby"])
        if c.get("smat") is not None:
            kw["stemmatrix"] = np.array(c["smat"])
        got = S.SQRNdbnseq(c["seq"], c["reacts"], c["restraints"], None, confs[c["conf"]], poollim=c["poollim"],
                           algos={"G"}, **kw)
        want = (c["cons"], [(d, tuple(sc), ps) for d, sc, ps in c["structs"]])
        if not T.same_prediction((got[0], got[1]), want):
            bad.append((c["conf"], c["seq"], c["kw"]))
    assert not bad, "%d of %d differ; first: %r" % (len(bad), len(cases), bad[0])


def test_sqrndbnseq_host_python_on_random_parameter_sets(monkeypatch):
    """the same on the reference's outputs under random parameter sets (tests/golden/seq_api_fuzz.json)"""
    from tests import common as T
    _stand_in(monkeypatch)
    bad = []
    cases = load("seq_api_fuzz.json")
    for c in cases:
        kw = dict(c["kw"])
        if "priority" in kw:
            kw["priority"] = set(kw["priority"])
        kw["rankby"] = tuple(kw["rankby"])
        psets = [dict(p, algorithms=set(p["algorithms"])) for p in c["paramsets"]]
        got = S.SQRNdbnseq(c["seq"], c["reacts"], c["restraints"], None, psets, poollim=c["poollim"], algos={"G"}, **kw)
        want = (c["cons"], [(d, tuple(sc), ps) for d, sc, ps in c["structs"]])
        if not T.same_prediction((got[0], got[1]), want):
            bad.append((c["seq"], c["kw"]))
    assert not bad, "%d of %d differ; first: %r" % (len(bad), len(cases), bad[0])


def _oracle_yield_many(entries, bpweights, interchainonly, minlen, minbpscore, device=0, matrix=None):
    """SQRNdbnali._yield_many with the oracle's AnnotateStems in place of the GPU call (matrix: the device-side sum of
    sqrn_stem_matrix_batch is stood in for by the host accumulation; the cells come back unsorted = None)"""
    import numpy as np
    from oracle import oracle as O
    if matrix is not None:
        from squarna_b200 import SQRNdbnali as A
        return A._accumulate_host(_oracle_yield_many(entries, bpweights, interchainonly, minlen, minbpscore), matrix[0]), None
    out = []
    ps = dict(bpweights=bpweights, minlen=minlen, minbpscore=minbpscore)
    for seq, reacts, rests in entries:
        seq = seq.upper().replace("T", "U")
        shortseq, shortrest = S.UnAlign(seq, rests if rests else "." * len(seq))
        keep = [k for k, ch in enumerate(seq) if ch not in S.GAPS]
        shortreacts = [reacts[k] for k in keep] if reacts else None
        st = O.annotate(shortseq, ps, shortreacts, shortrest, (), interchainonly, None)
        out.append((np.array(keep, dtype=np.int32), np.array([s[:3] for s in st], dtype=np.int32).reshape(-1, 3),
                    np.array([s[3] for s in st], dtype=np.float64)))
    return out


def _oracle_fast_predict(self, paramset, symbols, offsets):
    import numpy as np
    from oracle import oracle as O
    # (the library's symbol table folds case and T -> U, seq.py:1004; the oracle takes normalised symbols)
    norm = np.frombuffer(bytes(symbols).upper().replace(b"T", b"U"), dtype=np.uint8)
    codes, scores, nst = O.predict_batch_simple(norm, offsets, [paramset], poollim=1, nthreads=4)
    glyph_o, glyph_c = "([{<ABCDEFGHIJKLMNOPQRSTUVWXYZ", ")]}>abcdefghijklmnopqrstuvwxyz"
    lut = {0: ord(".")}
    for lv in range(1, 31):
        lut[lv], lut[-lv] = ord(glyph_o[lv - 1]), ord(glyph_c[lv - 1])
    dbn = np.array([lut[int(c)] for c in codes.tolist()], dtype=np.uint8)
    seps = (symbols == ord(";")) | (symbols == ord("&"))          # the kernel puts separators back itself
    dbn[seps] = symbols[seps]
    return dbn, scores.reshape(-1, 3), nst


with open(os.path.join(G, "cli_manifest.json")) as _f:
    _CLI_RUNS = json.load(_f)


@pytest.mark.parametrize("name", sorted(_CLI_RUNS))
def test_cli_text_with_the_oracle_standing_in_for_the_gpu(name, monkeypatch):
    """the whole host side of the CLI (option handling, parsers, batching, bulk lane, alignment mode, Nussinov /
    Hungarian / Edmonds sets, printing) against the reference's own text (tests/golden/cli/*.txt); the -m gpu
    version of this test (tests/test_gpu_cli.py) runs the same commands on the kernels"""
    from squarna_b200 import SQRNdbnali as A
    from tests import fake_rna
    _OracleContext.fast_predict = _oracle_fast_predict
    _stand_in(monkeypatch)
    monkeypatch.setattr(A, "_yield_many", _oracle_yield_many)
    S.set_rna_module(fake_rna if name.endswith("_fakerna") else None)     # the default configs ask ViennaRNA for bpp
    buf = io.StringIO()
    cwd = os.getcwd()
    os.chdir(G)
    try:
        with contextlib.redirect_stdout(buf):
            if name.endswith("_error"):            # a malformed entry: the same exception after the same partial output
                with open(os.path.join(G, "cli", name + ".err")) as f:
                    kind = f.read().strip()
                with pytest.raises(Exception) as caught:
                    CLI.Main(_CLI_RUNS[name])
                assert type(caught.value).__name__ == kind
            else:
                CLI.Main(_CLI_RUNS[name])
    finally:
        os.chdir(cwd)
        S.set_rna_module(None)
    with open(os.path.join(G, "cli", name + ".txt")) as f:
        want = f.read()
    got = buf.getvalue()
    if got != want:
        gl, wl = got.split("\n"), want.split("\n")
        for k, (a, b) in enumerate(zip(gl, wl)):
            assert a == b, "first difference at line %d of %s" % (k + 1, name)
        assert len(gl) == len(wl)


@pytest.mark.parametrize("fasta", [False, True], ids=["default", "fasta"])
def test_bulk_text_parse_of_a_long_text_in_segments(tmp_path, fasta):
    """texts above 4 MB are parsed in segments cut at entry boundaries, one host thread each: same entries as the
    entry parsers; a foreign shape anywhere in the text is still declined"""
    import random
    from squarna_b200 import _lib
    rng = random.Random(11)
    text = _rand_text(rng, 80000, fasta)
    assert len(text) > (4 << 20)
    path = tmp_path / "big.fa"
    path.write_bytes(text.encode())
    want = list(CLI.ParseFasta(str(path)) if fasta else CLI.ParseDefaultInput(str(path), "qtrf"))
    got = _lib.text_parse(text.encode(), fasta)
    assert got is not None and got.n == len(want)
    raw = text.encode()
    for k in range(0, got.n, 7):
        name, seq = want[k][0], want[k][1]
        b = int(got.name_begin[k])
        assert raw[b:b + int(got.name_len[k])].decode() == name
        assert bytes(got.seq[got.seq_offsets[k]:got.seq_offsets[k + 1]]).decode() == seq
    assert int(got.seq_offsets[-1]) == len(got.seq) == sum(len(w[1]) for w in want)
    if not fasta:
        cut = text.rfind("\n>", 0, len(text) * 3 // 4)
        broken = text[:cut] + "\n>x\nACGU\n0.1 0.2 0.3 0.4" + text[cut:]          # an entry with a reactivity line, far from the start
        assert _lib.text_parse(broken.encode(), False) is None


def test_packed_format_host_converters():
    """sqrn_pack_symbols / sqrn_unpack_dbn (host only): 2-bit codes of A C G U/T in either case, count of everything
    else; 4-bit bracket codes -> ASCII with every sequence starting on its own byte"""
    import numpy as np
    from squarna_b200 import _lib
    rng = np.random.default_rng(5)
    sym = np.frombuffer(b"ACGUacgutTNn-;&X", np.uint8)
    packed, bad = _lib.pack_symbols(sym)
    assert bad == 6
    codes = [(int(packed[k >> 2]) >> (2 * (k & 3))) & 3 for k in range(len(sym))]
    assert codes[:10] == [0, 1, 2, 3, 0, 1, 2, 3, 3, 3]
    big = rng.integers(0, 4, 5_000_003).astype(np.uint8)
    packed, bad = _lib.pack_symbols(np.frombuffer(b"ACGU", np.uint8)[big])
    assert bad == 0
    k = np.arange(len(big))
    assert ((packed[k >> 2] >> (2 * (k & 3)).astype(np.uint8)) & 3 == big).all()
    # unpack: lengths of both parities at offsets of both parities
    lens = rng.integers(0, 40, 3000)
    off = np.zeros(len(lens) + 1, np.uint32)
    off[1:] = np.cumsum(lens)
    total = int(off[-1])
    nib = np.zeros(total // 2 + len(lens) + 1, np.uint8)
    want = np.zeros(total, np.uint8)
    glyph = ".([{<ABC" + ".)]}>abc"
    for b in range(len(lens)):
        base = (int(off[b]) >> 1) + b
        for p in range(int(lens[b])):
            v = int(rng.integers(0, 16))
            if v == 8:
                v = 0
            nib[base + (p >> 1)] |= v << (4 * (p & 1))
            want[int(off[b]) + p] = ord(glyph[v])
    assert bytes(_lib.unpack_dbn(off, nib)) == bytes(want)


def test_alignment_rows_batch_equals_the_per_row_preparation(monkeypatch):
    """SQRNdbnali._rows_batch (the rows of an alignment as one CSR batch, no Python loop over rows) hands the device the
    same arrays as the per-row preparation: symbols, offsets, columns, restraint classes, surviving restraint pairs,
    reactivity values -- with gaps, a shared restraint line with nested / crossing brackets and a shared reactivity list"""
    import random
    import numpy as np
    import workloads
    from squarna_b200 import SQRNdbnali as A
    rows, _ = workloads.config4(40, 90, 120, seed=3)
    L = len(rows[0])
    rng = random.Random(1)
    rest = [rng.choice("....._/\\+") for _ in range(L)]
    for i, j, o, c in [(5, 100, '(', ')'), (6, 99, '(', ')'), (20, 60, '[', ']'), (30, 80, '(', ')'), (31, 79, '(', ')')]:
        rest[i], rest[j] = o, c
    rest = "".join(rest)
    reacts = [round(rng.random(), 2) for _ in range(L)]
    gap = np.frombuffer("".join(sorted(S.GAPS)).encode(), np.uint8)
    captured = {}

    class Ctx:
        def stem_matrix(self, ps, batch, thr):
            captured["b"] = batch

    monkeypatch.setattr(S, "get_context", lambda device=0: Ctx())
    weights = {"GC": 3.25, "AU": 2.0, "GU": -1.0}
    for ents in ([(r, None, None) for r in rows], [(r, reacts, rest) for r in rows], [(r, None, rest) for r in rows],
                 [(r, reacts, None) for r in rows]):
        fast = A._rows_batch(ents, L, gap, False)
        assert fast is not None
        with monkeypatch.context() as m:
            m.setattr(A, "_rows_batch", lambda *a: None)
            A._yield_many(ents, weights, False, 2, 4.5, device=0, matrix=(L, 10.0))
        slow = captured["b"]
        for name in ("symbols", "offsets", "cols", "restr_class", "rbp_offsets", "rbps"):
            a, b = getattr(fast, name), getattr(slow, name)
            if a is None or b is None:
                assert (a is None or not np.any(a)) and (b is None or not np.any(b)), name
                continue
            assert np.array_equal(np.asarray(a).ravel(), np.asarray(b).ravel()), name
        if fast.react_code is not None or slow.react_code is not None:
            assert np.array_equal(fast.react_values[fast.react_code], slow.react_values[slow.react_code])
    # rows with different restraint lines are left to the per-row path
    assert A._rows_batch([(rows[0], None, rest), (rows[1], None, "." * L)] * 8, L, gap, False) is None


def test_reactivity_letter_coding_equals_the_sorted_coding(monkeypatch):
    """_make_batch codes letter-encoded reactivities from a histogram of the letters: the same value table and codes as
    the sort over every processed value it replaces (gaps, '?', entries without reactivities included)"""
    import random
    import numpy as np
    captured = {}
    monkeypatch.setattr(S, "PackedBatch", lambda seqs, **kw: captured.update(kw=kw))
    rng = random.Random(3)
    letters = "abcdefghijklmnopqrstuvwxyz?"
    for trial in range(40):
        ents = []
        for _ in range(rng.randint(1, 6)):
            n = rng.randint(1, 60)
            seq = "".join(rng.choice("ACGU-") for _ in range(n))
            reacts = None if rng.random() < 0.3 else "".join(rng.choice(letters[:rng.randint(1, 27)]) for _ in range(n))
            ents.append((seq, reacts, None, None))
        preps = [S._prepare(*e) for e in ents]
        for comp in (False, True):
            idx = [k for k in range(len(preps)) if preps[k].compensated == comp]
            if not idx:
                continue
            S._make_batch(preps, idx, comp, None, False)
            fast = captured["kw"]
            saved = [p._rl for p in preps]
            for p in preps:
                p._rl = None                                   # the general path: a sort over the values
            S._make_batch(preps, idx, comp, None, False)
            slow = captured["kw"]
            for p, v in zip(preps, saved):
                p._rl = v
            assert (fast["react_values"] is None) == (slow["react_values"] is None)
            if fast["react_values"] is not None:
                assert np.array_equal(fast["react_values"].view(np.uint64), slow["react_values"].view(np.uint64))
                assert all(np.array_equal(x, y) and x.dtype == y.dtype for x, y in zip(fast["react_codes"], slow["react_codes"]))


def test_flat_result_round_trip():
    """FlatResult: per_sequence() of the flat arrays, from_sequences() back, rows that do not lie back to back"""
    import numpy as np
    from squarna_b200._lib import FlatResult
    rng = np.random.default_rng(5)
    seqs = []
    for n, ns in ((7, 3), (0, 0), (12, 1), (5, 0), (9, 4)):
        structs = [(rng.integers(-3, 4, n).astype(np.int8), tuple(np.round(rng.random(3), 3).tolist()), bool(k & 1), int(k + 1),
                    rng.integers(0, 9, (k, 3)).astype(np.int32)) for k in range(ns)]
        seqs.append((rng.integers(-2, 3, n).astype(np.int8), structs, ns + 2))
    flat = FlatResult.from_sequences(seqs)
    back = flat.per_sequence()
    assert len(back) == len(seqs)
    for (cons, structs, ntot), (cons2, structs2, ntot2, c2) in zip(seqs, back):
        assert np.array_equal(cons, cons2) and ntot == ntot2 and len(structs) == len(structs2)
        assert (c2 is None) == (len(structs) == 0)
        for q, ((codes, sc, ii, m, st), (codes2, sc2, ii2, m2, st2)) in enumerate(zip(structs, structs2)):
            assert np.array_equal(codes, codes2) and np.array_equal(codes, c2[q]) and sc == sc2 and ii == ii2 and m == m2
            assert np.array_equal(st, st2)
    # rows of one sequence apart from each other: codes2d gathers them
    flat.dbo[flat.so[4] + 2], flat.dbo[flat.so[4] + 3] = flat.dbo[flat.so[4] + 3], flat.dbo[flat.so[4] + 2]
    c2 = flat.codes2d(4)
    assert np.array_equal(c2[2], seqs[4][1][3][0]) and np.array_equal(c2[3], seqs[4][1][2][0])


def test_predict_many_result_assembly(monkeypatch):
    """predict_many's texts come from one glyph pass per sequence (the library's threaded converter, bytes.translate,
    or numpy tables): against the per-character definition (PairsToDBN glyphs, ReAlign, separators; seq.py:1239-1246)
    on gapped sequences, separators, the Cyrillic levels 31..49, levels beyond the alphabet, empty sequences"""
    import numpy as np
    from squarna_b200 import _lib
    rng = np.random.default_rng(11)
    seqs = ["GGGAAACCC", "GG-GA.AA~CC-C", "GGGA&AACC;C", "G-GG&AA-ACCC", "", "ACGUACGUACGUACGUACGU", "AC-GU&ACGUA"]
    deep = {5: 35, 6: 49, 1: 60}                   # entry -> highest level used

    class Ctx:
        def predict_batch_flat(self, paramsets, batch):
            out = []
            off = np.asarray(batch.offsets)
            for b in range(len(off) - 1):
                n = int(off[b + 1] - off[b])
                top = deep.get(b, 6)
                structs = []
                for q in range(3):
                    codes = rng.integers(-top, top + 1, n).astype(np.int8)
                    if n:
                        codes[rng.integers(0, n)] = top if q == 0 else -top
                    structs.append((codes, (float(q), 0.0 if q == 1 else q + 0.5, 0.25), q == 1, 1 + q, np.zeros((0, 3), np.int32)))
                out.append((rng.integers(-2, 3, n).astype(np.int8), structs, 3))
            Ctx.last = out
            return _lib.FlatResult.from_sequences(out)

    monkeypatch.setattr(S, "get_context", lambda device=0: Ctx())
    from tests import common as T
    ps = [dict(T.FASTEST, algorithms={"G"}) for _ in range(3)]
    got = S.predict_many([(s, None, None, None) for s in seqs], ps, poollim=5, device=0)

    def text(codes, seq):
        glyphs = ["." if c == 0 or abs(c) > len(S._OPEN) else (S._OPEN[c - 1] if c > 0 else S._CLOSE[-c - 1]) for c in codes.tolist()]
        out, k = [], 0                              # (a separator has a position in the ungapped sequence: its own symbol is printed)
        for ch in seq.upper():
            if ch in S.GAPS:
                out.append(".")
            else:
                out.append(ch if ch in ";&" else glyphs[k])
                k += 1
        return "".join(out)

    for seq, (cons, preds, m1, m2), (cons_codes, structs, _) in zip(seqs, got, Ctx.last):
        assert cons == text(cons_codes, seq)
        assert len(preds) == len(structs)
        for (dbn, sc, inds), (codes, osc, isint, mask, _) in zip(preds, structs):
            assert dbn == text(codes, seq), (seq, dbn, text(codes, seq))
            assert sc == (osc[0], 0 if isint else osc[1], osc[2]) and type(sc[1]) is (int if isint else float)
            assert inds == [b for b in range(3) if mask >> b & 1]


def test_unalign_on_byte_arrays_equals_the_per_character_definition():
    """UnAlign (seq.py:236-255) takes a byte-array path for latin-1 strings: against the per-character definition on
    random gapped sequences with brackets of several kinds, pairs that touch gap columns, unmatched brackets; Cyrillic
    brackets take the general path"""
    import random
    rng = random.Random(8)

    def slow(seq, dbn):
        clean = list(dbn)
        for v, w in S.DBNToPairs(dbn):
            if seq[v] in S.GAPS or seq[w] in S.GAPS:
                clean[v] = clean[w] = '.'
        keep = [k for k, ch in enumerate(seq) if ch not in S.GAPS]
        return ''.join(seq[k] for k in keep), ''.join(clean[k] for k in keep)

    for trial in range(400):
        n = rng.randint(1, 80)
        seq = "".join(rng.choice("ACGU-.~;") for _ in range(n))
        alphabet = ".....([{<)]}>Aa_/+" + ("Бб" if trial % 10 == 0 else "")
        dbn = "".join(rng.choice(alphabet) for _ in range(n))
        assert S.UnAlign(seq, dbn) == slow(seq, dbn), (seq, dbn)
    assert S.UnAlign("ACGU", "(..)") == ("ACGU", "(..)")


def test_dbn_pairs_in_the_library_equals_the_python_parser():
    """long dot-bracket lines are parsed by sqrn_dbn_pairs (host only): the same pairs as the Python restatement of
    DBNToPairs (seq.py:172-207) -- every bracket kind incl. the Cyrillic ones, unmatched brackets of both directions"""
    import random
    rng = random.Random(4)
    alphabet = "....." + S._OPEN + S._CLOSE + "_/+-;&?"
    f = S._dbn_pairs.__wrapped__
    for trial in range(1500):
        n = rng.randint(48, 300)
        kinds = rng.randint(1, 12)
        sub = "....." + "".join(rng.sample(S._OPEN, kinds)) + "_/+"
        sub += "".join(S._CLOSE[S._OPEN.index(c)] for c in sub if c in S._OPEN) + rng.choice(alphabet)
        line = "".join(rng.choice(sub) for _ in range(n))
        assert f(line) == S._dbn_pairs_py(line), line
    assert f("." * 60) == () and f("(" * 30 + ")" * 30) == tuple((k, 59 - k) for k in range(30))
    assert S.DBNToPairs(")" * 50 + "(" * 50) == []


def test_bulk_text_parse_with_more_entries_than_guessed():
    """text_parse guesses the entry capacity from the text length; very short entries take the retry with the exact count"""
    from squarna_b200 import _lib
    for fasta in (False, True):
        text = b"".join(b">e%d\n%s\n" % (k, b"ACGU"[k % 4:k % 4 + 1]) for k in range(3000))
        parsed = _lib.text_parse(text, fasta)
        assert parsed is not None and parsed.n == 3000
        assert bytes(parsed.seq) == b"".join(b"ACGU"[k % 4:k % 4 + 1] for k in range(3000))
        assert parsed.seq_offsets.tolist() == list(range(3001))
        assert [int(parsed.name_len[k]) for k in (0, 10, 2999)] == [3, 4, 6]      # ">e0", ">e10", ">e2999"


def test_bulk_lane_writes_slices_through_the_writer_thread(tmp_path, monkeypatch):
    """a binary sink and more entries than one slice: slices are formatted while the previous one is being written
    (two alternating buffers, one writer thread) -- the file must equal the one-slice text, also around an entry that is
    handed to the per-entry path in the middle"""
    import numpy as np
    import random

    class Stub:
        def fast_predict(self, ps, sym, off):
            n = len(off) - 1
            nst = np.ones(n, np.int32)
            nst[37] = -1                                     # "more than 30 pseudoknot levels": the per-entry path prints it
            return np.full(len(sym), ord("."), np.uint8), np.tile([1.5, 3.0, 0.5], (n, 1)), nst

    monkeypatch.setattr(S, "get_context", lambda device=0: Stub())
    rng = random.Random(12)
    path = tmp_path / "in.fa"
    path.write_text("".join(">s%d\n%s\n" % (k, "".join(rng.choice("ACGU") for _ in range(rng.randint(5, 60)))) for k in range(101)))
    texts = []
    for slice_entries in (1000, 7, 1):
        out = tmp_path / ("out%d.txt" % slice_entries)
        with open(out, "w") as sink:
            sink.write("header\n")                           # text written before the lane starts must stay in front
            assert CLI._bulk_lane(str(path), True, "fastestG", {"dummy": 1}, 1, sink, slice_entries=slice_entries,
                                  per_entry=lambda entries: print("<entry %s>" % entries[0][0], file=sink))
            sink.write("trailer\n")
        texts.append(out.read_text())
    assert texts[0] == texts[1] == texts[2]
    assert texts[0].startswith("header\n>s0\n") and texts[0].endswith("trailer\n") and "<entry >s37>" in texts[0]
    assert texts[0].index(">s36\n") < texts[0].index("<entry >s37>") < texts[0].index(">s38\n")
