"""The Edmonds builder on the device (sqrn_edmonds_batch) against the host builder SQRNalgos.Edmonds (NetworkX).  Prints
one JSON line with the card name, power limit and SM clock read in the same run.

Builder alone: a host clock around the C call (it returns after a device synchronise), after a warm-up call on two
of the sequences, and the kernel time from CUDA events; the stems come from sqrn_yield_stems_batch under
edmondsnobpp.conf's first set.  The workloads are scripts/bench_nussinov.py's, so that the builders compare: 20 000
sequences U{60..200} (mostly the warp tier) and 500 sequences U{300..1500} (CTA tier).  The host builder runs on a
stated prefix of a workload; its time for the whole workload is the prefix's mean per sequence times the count (the prefix is drawn from
the same length distribution), labelled as extrapolated.  The device pairs are compared with the host pairs on the
prefix.  The third workload of bench_nussinov.py (8 x 3000-5000 nt) is left out: the matching is a sequential search
per sequence, which takes minutes per sequence on the device at those lengths (NetworkX longer still).

End to end: predict_many with edmondsnobpp and nobpp on prefixes of the first two workloads, once with the library
context (device builder) and once through a context without `edmonds` (host builder; Nussinov and Hungarian stay on the
device); outputs compared."""
import argparse
import json
import os
import random
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np  # noqa: E402

from squarna_b200 import SQRNalgos, SQRNdbnseq as S, SQUARNA as CLI  # noqa: E402
from squarna_b200._lib import PackedBatch  # noqa: E402
from tests import common as T  # noqa: E402


def card():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True, check=True).stdout.strip().split("\n")[0]
    return [x.strip() for x in out.split(",")]


def conf(name):
    return CLI.ParseConfig(os.path.join(os.path.dirname(os.path.abspath(CLI.__file__)), name + ".conf"))[1]


class HostBuilderContext:
    """the library context without `edmonds`: _predict_many_mixed runs SQRNalgos.Edmonds on the host"""

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


def builder_leg(ctx, ps, name, seqs, host_prefix):
    batch = PackedBatch([s.encode() for s in seqs])
    stems = ctx.yield_stems(ps, batch)
    ctx.edmonds(batch.symbols[:batch.offsets[2]], batch.offsets[:3], stems[:2])   # warm-up (module load)
    t0 = time.perf_counter()
    got = ctx.edmonds(batch.symbols, batch.offsets, stems)
    dev_s = time.perf_counter() - t0
    st = ctx.stats()
    lens = np.diff(batch.offsets)
    rec = dict(workload=name, n_seqs=len(seqs), len_min=int(lens.min()), len_max=int(lens.max()),
               stems=int(sum(len(x[1]) for x in stems)), device_s=round(dev_s, 4),
               device_kernel_ms=round(st["kernel_ms"], 2), launches=st["launches"])
    if host_prefix:
        t0 = time.perf_counter()
        diffs = 0
        for b in range(host_prefix):
            lists = [[[(i + t, j - t) for t in range(ln)], ln, s_] for (i, j, ln), s_ in zip(stems[b][0].tolist(), stems[b][1].tolist())]
            want = sorted((min(v, w), max(v, w)) for v, w in SQRNalgos.Edmonds(lists))
            diffs += [tuple(p) for p in got[b].tolist()] != want
        host_s = time.perf_counter() - t0
        est = host_s / host_prefix * len(seqs)
        rec.update(host_prefix=host_prefix, host_prefix_s=round(host_s, 3), host_s_extrapolated=round(est, 1),
                   speedup_extrapolated=round(est / dev_s, 1), prefix_differences=diffs)
    else:
        rec.update(host_s="not measured")
    return rec


def e2e_leg(ctx, confname, name, seqs):
    entries = [(s, None, None, None) for s in seqs]
    pss = conf(confname)
    S.predict_many(entries[:2], pss, device=0)                             # warm-up
    t0 = time.perf_counter()
    dev = S.predict_many(entries, pss, device=0)
    dev_s = time.perf_counter() - t0
    real = S.get_context
    host_ctx = HostBuilderContext(real(0))
    S.get_context = lambda device=0: host_ctx
    try:
        t0 = time.perf_counter()
        host = S.predict_many(entries, pss, device=0)
        host_s = time.perf_counter() - t0
    finally:
        S.get_context = real
    same = all(T.same_prediction(a[:2], b[:2]) for a, b in zip(dev, host)) and len(dev) == len(host)
    return dict(workload=name, conf=confname, n_seqs=len(seqs), device_builder_s=round(dev_s, 3),
                host_builder_s=round(host_s, 3), speedup=round(host_s / dev_s, 2), outputs_equal=same)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--quick", action="store_true", help="small workloads (a rehearsal of the script)")
    a = ap.parse_args()
    q = a.quick
    name, power, clock, max_clock = card()
    ctx = S.get_context(0)
    ps = conf("edmondsnobpp")[0]
    work = {"short_20000x60-200": T.rand_seqs(1, 200 if q else 20000, 60, 200),
            "mid_500x300-1500": T.rand_seqs(2, 10 if q else 500, 300, 1500)}
    prefix = {"short_20000x60-200": 100, "mid_500x300-1500": 1}
    builder = []
    for k, v in work.items():
        builder.append(builder_leg(ctx, ps, k, v, prefix[k]))
        print(json.dumps(builder[-1]), file=sys.stderr, flush=True)          # progress
    e2e = []
    for confname, na, nb in (("edmondsnobpp", 60, 1), ("nobpp", 30, 0)):
        e2e.append(e2e_leg(ctx, confname, "short prefix", work["short_20000x60-200"][:na]))
        print(json.dumps(e2e[-1]), file=sys.stderr, flush=True)
        if nb:
            e2e.append(e2e_leg(ctx, confname, "mid prefix", work["mid_500x300-1500"][:nb]))
            print(json.dumps(e2e[-1]), file=sys.stderr, flush=True)
    print(json.dumps(dict(bench="edmonds", card=name, power_limit=power, sm_clock=clock, max_sm_clock=max_clock,
                          builder=builder, end_to_end=e2e)))


if __name__ == "__main__":
    main()
