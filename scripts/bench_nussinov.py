"""The Nussinov builder on the device (sqrn_nussinov_batch) against the host builder SQRNalgos.Nussinov.  Prints one
JSON line with the card name and power limit read in the same run.

Builder alone: a host clock around the C call (it returns after a device synchronise), after one warm-up call on the
same batch; the stems come from sqrn_yield_stems_batch under nussinovnobpp.conf's defN.  Workloads: 20 000 sequences
U{60..200} (all in the shared-memory tier, <= 238 nt on a B200), 500 sequences U{300..1500} (global tier) and
8 sequences U{3000..5000} (global tier, fewer sequences than SMs).  The host builder runs on a stated prefix of a
workload; its time for the whole workload is the prefix's mean per sequence times the count (the prefix is drawn from
the same length distribution), labelled as extrapolated.  The device pairs are compared with the host pairs on the
prefix.

End to end: predict_many with nussinovnobpp and nobpp on prefixes of the first two workloads, once with the library
context (device builder) and once through a context without `nussinov` (host builder); outputs compared."""
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
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                         capture_output=True, text=True, check=True).stdout.strip().split("\n")[0]
    name, power = (x.strip() for x in out.split(","))
    return name, power


def conf(name):
    return CLI.ParseConfig(os.path.join(os.path.dirname(os.path.abspath(CLI.__file__)), name + ".conf"))[1]


class HostBuilderContext:
    """the library context without `nussinov`: _predict_many_mixed runs SQRNalgos.Nussinov on the host"""

    def __init__(self, ctx):
        self._ctx = ctx

    def yield_stems(self, *a, **k):
        return self._ctx.yield_stems(*a, **k)

    def predict_batch(self, *a, **k):
        return self._ctx.predict_batch(*a, **k)


def builder_leg(ctx, ps, name, seqs, host_prefix):
    batch = PackedBatch([s.encode() for s in seqs])
    stems = ctx.yield_stems(ps, batch)
    ctx.nussinov(batch.symbols, batch.offsets, stems)                      # warm-up
    t0 = time.perf_counter()
    got = ctx.nussinov(batch.symbols, batch.offsets, stems)
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
            want = SQRNalgos.Nussinov(seqs[b], lists, len(seqs[b]), S.SEPS)
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
    name, power = card()
    ctx = S.get_context(0)
    ps = conf("nussinovnobpp")[0]
    work = {"smem_20000x60-200": T.rand_seqs(1, 200 if q else 20000, 60, 200),
            "global_500x300-1500": T.rand_seqs(2, 10 if q else 500, 300, 1500),
            "long_8x3000-5000": T.rand_seqs(3, 2 if q else 8, 3000, 5000)}
    prefix = {"smem_20000x60-200": 40, "global_500x300-1500": 3, "long_8x3000-5000": 0}
    builder = [builder_leg(ctx, ps, k, v, prefix[k]) for k, v in work.items()]
    e2e = []
    for confname, na, nb in (("nussinovnobpp", 200, 4), ("nobpp", 60, 2)):
        e2e.append(e2e_leg(ctx, confname, "smem prefix", work["smem_20000x60-200"][:na]))
        e2e.append(e2e_leg(ctx, confname, "global prefix", work["global_500x300-1500"][:nb]))
    print(json.dumps(dict(bench="nussinov", card=name, power_limit=power, builder=builder, end_to_end=e2e)))


if __name__ == "__main__":
    main()
