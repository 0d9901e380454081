#!/usr/bin/env python
"""bench.py -- throughput of the greedy hot path on BASELINE.json's configs.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--config 2|3|4|5] [--seqs S] [--impl ours|reference]
                    [--dump-outputs DIR]

--config 2 (default, the configuration the metric is quoted on): 1 M synthetic random RNAs U{60..200} per GPU,
            `byseq pl=1 c=fastest.conf`; weak scaling (S per GPU, ranks take disjoint batches).
--config 5: 10 k sequences U{2900..5000}, 1000nobpp.conf G set, pl=1; STRONG scaling: one global batch, dealt
            to the ranks by length ** 3 (squarna_b200/sharding.py), results gathered on rank 0 in input order.
--config 3: 100 k sequences U{300..1500} with reactivity letters and restraints, G sets by length, pl=100
            (pool rounds); strong scaling; a cap on the number of sequences is named in config.workload.

A "step" is one pass of the hot path over the batch.  For N > 1 the driver launches one process per GPU with
torchrun; sequences are independent, so there is no data-path collective (NCCL carries only the timing barrier,
the max over ranks and the gather of finished results).

Printed by rank 0 as ONE JSON line:
  value    sequences/s with inputs resident in HBM (device-pointer C-ABI call; config 3: the C-ABI batch call
           on prepared host batches -- its general entry has no device-pointer form)
  e2e      the same through the host-buffer C-ABI call (config 3: through predict_many from Python strings):
           host -> device copies and device -> host reads inside the timed region
  e2e_cli  (config 2, N = 1) the CLI surface: Predict(inputfile=<1 M-sequence FASTA>, c=fastest, byseq, pl=1),
           text file in, text out
  roofline algorithmic bytes per launch / measured kernel time vs the measured HBM peak
  cpu_baseline  the UNMODIFIED Python reference (baseline/_ref/SQUARNA, `byseq t=<cores>`) on a bounded sample of
           the same workload, and the plain-C oracle port beside it
`--impl reference` times only the CPU side: the Python reference through its own Predict() (rank 0; other ranks exit).
`--dump-outputs DIR` writes, after the timed steps, what the timed path returned in its last step (rank 0's share) as
float32 / float64 .npy files, at most 64 MB in all (see dump_outputs); the inputs are a pure function of the arguments.
"""
import argparse
import io
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import workloads  # noqa: E402

SEED = workloads.SEED
FASTEST = dict(algorithms={"G"}, bpp=0.0, bpweights={"GC": 3.25, "AU": 1.25, "GU": -1.25},
               suboptmax=1.0, suboptmin=1.0, suboptsteps=1.0, minlen=4.0, minbpscore=7.0,
               minfinscorefactor=1.25, distcoef=0.09, bracketweight=-2.0, orderpenalty=1.0,
               loopbonus=0.125, maxstemnum=1e6)          # the reference's fastest.conf
WORKLOAD = "config2: synthetic random RNA, len U{60..200}, byseq pl=1 c=fastest.conf"
METRIC = {2: "sequences/sec (SQRNdbnseq greedy, byseq pl=1 fastest.conf)",
          5: "sequences/sec (SQRNdbnseq greedy, 2900-5000 nt, 1000nobpp.conf G set, pl=1)",
          3: "sequences/sec (SQRNdbnseq greedy, 300-1500 nt, reactivities + restraints, G sets by length, pl=100)"}
REF_DIR = os.path.join(ROOT, "baseline", "_ref", "SQUARNA")


def make_batch(n, seed):
    """config 2's batch (kept under this name for the tests)"""
    return workloads.config2(n, seed)


def algorithmic_bytes(lens):
    """SURVEY.md 8(d): ceil(N/4) + 8 + S*(N + 32) + N per sequence, S = 1 structure"""
    return workloads.algorithmic_bytes(lens)


def conf_gsets(name):
    """bpp-free greedy parameter sets of a shipped .conf (the sets the GPU path serves without ViennaRNA)"""
    from squarna_b200 import SQUARNA as CLI
    psets = CLI.ParseConfig(os.path.join(ROOT, "squarna_b200", name + ".conf"))[1]
    return [p for p in psets if p["algorithms"] == {"G"} and not p.get("bpp", 0)]


def host_cores():
    """cores this process may run on (the box's count when no affinity mask is set)"""
    try:
        return len(os.sched_getaffinity(0)) or (os.cpu_count() or 1)
    except Exception:
        return os.cpu_count() or 1


def cpu_model():
    try:
        with open("/proc/cpuinfo") as f:
            for ln in f:
                if ln.startswith("model name"):
                    return ln.split(":", 1)[1].strip()
    except Exception:
        pass
    return "unknown"


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons during the timed region"""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.rows, self.stop_flag = index, [], False

    def run(self):
        while not self.stop_flag:
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                      "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5).stdout
                f = [x.strip() for x in out.strip().split(",")]
                if len(f) >= 6:
                    self.rows.append(f)
            except Exception:
                pass
            time.sleep(0.05)

    def summary(self):
        if not self.rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
        sm = sorted(float(r[0]) for r in self.rows)
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for k, n in enumerate(names) if any(r[2 + k].lower().startswith("active") for r in self.rows)]
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": float(self.rows[0][1]), "reasons": reasons,
                "samples": len(self.rows)}


# ------------------------------------------------------------------ CPU side: the reference and the port
def write_fasta(path, sym, off, count, reacts=None, rests=None):
    with open(path, "w") as f:
        for b in range(count):
            f.write(">s%d\n" % b)
            f.write(sym[int(off[b]):int(off[b + 1])].tobytes().decode())
            f.write("\n")
            if reacts is not None:
                f.write(reacts[b] + "\n" + rests[b] + "\n")


def run_python_reference(inp, kwargs, timeout=3600):
    """the UNMODIFIED reference through its own Predict() in a child process (scripts/ref_runner.py).
    Returns (seconds inside Predict, output text path) or (None, reason)."""
    if not os.path.isdir(REF_DIR):
        return None, "baseline/_ref/SQUARNA is missing (scripts/install_reference.py copies it from /root/reference)"
    outp = inp + ".out"
    res = subprocess.run([sys.executable, os.path.join(ROOT, "scripts", "ref_runner.py"), inp, outp, json.dumps(kwargs)],
                         capture_output=True, text=True, timeout=timeout)
    if res.returncode != 0:
        return None, "reference failed: " + res.stderr.strip().split("\n")[-1][:200]
    return json.loads(res.stdout.strip().split("\n")[-1])["seconds"], outp


def reference_rate_config2(sym, off, lens, sample, threads, tmpdir):
    """seq/s of the Python reference on the first `sample` sequences: `byseq pl=1 c=fastest.conf t=threads`
    (README usage example 9; SQUARNA.py:887-935)"""
    inp = os.path.join(tmpdir, "ref_c2_%d.fa" % sample)
    write_fasta(inp, sym, off, sample)
    secs, outp = run_python_reference(inp, dict(configfile="fastest", byseq=True, poollim=1, threads=threads))
    if secs is None:
        return None, outp, None
    return sample / secs, secs, outp


def cpu_oracle_rate(sym, off, lens, sample, threads, ps=None):
    """oracle port on `threads` host threads over the first `sample` sequences"""
    from oracle import oracle as O
    O.lib()
    s_off = off[:sample + 1]
    s_sym = sym[:int(s_off[-1])]
    t0 = time.perf_counter()
    O.predict_batch_simple(s_sym, s_off, [ps or FASTEST], poollim=1, nthreads=threads)
    dt = time.perf_counter() - t0
    return sample / dt, float((lens[:sample].astype(np.float64) ** 2).sum()) / dt, dt


def cpu_baseline_config2(sym, off, lens, threads, budget_s=20.0):
    """both CPU rates on a bounded prefix: the Python reference (kind "reference") and the C port beside it"""
    with tempfile.TemporaryDirectory() as tmp:
        cal = min(len(lens), max(threads * 10, 64))                   # one Pool batch per worker (SQUARNA.py:888)
        rate, secs, _ = reference_rate_config2(sym, off, lens, cal, threads, tmp)
        ref = None
        if rate is not None:
            sample = int(min(len(lens), 20000, max(cal, rate * budget_s)))
            rate, secs, _ = reference_rate_config2(sym, off, lens, sample, threads, tmp)
            if rate is not None:
                ref = {"value": rate, "unit": "seq/s", "cores": threads, "kind": "reference", "cpu_model": cpu_model(),
                       "nt2_per_s": float((lens[:sample].astype(np.float64) ** 2).sum()) / secs,
                       "sample": "first %d sequences of the workload, %.1f s inside the reference's own Predict(byseq=True, "
                                 "poollim=1, configfile='fastest', threads=%d) -- baseline/_ref/SQUARNA, unmodified"
                                 % (sample, secs, threads)}
        psample = int(min(len(lens), 50000 * threads))
        prate, pnt2, pdt = cpu_oracle_rate(sym, off, lens, psample, threads)
        port = {"value": prate, "unit": "seq/s", "cores": threads, "kind": "port", "nt2_per_s": pnt2,
                "sample": "first %d sequences, %.1f s, oracle/sqrn_oracle.c (plain-C restatement) on %d threads"
                          % (psample, pdt, threads)}
        if ref is None:
            port["note"] = "Python reference unavailable: " + str(secs)
            return port
        ref["port"] = port
        return ref


def run_reference(args, rank):
    """`--impl reference`: the reference's own CPU implementation of the path on the box's host cores"""
    if rank != 0:
        return
    threads = host_cores()
    if args.config != 2:
        print(json.dumps({"impl": "reference", "unavailable": "the reference arm is defined for the headline config 2; "
                          "configs 3 and 5 report their CPU baseline inside their own line"}), flush=True)
        return
    sym, off, lens = make_batch(min(args.seqs, 40000), SEED)
    with tempfile.TemporaryDirectory() as tmp:
        cal = max(threads * 10, 64)
        rate, secs, _ = reference_rate_config2(sym, off, lens, cal, threads, tmp)
        if rate is None:                                              # no Python reference on this box: the port
            sample = max(1000, min(len(lens), 3000 * threads))
            t0 = time.perf_counter()
            for _ in range(args.steps):
                cpu_oracle_rate(sym, off, lens, sample, threads)
            dt = (time.perf_counter() - t0) / args.steps
            kind, how = "port", "oracle/sqrn_oracle.c on %d threads (%s)" % (threads, secs)
        else:
            # every step = Predict() on a prefix sized so that steps + warm-ups end within ~3 minutes
            budget = 200.0 / max(args.steps + min(args.warmup, 1), 1)
            sample = int(min(len(lens), max(cal, rate * budget)))
            for _ in range(min(args.warmup, 1)):
                reference_rate_config2(sym, off, lens, cal, threads, tmp)
            tot = 0.0
            for _ in range(args.steps):
                tot += reference_rate_config2(sym, off, lens, sample, threads, tmp)[1]
            dt = tot / args.steps
            kind, how = "reference", ("the reference's own Predict(byseq=True, poollim=1, configfile='fastest', threads=%d), "
                                      "baseline/_ref/SQUARNA unmodified" % threads)
    val = sample / dt
    line = {"impl": "reference", "metric": METRIC[2], "value": val, "unit": "seq/s", "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic", "nt2_per_s": float((lens[:sample].astype(np.float64) ** 2).sum()) / dt,
            "config": {"workload": WORKLOAD, "seqs_per_step": sample},
            "cpu_baseline": {"value": val, "unit": "seq/s", "cores": threads, "kind": kind, "cpu_model": cpu_model(),
                             "sample": "first %d sequences of the workload per step; %s" % (sample, how)},
            "e2e": {"value": val, "unit": "seq/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


def bind_near_gpu(index):
    """Multi-GPU runs: keep this rank's host threads (and, by first touch, its pinned buffers) on the CPUs local to
    its GPU -- sysfs local_cpulist of the PCI device when it names a proper subset, else NVML's affinity mask --
    so that the H2D / D2H traffic of the end-to-end leg does not cross sockets.  Best effort: any failure leaves
    the affinity alone.  SQRN_BENCH_NO_BIND=1 switches it off."""
    if os.environ.get("SQRN_BENCH_NO_BIND"):
        return None
    try:
        import pynvml
        pynvml.nvmlInit()
        vis = os.environ.get("CUDA_VISIBLE_DEVICES")
        if vis:
            ids = [x.strip() for x in vis.split(",") if x.strip()]
            if not all(x.isdigit() for x in ids) or index >= len(ids):
                return None
            index = int(ids[index])
        handle = pynvml.nvmlDeviceGetHandleByIndex(index)
        allowed = os.sched_getaffinity(0)
        cpus = []
        try:
            bus = pynvml.nvmlDeviceGetPciInfo(handle).busId
            bus = (bus.decode() if isinstance(bus, bytes) else bus).lower()
            if len(bus.split(":")[0]) == 8:
                bus = bus[4:]
            with open("/sys/bus/pci/devices/%s/local_cpulist" % bus) as f:
                for part in f.read().strip().split(","):
                    lo, _, hi = part.partition("-")
                    cpus += list(range(int(lo), int(hi or lo) + 1))
            cpus = sorted(c for c in cpus if c in allowed)
        except Exception:
            cpus = []
        if not (4 <= len(cpus) < len(allowed)):
            ncpu = os.cpu_count() or 1
            words = pynvml.nvmlDeviceGetCpuAffinity(handle, (ncpu + 63) // 64)
            cpus = sorted(c for c in (64 * w + b for w, m in enumerate(words) for b in range(64) if (int(m) >> b) & 1)
                          if c in allowed)
        if 4 <= len(cpus) < len(allowed):
            os.sched_setaffinity(0, cpus)
            return len(cpus)
    except Exception:
        pass
    return None


def load_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return json.load(f)
    except Exception:
        return {}


def load_traffic(kernel):
    """DRAM bytes and issue metrics of one launch of `kernel` from the committed ncu capture (profiles/traffic_latest.json)"""
    try:
        with open(os.path.join(ROOT, "profiles", "traffic_latest.json")) as f:
            tr = json.load(f)
        for rec in (tr if isinstance(tr, list) else [tr]):
            if rec.get("kernel") == kernel:
                return rec
    except Exception:
        pass
    return None


DUMP_BYTES = 64 * 10 ** 6


def dump_outputs(dirname, n, rows=None, ragged=None, ids=None):
    """--dump-outputs: what the timed path returned for its n output items, as DIR/<name>.npy, so that two builds can be
    compared output for output.  rows: name -> array whose first axis runs over the items; ragged: name -> (offsets,
    values), item k's values at values[offsets[k]:offsets[k + 1]] (written as <name>.npy + <name>_offsets.npy).  float64
    arrays stay float64, one- and two-byte codes become float32, wider integers float64.  When everything does not fit
    in 64 MB, items are taken in a fixed seeded order until the budget is spent.  item_index.npy lists the kept items, as
    positions in the workload's input order when `ids` maps each item to one."""
    from squarna_b200.sharding import take_csr

    def out_size(dt):
        return 4 if np.dtype(dt).itemsize <= 2 and np.dtype(dt).kind != "f" else 8

    def as_float(a):
        return np.asarray(a, dtype=np.float32 if out_size(a.dtype) == 4 else np.float64)

    rows = {k: np.asarray(v) for k, v in (rows or {}).items()}
    ragged = {k: (np.asarray(o, dtype=np.int64), np.asarray(v)) for k, (o, v) in (ragged or {}).items()}
    per_item = np.full(n, 8, dtype=np.int64)                                       # item_index
    for v in rows.values():
        per_item += v.size // max(n, 1) * out_size(v.dtype)
    for o, v in ragged.values():
        per_item += np.diff(o) * out_size(v.dtype) + 8
    order = np.random.default_rng(SEED).permutation(n)
    budget = DUMP_BYTES - 256 * (1 + len(rows) + 2 * len(ragged))                 # (.npy headers)
    keep = np.sort(order[np.cumsum(per_item[order]) <= budget])
    os.makedirs(dirname, exist_ok=True)
    np.save(os.path.join(dirname, "item_index.npy"), (keep if ids is None else np.asarray(ids)[keep]).astype(np.float64))
    for name, v in rows.items():
        np.save(os.path.join(dirname, name + ".npy"), as_float(v[keep]))
    for name, (o, v) in ragged.items():
        sub, sub_off = take_csr(v, o, keep)
        np.save(os.path.join(dirname, name + ".npy"), as_float(sub))
        np.save(os.path.join(dirname, name + "_offsets.npy"), sub_off.astype(np.float64))
    return len(keep)


# ------------------------------------------------------------------------------ configs 2 and 5: the fast lane
def bench_fast(args, rank, world, local):
    import torch
    import torch.distributed as dist
    from squarna_b200 import _lib
    from squarna_b200._abi import ParamSet
    from squarna_b200.sharding import shard_plan, take_csr, plan_imbalance

    cfg = args.config
    strong = cfg == 5
    torch.cuda.set_device(local)
    bound = bind_near_gpu(local) if world > 1 else None
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    ctx = _lib.Context(local)
    stream = torch.cuda.Stream()
    ctx.set_stream(stream.cuda_stream)
    if cfg == 2:
        psd = FASTEST
        n_global = args.seqs * world
        sym, off, lens = make_batch(args.seqs, SEED + rank)                 # weak: every rank its own batch
        workload = WORKLOAD
        imbalance = None
    else:
        psd = conf_gsets("1000nobpp")[0]
        n_global = args.seqs
        gsym, goff, glens = workloads.config5(n_global, SEED)
        plan = shard_plan(glens, world, 3.0)
        idx = plan[rank]
        sym, off = take_csr(gsym, goff, idx)                                 # strong: this rank's queue, longest first
        lens = np.diff(off)
        imbalance = plan_imbalance(glens, plan, 3.0)
        workload = "config5: %d synthetic random RNAs, len U{2900..5000}, 1000nobpp.conf G set, pl=1" % n_global
    ps = ParamSet.from_dict(psd)
    n = len(lens)
    total, max_len = int(off[-1]), int(lens.max())
    h_sym = torch.from_numpy(np.ascontiguousarray(sym)).pin_memory()
    h_off = torch.from_numpy(off).pin_memory()
    h_dbn = torch.empty(total, dtype=torch.uint8).pin_memory()
    h_sc = torch.empty(n * 3, dtype=torch.float64).pin_memory()
    h_ns = torch.empty(n, dtype=torch.int32).pin_memory()
    # the packed boundary format of the same batch (include/sqrn.h): 2-bit base codes + uint32 offsets in,
    # 4-bit bracket codes + scores in thousandths + uint16 stem counts + flags out
    pk_np, n_other = _lib.pack_symbols(sym)
    assert n_other == 0
    p_sym = torch.from_numpy(pk_np).pin_memory()
    p_off = torch.from_numpy(off.astype(np.uint32).view(np.int32)).pin_memory()      # (uint32 values)
    p_nib = torch.empty(total // 2 + n + 1, dtype=torch.uint8).pin_memory()
    p_milli = torch.empty(2 * n, dtype=torch.int32).pin_memory()
    p_ns = torch.empty(n, dtype=torch.int16).pin_memory()                              # (uint16 values)
    p_fl = torch.empty(n, dtype=torch.uint8).pin_memory()
    with torch.cuda.stream(stream):
        d_sym = h_sym.cuda(non_blocking=True)
        d_off = h_off.cuda(non_blocking=True)
        d_dbn = torch.empty(total, dtype=torch.uint8, device="cuda")
        d_sc = torch.empty(n * 3, dtype=torch.float64, device="cuda")
        d_ns = torch.empty(n, dtype=torch.int32, device="cuda")
        dp_sym = p_sym.cuda(non_blocking=True)
        dp_nib = torch.empty(total // 2 + n + 1, dtype=torch.uint8, device="cuda")
        dp_milli = torch.empty(2 * n, dtype=torch.int32, device="cuda")
        dp_ns = torch.empty(n, dtype=torch.int16, device="cuda")
        dp_fl = torch.empty(n, dtype=torch.uint8, device="cuda")
    stream.synchronize()

    def step_device_packed():
        rc = ctx.L.sqrn_fast_predict_packed_device(ctx.h, ps, n, total, max_len, d_off.data_ptr(), dp_sym.data_ptr(), dp_nib.data_ptr(),
                                                   dp_milli.data_ptr(), dp_ns.data_ptr(), dp_fl.data_ptr())
        ctx._check(rc)

    def step_device():
        ctx.fast_predict_device(ps, n, total, max_len, d_off.data_ptr(), d_sym.data_ptr(), d_dbn.data_ptr(),
                                d_sc.data_ptr(), d_ns.data_ptr())

    def step_host():
        rc = ctx.L.sqrn_fast_predict_host(ctx.h, ps, n, h_off.data_ptr(), h_sym.data_ptr(), h_dbn.data_ptr(),
                                          h_sc.data_ptr(), h_ns.data_ptr())
        ctx._check(rc)

    def step_packed():
        rc = ctx.L.sqrn_fast_predict_packed_host(ctx.h, ps, n, p_off.data_ptr(), p_sym.data_ptr(), p_nib.data_ptr(),
                                                 p_milli.data_ptr(), p_ns.data_ptr(), p_fl.data_ptr())
        ctx._check(rc)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps):
        """K steps between barriers; device time by CUDA events on the launch stream, max over ranks"""
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        t0 = time.perf_counter()
        e0.record(stream)
        for _ in range(steps):
            fn()
        e1.record(stream)
        stream.synchronize()
        barrier()
        wall = time.perf_counter() - t0
        ms = e0.elapsed_time(e1)
        t = torch.tensor([ms, wall * 1e3], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t[0]), float(t[1])

    warm = max(args.warmup, 3)
    for _ in range(warm):
        step_device()
    stream.synchronize()
    sampler = ClockSampler(local)
    sampler.start()
    dev_ms, _ = timed(step_device, args.steps)
    dev_stats = ctx.stats()
    dev_bytes_ms = dev_ms
    if cfg == 2:
        # the same launch on the packed boundary format (2-bit codes in, 4-bit codes + thousandths out): the kernel of
        # that format carries less code and moves a third of the bytes -- `value` is the faster of the two
        for _ in range(warm):
            step_device_packed()
        stream.synchronize()
        dev_packed_ms, _ = timed(step_device_packed, args.steps)
        dev_ms = min(dev_ms, dev_packed_ms)
    kern_ms = dev_ms / args.steps
    for _ in range(2 if cfg == 2 else 1):
        step_host()
    _, bytes_wall_ms = timed(step_host, args.steps)
    e2e_stats = ctx.stats()
    use_packed = cfg == 2          # rRNA-scale structures go beyond the 7 pseudoknot levels of the 4-bit codes: byte format
    if use_packed:
        for _ in range(2):
            step_packed()
        _, e2e_wall_ms = timed(step_packed, args.steps)
        e2e_stats = ctx.stats()
    else:
        e2e_wall_ms = bytes_wall_ms
    sampler.stop_flag = True
    sampler.join(timeout=2)

    # the two legs produced the same structures, stem counts and (after round(x, 3)) scores
    assert np.array_equal(h_dbn.numpy(), d_dbn.cpu().numpy()), "device and host legs disagree (dot-brackets)"
    assert np.array_equal(h_ns.numpy(), d_ns.cpu().numpy()), "device and host legs disagree (stem counts)"
    dsc, hsc = d_sc.cpu().numpy(), h_sc.numpy()
    near = np.round(dsc, 3)
    for k in np.flatnonzero(near != hsc).tolist():                       # rounding ties: Python's round() decides
        assert round(float(dsc[k]), 3) == float(hsc[k]), "device and host legs disagree (scores)"

    # ... and the packed leg the same again: 4-bit codes -> ASCII, thousandths -> the rounded doubles
    if use_packed:
        assert not (p_fl.numpy() & 2).any(), "a structure has more than 7 pseudoknot levels (packed format)"
        assert np.array_equal(_lib.unpack_dbn(p_off.numpy().view(np.uint32), p_nib.numpy()), h_dbn.numpy()[:total]), "packed and byte legs disagree"
        pm = p_milli.numpy().reshape(-1, 2)
        assert np.array_equal(pm[:, 0] / 1000.0, hsc.reshape(-1, 3)[:, 0]) and np.array_equal(pm[:, 1] / 1000.0, hsc.reshape(-1, 3)[:, 1])
        assert np.array_equal(p_ns.numpy().view(np.uint16).astype(np.int32), h_ns.numpy())
        # the device-resident packed leg: the same codes and thousandths (scores next to a rounding tie are left to the host)
        dfl = dp_fl.cpu().numpy()
        assert not (dfl & 2).any()
        assert np.array_equal(_lib.unpack_dbn(p_off.numpy().view(np.uint32), dp_nib.cpu().numpy()), h_dbn.numpy()[:total])
        keep = (dfl & 8) == 0
        assert np.array_equal(dp_milli.cpu().numpy().reshape(-1, 2)[keep], pm[keep])
        assert np.array_equal(dp_ns.cpu().numpy().view(np.uint16), p_ns.numpy().view(np.uint16))

    # the device leg's last step in the byte format (the other legs were checked equal to it above): raw scores,
    # ASCII dot-brackets, stem counts of this rank's batch
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, n, rows={"scores": dsc.reshape(n, 3), "n_stems": d_ns.cpu().numpy()},
                     ragged={"dbn": (off, d_dbn.cpu().numpy())}, ids=idx if strong else None)

    # strong scaling: finished results gathered on rank 0 in input order (host-side, after the timed region)
    gathered = None
    if strong and world > 1:
        from squarna_b200.sharding import gather_to_root
        per_seq, per_pos = gather_to_root(idx, {"scores": hsc.reshape(-1, 3), "n_stems": h_ns.numpy()},
                                          {"dbn": h_dbn.numpy()}, off, goff, rank, world, dist)
        if rank == 0:
            gathered = int(per_seq["n_stems"].shape[0]) == n_global and int(per_pos["dbn"].shape[0]) == int(goff[-1])

    value = n_global / (dev_ms / args.steps / 1e3)
    e2e = n_global / (e2e_wall_ms / args.steps / 1e3)
    nt2_sum = float((lens.astype(np.float64) ** 2).sum())
    if world > 1:
        t = torch.tensor([nt2_sum], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        nt2_sum = float(t[0])
    nt2 = nt2_sum / (dev_ms / args.steps / 1e3)
    if rank == 0:
        peaks = load_peaks()
        peak = float(peaks.get("hbm_gbs", 6650.0))
        abytes = algorithmic_bytes(lens)
        kernel = "k_fast<224>" if cfg == 2 else "k_long<32>"
        tr = load_traffic(kernel)
        traffic, ncu_note = None, {}
        if tr and tr.get("seqs"):
            traffic = int((tr["dram_bytes_read"] + tr["dram_bytes_write"]) * (n / float(tr["seqs"])))
            ncu_note = {k: tr.get(k) for k in ("issue_slots_busy_pct", "ipc_active", "icc_hit_rate_pct",
                                               "warp_instructions_per_sequence", "active_threads_per_warp_instruction")}
            ncu_note.update({"traffic_source": tr.get("source"), "traffic_capture_seqs": tr["seqs"]})
        achieved = abytes / (kern_ms / 1e3) / 1e9
        threads = host_cores()
        skip_cpu = args.no_cpu or world > 1
        if skip_cpu:
            cpu = {"value": 0.0, "unit": "seq/s", "cores": threads, "kind": "reference",
                   "sample": "not run (N > 1 or --no-cpu): see the N = 1 line and the reference arm"}
        elif cfg == 2:
            cpu = cpu_baseline_config2(sym, off, lens, threads)
        else:
            cpu = cpu_baseline_config5(threads, psd, dev_stats, n)
        h2d_bytes = int(sym.nbytes + off.nbytes)
        d2h_bytes = int(total + n * 3 * 8 + n * 4 + n)
        h2d = int((total + 3) // 4 + (n + 1) * 4) if use_packed else h2d_bytes
        d2h = int(total // 2 + n + n * 2 * 4 + n * 2 + n) if use_packed else d2h_bytes
        line = {"metric": METRIC[cfg], "value": value, "unit": "seq/s", "n_gpus": world, "steps": args.steps, "warmup": warm,
                "ms_per_step": dev_ms / args.steps, "higher_is_better": True, "scaling": "strong" if strong else "weak",
                "vs_baseline": None, "dtype": "f64", "data": "synthetic", "nt2_per_s": nt2,
                "config": {"workload": workload, "seqs_per_gpu_per_step": n, "total_nt_per_gpu": total,
                           "l2_policy": "inputs+outputs per step (%.0f MB) exceed the 126 MB L2; no flush" % ((h2d_bytes + d2h_bytes) / 1e6)
                           if cfg == 2 else "every step streams the sequences' candidate lists (GBs) through L2; no flush",
                           "sharding": ("one global batch dealt by length^3, imbalance %.4f, results gathered on rank 0: %s"
                                        % (imbalance, gathered)) if strong else "independent sequences per rank, no collective",
                           "host_cpus_bound_to_gpu_locality": bound},
                "e2e": {"value": e2e, "unit": "seq/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                        "ms_per_step": e2e_wall_ms / args.steps,
                        "kernel_ms_in_step": e2e_stats["kernel_ms"], "launches_per_step": e2e_stats["launches"],
                        "pipeline": "chunked: H2D, kernel and D2H of neighbouring chunks overlap on 4 streams",
                        "call": ("sqrn_fast_predict_packed_host: pinned host buffers in the packed boundary format (2-bit base codes + "
                                 "uint32 offsets in; 4-bit bracket codes + int32 thousandths + uint16 stem counts + flags out)") if use_packed
                                else "sqrn_fast_predict_host: pinned host buffers, byte format (structures of this length exceed the 7 "
                                     "pseudoknot levels a 4-bit code holds)",
                        "byte_format": {"value": n_global / (bytes_wall_ms / args.steps / 1e3), "unit": "seq/s",
                                        "ms_per_step": bytes_wall_ms / args.steps, "h2d_bytes_per_step": h2d_bytes,
                                        "d2h_bytes_per_step": d2h_bytes,
                                        "call": "sqrn_fast_predict_host: ASCII symbols + int64 offsets in, ASCII dot-bracket + "
                                                "3 float64 scores + int32 stem counts out"}},
                "gpu_launches": args.steps * (2 if cfg == 2 else max(int(dev_stats["launches"]), 1) * 2),
                "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                             "traffic": traffic, "peak_source": "MEASURED_PEAKS.json" if peaks else "fallback",
                             "kernel": kernel, "algorithmic_bytes_per_launch": abytes, "kernel_ms": kern_ms,
                             "device_legs_ms": ({"byte_format": dev_bytes_ms / args.steps, "packed_format": dev_packed_ms / args.steps}
                                                if cfg == 2 else None),
                             "optimal_calls_per_step": dev_stats["optimal_calls"],
                             "note": "issue / latency-bound integer path, not HBM-bound: see the ncu figures (profiles/)",
                             **ncu_note},
                "cpu_baseline": cpu,
                "clocks": sampler.summary()}
        if cfg == 2 and world == 1 and not args.no_cli:
            line["e2e_cli"] = cli_leg(sym, off, lens, h_dbn.numpy())
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def cli_leg(sym, off, lens, want_dbn):
    """the CLI surface on the whole batch: Predict(inputfile=<FASTA>, c=fastest, byseq, pl=1) -- text file in, text out
    (the bulk text lane: csrc/sqrn_textio.cpp + the fast lane), checked against the C-ABI leg's dot-brackets"""
    from squarna_b200 import SQUARNA as CLI
    n = len(lens)
    with tempfile.TemporaryDirectory() as tmp:
        inp, outp = os.path.join(tmp, "c2.fa"), os.path.join(tmp, "c2.out")
        # the FASTA text: ">s<k>\n<sequence>\n", built vectorised (1 M entries)
        names = np.char.add(np.char.add(">s", np.arange(n).astype(str)), "\n").astype("S")
        with open(inp, "wb") as f:
            parts = []
            for b in range(n):
                parts.append(names[b])
                parts.append(sym[int(off[b]):int(off[b + 1])].tobytes())
                parts.append(b"\n")
            f.write(b"".join(parts))
        best = None
        for _ in range(2):                                   # the second run has the page cache and the contexts warm
            with open(outp, "w") as sink:
                t0 = time.perf_counter()
                CLI.Predict(inputfile=inp, configfile="fastest", byseq=True, poollim=1, write_to=sink)
                sink.flush()
                dt = time.perf_counter() - t0
            best = dt if best is None else min(best, dt)
        # parity of the text with the C-ABI leg: line 4 of every 6-line block is the consensus dot-bracket
        ok = True
        with open(outp, "rb") as f:
            for b, block in zip(range(2000), iter(lambda: [f.readline() for _ in range(6)], None)):
                cons = block[3].split(b"\t")[0]
                if cons != want_dbn[int(off[b]):int(off[b + 1])].tobytes():
                    ok = False
        return {"value": n / best, "unit": "seq/s", "seconds": best, "input_bytes": os.path.getsize(inp),
                "output_bytes": os.path.getsize(outp), "matches_c_abi_leg_first_2000": ok,
                "call": "Predict(inputfile=<FASTA of %d sequences>, configfile='fastest', byseq=True, poollim=1, write_to=<file>)" % n}


def cpu_baseline_config5(threads, psd, dev_stats, n):
    """The reference needs about an hour per sequence at these lengths (O(N^3); BASELINE.md: 293 s at 1000 nt), so
    what is timed is bounded and labelled: the C port on `threads` sequences of 2900 nt (the CHEAPEST length of the
    workload: an upper bound of the CPU rate), and the Python reference on the same number of 2900-nt sequences with
    maxstemnum=1 (ONE greedy step), extrapolated by the steps per sequence the GPU run counted."""
    k = max(1, min(threads, 32))
    sym, off, lens = workloads.config5(k, SEED + 1, lo=2900, hi=2900)
    rate, nt2, dt = cpu_oracle_rate(sym, off, lens, k, threads, psd)
    out = {"value": rate, "unit": "seq/s", "cores": threads, "kind": "port", "nt2_per_s": nt2, "cpu_model": cpu_model(),
           "sample": "%d sequences of 2900 nt (the shortest of the workload: an UPPER bound of the CPU rate), %.1f s, "
                     "oracle/sqrn_oracle.c on %d threads" % (k, dt, threads)}
    steps_per_seq = dev_stats["optimal_calls"] / max(n, 1)
    with tempfile.TemporaryDirectory() as tmp:
        inp = os.path.join(tmp, "ref_c5.fa")
        write_fasta(inp, sym, off, k)
        secs, _ = run_python_reference(inp, dict(configfile="1000nobpp", byseq=True, poollim=1, threads=threads,
                                                 algorithms="G", maxstemnum=1), timeout=1200)
    if secs is not None:
        per_step = secs / (k / min(k, threads))
        out["reference"] = {"kind": "reference", "seconds_for_one_greedy_step": per_step, "cores": threads,
                            "extrapolated_seq_per_s": min(k, threads) / (per_step * max(steps_per_seq, 1.0)),
                            "sample": "the reference's own Predict(byseq, pl=1, c=1000nobpp, algo=G, msn=1) on %d sequences of 2900 nt: "
                                      "%.1f s = BPMatrix + ONE greedy step each; a full prediction takes ~%.0f steps (counted by "
                                      "the GPU run), so the rate is EXTRAPOLATED, not measured" % (k, secs, steps_per_seq)}
    return out


# ------------------------------------------------------------------------------ config 3: pool rounds
def bench_config3(args, rank, world, local):
    import torch
    import torch.distributed as dist
    from squarna_b200 import SQRNdbnseq as S
    from squarna_b200.sharding import shard_plan, plan_imbalance

    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    n_global = args.seqs
    entries = workloads.config3(n_global, SEED)
    glens = np.array([len(e[0]) for e in entries])
    plan = shard_plan(glens, world, 3.0)
    idx = plan[rank]
    mine = [entries[k] for k in idx.tolist()]
    lens = glens[idx]
    groups = {}
    for e in mine:
        groups.setdefault(workloads.config3_conf(len(e[0])), []).append((e[0], e[1], e[2], None))
    psets = {c: conf_gsets(c) for c in groups}
    ctx = S.get_context(local)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # warm-up: three passes over a small prefix of every group (module load, parameter digests, scratch buffers)
    for _ in range(max(args.warmup, 3)):
        for c, es in groups.items():
            S.predict_many(es[:8], psets[c], poollim=100, device=local)
    # ... and one full-size pass (the library sizes its device scratch -- base lists, candidate lists -- on first use)
    for c, es in groups.items():
        S.predict_many(es, psets[c], poollim=100, device=local)
    sampler = ClockSampler(local)
    sampler.start()
    # e2e leg: predict_many from Python strings (prepare, pack, C-ABI call with host buffers, result assembly)
    barrier()
    t0 = time.perf_counter()
    kern_ms, launches, calls, structs = 0.0, 0, 0, 0
    results = {}
    for _ in range(args.steps):
        for c, es in groups.items():
            results[c] = S.predict_many(es, psets[c], poollim=100, device=local)
            st = ctx.stats()
            kern_ms += st["kernel_ms"]; launches += st["launches"]; calls += st["optimal_calls"]
            structs += sum(len(r[1]) for r in results[c])
    barrier()
    e2e_s = (time.perf_counter() - t0) / args.steps
    if args.dump_outputs and rank == 0:
        # the last predict_many of every length class, back in this rank's entry order: consensus, the structures of
        # each entry back to back, their three scores each
        preds = [None] * len(mine)
        for c in groups:
            for k, r in zip([k for k, e in enumerate(mine) if workloads.config3_conf(len(e[0])) == c], results[c]):
                preds[k] = r

        def offsets(parts):
            o = np.zeros(len(parts) + 1, dtype=np.int64)
            np.cumsum([len(p) for p in parts], out=o[1:])
            return o

        cons = [p[0].encode() for p in preds]
        dbns = [b"".join(s[0].encode() for s in p[1]) for p in preds]
        scores = [[float(x) for s in p[1] for x in s[1]] for p in preds]
        dump_outputs(args.dump_outputs, len(mine), rows={"n_structures": np.array([len(p[1]) for p in preds])},
                     ragged={"consensus": (offsets(cons), np.frombuffer(b"".join(cons), np.uint8)),
                             "structures": (offsets(dbns), np.frombuffer(b"".join(dbns), np.uint8)),
                             "scores": (offsets(scores), np.array([x for s in scores for x in s], np.float64))}, ids=idx)
    # value leg: the C-ABI batch call alone on prepared batches (no Python preparation / result assembly)
    batches = []
    for c, es in groups.items():
        preps = [S._prepare(*e) for e in es]
        for comp in (False, True):
            ii = [k for k, p in enumerate(preps) if p.compensated == comp]
            if ii:
                batches.append((c, S._make_batch(preps, ii, comp, None, False, hardrest=False, rankbydiff=False, poollim=100,
                                                 conslim=1, rankby=(0, 2, 1), priority_mask=0)))
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        for c, b in batches:
            ctx.predict_batch_flat(psets[c], b)          # (the flat arrays the C call filled: no per-structure Python objects)
    barrier()
    abi_s = (time.perf_counter() - t0) / args.steps
    sampler.stop_flag = True
    sampler.join(timeout=2)
    t = torch.tensor([e2e_s, abi_s, kern_ms / args.steps], dtype=torch.float64, device="cuda")
    tot = torch.tensor([float(launches), float(calls), float(structs), float((lens.astype(np.float64) ** 2).sum())],
                       dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dist.all_reduce(tot, op=dist.ReduceOp.SUM)
    e2e_s, abi_s, kms = (float(x) for x in t)
    if rank == 0:
        peaks = load_peaks()
        peak = float(peaks.get("hbm_gbs", 6650.0))
        s_mean = float(tot[2]) / args.steps / max(n_global, 1)
        abytes = workloads.algorithmic_bytes(glens, n_structs=min(5.0, s_mean), reacts=True, restraints=True)
        achieved = abytes / max(kms / 1e3, 1e-9) / 1e9
        threads = host_cores()
        cpu = {"value": 0.0, "unit": "seq/s", "cores": threads, "kind": "reference", "sample": "not run (N > 1 or --no-cpu)"}
        if not (args.no_cpu or world > 1):
            cpu = cpu_baseline_config3(entries, threads)
        cap = "" if n_global >= 100000 else " (CAPPED at %d of the 100 000 sequences)" % n_global
        line = {"metric": METRIC[3], "value": n_global / abi_s, "unit": "seq/s", "n_gpus": world, "steps": args.steps,
                "warmup": max(args.warmup, 3), "ms_per_step": abi_s * 1e3, "higher_is_better": True, "scaling": "strong",
                "vs_baseline": None, "dtype": "f64", "data": "synthetic", "nt2_per_s": float(tot[3]) / abi_s,
                "config": {"workload": "config3: %d synthetic RNAs%s, len U{300..1500}, rf=26 reactivity letters (3%% '?'), restraints "
                                       "(5%% '_', 1%% '/', 1%% '\\', 0-2 planted stems), G sets by length (greedynobpp / 500nobpp / "
                                       "1000nobpp), pl=100" % (n_global, cap),
                           "warmup_note": "warm-up: three passes over an 8-sequence prefix of every length class, then one full-size pass",
                           "sharding": "one global batch dealt by length^3, imbalance %.4f" % plan_imbalance(glens, plan, 3.0),
                           "l2_policy": "inputs larger than L2 per pass; no flush"},
                "e2e": {"value": n_global / e2e_s, "unit": "seq/s", "ms_per_step": e2e_s * 1e3,
                        "h2d_bytes_per_step": int(sum(len(e[0]) * 4 + 8 for e in mine)),
                        "d2h_bytes_per_step": int(float(tot[2]) / args.steps / world * (float(lens.mean()) + 40)),
                        "call": "squarna_b200.SQRNdbnseq.predict_many(entries, paramsets, poollim=100) per length class"},
                "gpu_launches": int(float(tot[0])),
                "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                             "traffic": None, "peak_source": "MEASURED_PEAKS.json" if peaks else "fallback",
                             "kernel": "k_work<8> (MODE_STEP pool rounds)", "algorithmic_bytes_per_launch": abytes,
                             "kernel_ms": kms, "optimal_calls_per_step": float(tot[1]) / args.steps,
                             "structures_per_sequence": s_mean},
                "cpu_baseline": cpu, "clocks": sampler.summary()}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def cpu_baseline_config3(entries, threads):
    """the Python reference on a BOUNDED sample: the `threads` sequences nearest to 300 nt, one per worker -- the SHORT end
    of the workload.  Measured: one 302-nt sequence of this workload with pl=100 takes the reference 83 s on one core; its
    cost grows faster than N^3 (500-600 nt: more than 10 minutes for 8 sequences on 16 threads), so no bench run can afford
    the stated length mix and the rate reported here flatters the reference by orders of magnitude.
    Predict(byseq, algo=G, pl=100) with the reference's own autoconfig replaced by the bpp-free G set of that length."""
    lens = np.array([len(e[0]) for e in entries])
    pick = np.argsort(np.abs(lens - 300), kind="stable")[:max(1, min(threads, 32))].tolist()
    out = {"unit": "seq/s", "cores": threads, "kind": "reference", "cpu_model": cpu_model()}
    with tempfile.TemporaryDirectory() as tmp:
        inp = os.path.join(tmp, "ref_c3_greedynobpp.fa")
        with open(inp, "w") as f:
            for k in pick:
                f.write(">s%d\n%s\n%s\n%s\n" % (k, entries[k][0], entries[k][1], entries[k][2]))
        budget = 420
        try:
            secs, _ = run_python_reference(inp, dict(configfile="greedynobpp", byseq=True, poollim=100, threads=threads, algorithms="G",
                                                     inputformat="qtr", reactformat=26), timeout=budget)
        except subprocess.TimeoutExpired:
            out.update({"value": len(pick) / float(budget), "sample": "UPPER bound: the reference did not finish %d sequences of "
                        "%d-%d nt (Predict(byseq, algo=G, pl=100, greedynobpp)) within %d s" % (len(pick), int(lens[pick].min()),
                                                                                                 int(lens[pick].max()), budget)})
            return out
    if secs is None:
        out.update({"value": 0.0, "sample": "Python reference unavailable"})
        return out
    out.update({"value": len(pick) / secs, "sample": "%d sequences of %d-%d nt (the short end of the 300-1500 nt workload; longer ones "
                "are out of reach: see the docstring), the reference's own Predict(byseq, algo=G, pl=100, greedynobpp, threads=%d): %.1f s"
                % (len(pick), int(lens[pick].min()), int(lens[pick].max()), threads, secs)})
    return out


# ------------------------------------------------------------------------------ config 4: alignment mode
def bench_config4(args, rank, world, local):
    """BASELINE config 4: alignment mode on a synthetic 2000-sequence x 400-column alignment (workloads.config4).
    `value`: rows / second of step 1 through the C ABI (sqrn_stem_matrix_batch on a prepared batch, twice -- the second
    iteration feeds the first structure back as restraints): stems, the sequence-ordered sum and the ranking of the
    conserved cells on the device.  `e2e`: the whole alignment mode through the unchanged Predict() surface (input file in,
    text out: step 1, step 2 = stem-matrix-weighted single-sequence predictions of every row, consensus on the host)."""
    import io
    import torch
    from squarna_b200 import SQRNdbnali as A
    from squarna_b200 import SQRNdbnseq as S
    from squarna_b200 import SQUARNA as CLI
    if rank != 0:
        return                                                     # one alignment: the path does not shard at step 1
    torch.cuda.set_device(local)
    n_rows = args.seqs
    rows, ref = workloads.config4(n_rows, 300, 400)
    L = len(rows[0])
    names, psets = CLI.ParseConfig(os.path.join(os.path.dirname(os.path.abspath(CLI.__file__)), "ali.conf"))
    first = psets[0]
    os.environ["SQRN_DEVICES"] = str(local)
    ctx = S.get_context(local)
    entries = [(r, None, None) for r in rows]
    thr = first["minbpscore"] * n_rows

    def step1():
        mat, cells = A._yield_many(entries, first["bpweights"], False, first["minlen"], first["minbpscore"], device=local, matrix=(L, thr))
        dbn = A.MatrixToDBNs(mat, first["minbpscore"], n_rows, cells=cells)[0]
        ent2 = [(r, None, dbn) for r in rows]
        mat2, cells2 = A._yield_many(ent2, first["bpweights"], False, first["minlen"], first["minbpscore"], device=local, matrix=(L, thr))
        return dbn, mat2, cells2

    for _ in range(max(args.warmup, 3)):
        dbn1 = step1()
    sampler = ClockSampler(local)
    sampler.start()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    kms, launches = 0.0, 0
    for _ in range(args.steps):
        dbn, mat, cells = step1()
        st = ctx.stats()
        kms += st["kernel_ms"]; launches += st["launches"]
    torch.cuda.synchronize()
    step1_s = (time.perf_counter() - t0) / args.steps
    if args.dump_outputs:
        # one item, the alignment: the first iteration's structure, the second iteration's stem matrix and the cells
        # MatrixToDBNs would walk (empty when there are too many for the device ranking)
        cells = np.zeros(0, np.int32) if cells is None else cells
        dump_outputs(args.dump_outputs, 1, rows={"stem_matrix": mat[None]},
                     ragged={"dbn": ([0, L], np.frombuffer(dbn.encode(), np.uint8)), "cells": ([0, len(cells)], cells)})
    with tempfile.TemporaryDirectory() as tmp:
        path = os.path.join(tmp, "c4.afa")
        with open(path, "w") as f:
            f.write(workloads.config4_text(rows, ref))
        buf = io.StringIO()
        CLI.Predict(inputfile=path, alignment=True, write_to=buf)                  # warm-up of the step-2 kernels
        t0 = time.perf_counter()
        for _ in range(args.steps):
            buf = io.StringIO()
            CLI.Predict(inputfile=path, alignment=True, write_to=buf)
        e2e_s = (time.perf_counter() - t0) / args.steps
    sampler.stop_flag = True
    sampler.join(timeout=2)
    text = buf.getvalue()
    step3 = [ln for ln in text.split("\n") if "Step-3" in ln]
    peaks = load_peaks()
    peak = float(peaks.get("hbm_gbs", 6650.0))
    lens = np.array([len(r) - r.count("-") for r in rows])
    abytes = workloads.algorithmic_bytes(lens) + 8 * L * L
    achieved = abytes / max(step1_s, 1e-9) / 1e9
    line = {"metric": "alignment rows/sec (SQRNdbnali step 1; e2e: the whole alignment mode)", "value": n_rows / step1_s, "unit": "seq/s",
            "n_gpus": 1, "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": step1_s * 1e3, "higher_is_better": True,
            "scaling": "replicas only", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": "config4: alignment mode on a synthetic %d-sequence x %d-column alignment (ancestor with planted "
                                   "hairpins, 10%% substitutions, 2%% deletions, shared gap columns), ali.conf" % (n_rows, L),
                       "l2_policy": "the stems of all rows (tens of MB) are re-read per row band through L2; no flush"},
            "e2e": {"value": n_rows / e2e_s, "unit": "seq/s", "ms_per_step": e2e_s * 1e3,
                    "h2d_bytes_per_step": int(3 * (lens.sum() * 5 + 8 * n_rows)), "d2h_bytes_per_step": int(2 * 8 * L * L + n_rows * L * 2),
                    "call": "squarna_b200.SQUARNA.Predict(inputfile=<alignment>, alignment=True): steps 1-3, text out",
                    "step3_line": step3[0] if step3 else None},
            "gpu_launches": int(launches),
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": None,
                         "peak_source": "MEASURED_PEAKS.json" if peaks else "fallback", "kernel": "k_work<8> (MODE_YIELD) + k_stem_matrix",
                         "algorithmic_bytes_per_launch": abytes, "kernel_ms": kms / args.steps,
                         "note": "host-bound: the Python preparation of the rows and the text dominate (DESIGN.md)"},
            "cpu_baseline": {"value": 0.0, "unit": "seq/s", "cores": host_cores(), "kind": "reference", "sample": "not run (see BASELINE.md: "
                             "the reference needs minutes per alignment of this size)"},
            "clocks": sampler.summary()}
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--config", type=int, default=2, choices=[2, 3, 4, 5])
    ap.add_argument("--seqs", type=int, default=None,
                    help="config 2: sequences per GPU per step (default 1 000 000); configs 3 / 5: sequences of the global batch")
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg (profiling runs)")
    ap.add_argument("--no-cli", action="store_true", help="skip the CLI-level end-to-end leg of config 2")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the timed path returned in its last step as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps is None:
        args.steps = {2: 20, 5: 3, 3: 1, 4: 3}[args.config]
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes this project's outputs; the reference arm has none")
    if args.seqs is None:
        args.seqs = {2: 1_000_000, 5: 10_000, 3: 100_000 if args.gpus >= 8 else 20_000, 4: 2000}[args.config]
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank)
        return
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback)")
    if args.config == 3:
        bench_config3(args, rank, world, local)
    elif args.config == 4:
        bench_config4(args, rank, world, local)
    else:
        bench_fast(args, rank, world, local)


if __name__ == "__main__":
    main()
