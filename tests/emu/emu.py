"""ctypes front-end of tests/emu/sqrn_emu.cpp (TEST INFRASTRUCTURE, see that file)."""
import ctypes as C
import os
import subprocess

import numpy as np

from squarna_b200._abi import ParamSet, pack_sequences, ptr

_HERE = os.path.dirname(os.path.abspath(__file__))
_SO = os.path.join(_HERE, "_build", "libsqrn_emu.so")
_ROOT = os.path.dirname(os.path.dirname(_HERE))
MODE_TAIL, MODE_STEP, MODE_YIELD = 0, 1, 2


def build():
    srcs = [os.path.join(_HERE, "sqrn_emu.cpp"),
            os.path.join(_ROOT, "squarna_b200", "csrc", "sqrn_device.cuh"),
            os.path.join(_ROOT, "squarna_b200", "csrc", "sqrn_params.h")]
    if not os.path.exists(_SO) or any(os.path.getmtime(s) > os.path.getmtime(_SO) for s in srcs):
        os.makedirs(os.path.dirname(_SO), exist_ok=True)
        # parallel test workers may all build: each writes its own file and renames it into place, so that no
        # worker loads a library another one is still writing
        tmp = "%s.%d.tmp" % (_SO, os.getpid())
        subprocess.check_call(["g++", "-O2", "-g", "-std=c++17", "-ffp-contract=off", "-fPIC", "-shared",
                               "-Wno-unknown-pragmas", "-o", tmp, srcs[0], "-lm"])
        os.replace(tmp, _SO)
    return _SO


_lib = None


def lib():
    global _lib
    if _lib is None:
        _lib = C.CDLL(build())
        _lib.emu_run.argtypes = [C.POINTER(ParamSet), C.c_int64] + [C.c_void_p] * 4 + [C.c_int, C.c_int] + \
            [C.c_void_p] * 4 + [C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_int] + [C.c_void_p] * 13 + \
            [C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_int]
        _lib.emu_pyround3.restype = C.c_double
        _lib.emu_persist_steps.restype = C.c_long
        _lib.emu_gl_rebuilds.restype = C.c_long
        _lib.emu_base_sweeps.restype = C.c_long
        _lib.emu_gl_catchups.restype = C.c_long
        _lib.emu_gl_set_rebuild.argtypes = [C.c_int]
        _lib.emu_pyround3.argtypes = [C.c_double]
    return _lib


def run(paramset, seqs, mode=MODE_TAIL, react_codes=None, react_values=None, react_comp=False,
        restr_class=None, rbps=None, smat=None, cols=None, interchainonly=False,
        item_seq=None, init_stems=None, item_subopt=None, ccap=128, stem_cap=None, region_mode=0, flavour=0,
        pcap=0):
    """seqs: list of normalised ungapped strings.  react_codes/restr_class: list of per-sequence uint8
    arrays; rbps: list of per-sequence (n,2) arrays; init_stems: list per item of (i,j,len) lists.
    Returns dict of numpy outputs."""
    L = lib()
    sym, off = pack_sequences(seqs)
    nseq = len(seqs)
    cat = lambda lst, dt: (np.concatenate([np.asarray(x, dtype=dt).ravel() for x in lst]) if sum(len(x) for x in lst) else np.zeros(1, dt))
    rcode = cat(react_codes, np.uint16) if react_codes is not None else None
    rvals = np.ascontiguousarray(react_values, dtype=np.float64) if react_values is not None else None
    rcl = cat(restr_class, np.uint8) if restr_class is not None else None
    rb_off = rb = None
    if rbps is not None:
        rb_off = np.zeros(nseq + 1, dtype=np.int64)
        np.cumsum([len(x) for x in rbps], out=rb_off[1:])
        rb = cat(rbps, np.int32)
    sm = np.ascontiguousarray(smat, dtype=np.float64) if smat is not None else None
    cl = cat(cols, np.int32) if cols is not None else None
    n_items = len(item_seq) if item_seq is not None else nseq
    iseq = np.ascontiguousarray(item_seq, dtype=np.int32) if item_seq is not None else None
    ioff = ist = None
    if init_stems is not None:
        ioff = np.zeros(n_items + 1, dtype=np.int64)
        np.cumsum([len(x) for x in init_stems], out=ioff[1:])
        ist = cat(init_stems, np.int32)
    isub = np.ascontiguousarray(item_subopt, dtype=np.float64) if item_subopt is not None else None
    lens = np.diff(off)
    ilen = lens[iseq] if iseq is not None else lens
    if stem_cap is None:
        stem_cap = (ilen // 2 + 1) if mode != MODE_YIELD else (ilen * ilen // 4 + 8)
    out_off = np.zeros(n_items + 1, dtype=np.int64)
    np.cumsum(np.broadcast_to(stem_cap, (n_items,)), out=out_off[1:])
    out_stems = np.zeros((max(int(out_off[-1]), 1), 3), dtype=np.int32)
    out_n = np.zeros(max(n_items, 1), dtype=np.int32)
    out_fin = np.zeros(max(int(out_off[-1]), 1), dtype=np.float64)
    out_raw = np.zeros((max(n_items, 1), 3), dtype=np.float64)
    out_flags = np.zeros(max(n_items, 1), dtype=np.uint8)
    dbn_off = np.zeros(n_items + 1, dtype=np.int64)
    np.cumsum(ilen, out=dbn_off[1:])
    dbn_a = np.zeros(max(int(dbn_off[-1]), 1), dtype=np.uint8)
    dbn_c = np.zeros(max(int(dbn_off[-1]), 1), dtype=np.int8)
    ncalls = C.c_ulonglong(0)
    ps = ParamSet.from_dict(paramset)
    rc = L.emu_run(C.byref(ps), nseq, ptr(off), ptr(sym), ptr(rcode), ptr(rvals),
                   0 if rvals is None else len(rvals), int(react_comp), ptr(rcl), ptr(rb_off), ptr(rb),
                   ptr(sm), 0 if sm is None else sm.shape[0], ptr(cl), int(interchainonly),
                   mode, n_items, ptr(iseq), ptr(ioff), ptr(ist), ptr(isub),
                   ptr(out_off), ptr(out_stems), ptr(out_n), ptr(out_fin), ptr(out_raw), ptr(out_flags),
                   ptr(dbn_off), ptr(dbn_a), ptr(dbn_c), int(ccap), C.byref(ncalls), int(region_mode), int(flavour), int(pcap))
    assert rc == 0
    return dict(off=out_off, stems=out_stems, n=out_n[:n_items], fin=out_fin, raw=out_raw[:n_items],
                flags=out_flags[:n_items], dbn_off=dbn_off, dbn_ascii=dbn_a, dbn_code=dbn_c,
                ncalls=ncalls.value)
