"""Command line and Python API front-end: the surface of the reference's
SQUARNA.py (ParseConfig, the input parsers, Predict with all its keyword
synonyms, Main) over the GPU hot path.

Host-only code: parsing and option checking.  Line numbers cited as cli.py:N are
/root/reference/src/SQUARNA/SQUARNA.py.

Behavioural differences from the reference, all outside the hot path:
  * `threads` / `byseq` only chose a multiprocessing layout in the reference and
    never changed the output; here every mode batches entries into GPU calls and
    prints in input order.
  * parameter sets with `bpp != 0` (ViennaRNA, not installed: parity unpinned) and the
    rfam/g4/rbp restraint discovery (external binaries / network) raise NotImplementedError.
    Nussinov / Hungarian / Edmonds parameter sets build on GPU-enumerated stems, and the three builders run on the
    device too.
"""
import os
import sys

from .SQRNdbnseq import GAPS, SEPS, ProcessReacts, ReactDict, RunSQRNdbnseqBatch

_MANDATORY = ("algorithms", "bpweights", "suboptmax", "suboptmin", "suboptsteps", "minlen", "minbpscore",
              "minfinscorefactor", "distcoef", "bracketweight", "orderpenalty", "loopbonus", "maxstemnum")

BATCH_ENTRIES = 8192        # entries per GPU call when streaming an input file


def ParseConfig(configfile):
    """.conf file -> (names, paramsets) (cli.py:15-77).  Sets after the first start
    as copies of the FIRST set; `bpweights` is a dict, `algorithms` a set,
    everything else a float."""
    names, paramsets = [], []
    current = None
    with open(configfile) as fh:
        for raw in fh:
            line = raw.split('#', 1)[0].strip()
            if not line:
                continue
            if line.startswith('>'):
                names.append(line[1:])
                if current is not None:
                    paramsets.append(current)
                    current = dict(paramsets[0])
                else:
                    current = {}
                continue
            key, val = line.split(maxsplit=1)
            if key == "bpweights":
                weights = {}
                for item in val.split(','):
                    k, v = item.strip().split('=')
                    weights[k] = float(v)
                current[key] = weights
            elif key == "algorithms":
                current[key] = set(val.split(','))
            else:
                current[key] = float(val)
    paramsets.append(current)
    missing = [k for k in _MANDATORY if k not in paramsets[0]]
    if missing:
        raise ValueError("Missing some of the parameters in the first parameter set of the config file: {}"
                         .format(', '.join(missing)))
    return names, paramsets


# ------------------------------------------------------------------ parsers
def _resolve_reacts(text, n, M, B):
    """reactivity line: n floats or an n-character code string (cli.py:144-149)"""
    if len(text) != n:
        return ProcessReacts(list(map(float, text.split())), M=M, B=B)
    return ProcessReacts([ReactDict[ch] for ch in text], M=M, B=B)


def ParseDefaultInput(inputname, inputformat, returndefaults=False, ignore=False, M=1.8, B=-0.6):
    """SQUARNA's fasta-like format (cli.py:80-203): yields (name, seq, reacts, restraints,
    reference); lines before the first '>' are defaults; with returndefaults only those."""
    q_ind = inputformat.index('q')
    t_ind, r_ind, f_ind = (inputformat.find(ch) for ch in "trf")
    defaults = {"t": None, "r": None, "f": None}
    warned = set()
    resolved = {}

    def pick(data, ind, first_token):
        if ind <= 0 or ind >= len(data) or not data[ind]:       # find() > 0: position 0 is ignored (cli.py:102-104)
            return None
        return data[ind].split()[0] if first_token else data[ind]

    def default_for(kind, label, n):
        d = defaults[kind]
        if not d:
            return None
        ok = (len(d) == n or len(d.split()) == n) if kind == "t" else len(d) == n
        if ok:
            return d
        if kind not in warned:
            warned.add(kind)
            msg = "WARNING: some sequences differ in length from the default {} line".format(label)
            if ignore:
                print(msg, file=sys.stderr)
            else:
                raise ValueError(msg + " [Switch on the iw/ignore parameter to proceed anyway]")
        return None

    def finish(name, data):
        data = list(data) + [None] * (len(inputformat) - len(data))
        sequence = data[q_ind].split()[0]
        n = len(sequence)
        reactivities = data[t_ind] if t_ind > 0 else None
        restraints = pick(data, r_ind, True)
        reference = pick(data, f_ind, True)
        if not reactivities:
            reactivities = default_for("t", "reactivities", n)
        if not restraints:
            restraints = default_for("r", "restraints", n)
        if not reference:
            reference = default_for("f", "reference", n)
        try:
            if reactivities:
                key = (reactivities, n)                 # the default line is shared by every entry: processed once
                if key not in resolved:
                    if len(resolved) > 64:
                        resolved.clear()
                    resolved[key] = _resolve_reacts(reactivities, n, M, B)
                reactivities = list(resolved[key])
            assert not reactivities or len(reactivities) == n
        except Exception:
            raise ValueError('Inappropriate reactivities line for entry "{}":\n {}'.format(name[1:], reactivities))
        assert not restraints or len(restraints) == n, \
            'Inappropriate restraints line for entry "{}":\n {}'.format(name[1:], restraints)
        assert not reference or len(reference) == n, \
            'Inappropriate reference line for entry "{}":\n {}'.format(name[1:], reference)
        return name, sequence, reactivities, restraints, reference

    name, data = None, []
    with open(inputname) as fh:
        for line in fh:
            if line.startswith('>'):
                if name:
                    yield finish(name, data)
                else:
                    head = list(data) + [None] * (len(inputformat) - 1 - len(data))
                    head.insert(q_ind, None)
                    defaults["t"] = head[t_ind] if t_ind > 0 else None
                    defaults["r"] = head[r_ind] if r_ind > 0 else None
                    defaults["f"] = head[f_ind] if f_ind > 0 else None
                    if returndefaults:
                        yield (defaults["t"], defaults["r"], defaults["f"])
                        return
                name, data = line.strip(), []
            else:
                data.append(line.strip())
    if name:
        yield finish(name, data)


def GuessFormat(inp):
    """default / fasta / stockholm / clustal, and whether there is a single entry (cli.py:206-236)"""
    with open(inp) as fh:
        first = fh.readline()
        if first.startswith('#') and "STOCKHOLM" in first:
            return "stockholm", 0
        if first.startswith("CLUSTAL"):
            return "clustal", 0
        entries = 1 if first.startswith(">") else 0
        seqlines = 0
        for line in fh:
            if line.startswith(">"):
                entries += 1
                continue
            if sum(1 for ch in line.upper() if ch in "ACGUT") > len(line) / 2:
                seqlines += 1
            if seqlines > 1000:
                break
        if seqlines > entries and entries > 0:
            return "fasta", (entries == 1)
    return "default", (entries == 1)


def ParseFasta(inp, returndefaults=False):
    """plain FASTA, sequences may span several lines (cli.py:239-256)"""
    if returndefaults:
        yield (None, None, None)
        return
    name, chunks = None, []
    with open(inp) as fh:
        for line in fh:
            if line.startswith('>'):
                if name:
                    yield (name, ''.join(chunks), None, None, None)
                name, chunks = line.strip(), []
            elif line.strip():
                chunks.append(line.strip())
    yield (name, ''.join(chunks), None, None, None)


def ReadStockholm(stkfile):
    """-> headers, seqnames, seqdict, gcnames, gcdict (cli.py:259-312)"""
    try:
        with open(stkfile) as fh:
            lines = fh.readlines()
    except UnicodeDecodeError:
        with open(stkfile, encoding="iso8859-15") as fh:
            lines = fh.readlines()
    headers, seqnames, seqdict, gcnames, gcdict = [], [], {}, [], {}
    for line in lines:
        if line.startswith('#=GC '):
            parts = line.strip().split()
            key, target, order = ' '.join(parts[1:-1]), gcdict, gcnames
        elif line.startswith('#'):
            headers.append(line)
            continue
        elif line.startswith('//') or not line.strip():
            continue
        else:
            parts = line.strip().split()
            key, target, order = ' '.join(parts[:-1]), seqdict, seqnames
        if key not in target:
            order.append(key)
            target[key] = parts[-1]
        else:
            target[key] += parts[-1]
    headers = [h for h in headers if not h.startswith("#=GF SQ")] + [h for h in headers if h.startswith("#=GF SQ")]
    return headers, seqnames, seqdict, gcnames, gcdict


def ParseStockholm(inp, returndefaults=False):
    """SS_cons becomes the default reference (cli.py:315-327)"""
    _, seqnames, seqdict, gcnames, gcdict = ReadStockholm(inp)
    sscons = gcdict["SS_cons"] if "SS_cons" in gcnames else None
    if returndefaults:
        return None, None, sscons
    return [('>' + n, seqdict[n], None, None, sscons) for n in seqnames], len(seqnames) == 1


def ParseClustal(inp, returndefaults=False):
    if returndefaults:
        return None, None, None
    names, seqs = [], {}
    with open(inp) as fh:
        for line in fh:
            if line.strip() and not line.startswith("CLUSTAL") and not line.startswith(' '):
                name, chunk = line.strip().split()
                if name not in seqs:
                    names.append(name)
                    seqs[name] = ''
                seqs[name] += chunk
    return [('>' + n, seqs[n], None, None, None) for n in names], len(names) == 1


def ParseSeq(inputseq, returndefaults, inputrestr):
    if returndefaults:
        return None, None, None
    return [('>inputseq', inputseq, None, inputrestr, None)]


def ParseInput(inputseq, inputname, inputformat, returndefaults=False, fmt="unknown", ignore=False,
               inputrestr=None, M=1.8, B=-0.6):
    """parser selector (cli.py:357-390)"""
    if inputseq:
        return ParseSeq(inputseq, returndefaults, inputrestr), fmt, True
    single = None
    if fmt == "unknown":
        fmt, single = GuessFormat(inputname)
        if fmt != "default":
            print("Non-default input file format is recognized: {}".format(fmt.upper()))
    if fmt == "default":
        if returndefaults:
            return next(ParseDefaultInput(inputname, inputformat, True, M=M, B=B)), fmt
        return ParseDefaultInput(inputname, inputformat, False, ignore=ignore, M=M, B=B), fmt, single
    if fmt == "fasta":
        if returndefaults:
            return next(ParseFasta(inputname, True)), fmt
        return ParseFasta(inputname, False), fmt, single
    parser = ParseStockholm if fmt == "stockholm" else ParseClustal
    if returndefaults:
        return parser(inputname, True), fmt
    parsed, single = parser(inputname, False)
    return parsed, fmt, single


# ------------------------------------------------------------------ Predict
_SYNONYMS = (("i", "inputfile"), ("ff", "fileformat"), ("config", "configfile"), ("c", "configfile"),
             ("seq", "inputseq"), ("s", "inputseq"), ("ali", "alignment"), ("a", "alignment"),
             ("algorithm", "algorithms"), ("algo", "algorithms"), ("rb", "rankby"), ("freqlim", "freqlimit"),
             ("fl", "freqlimit"), ("levlim", "levellimit"), ("ll", "levellimit"), ("tl", "toplim"),
             ("ol", "outplim"), ("cl", "conslim"), ("pl", "poollim"), ("pr", "priority"), ("s3", "step3"),
             ("msn", "maxstemnum"), ("rf", "reactformat"), ("eo", "evalonly"), ("hr", "hardrest"),
             ("ico", "interchainonly"), ("ignore", "ignorewarn"), ("iw", "ignorewarn"), ("t", "threads"),
             ("bs", "byseq"), ("v", "verbose"))


def _positive_int(value, label):
    try:
        value = int(float(value))
        assert value > 0
    except Exception:
        raise ValueError("Inappropriate {} value (positive integer): {}".format(label, value))
    return value


def Predict(inputfile=None, fileformat="unknown", inputseq=None,
            configfile=None, inputformat="qtrf", maxstemnum=None,
            threads=os.cpu_count(), byseq=False, algorithms='',
            entropy=False, rankby="r", evalonly=False, hardrest=False,
            interchainonly=False, toplim=5, outplim=None, conslim=1,
            poollim=1000, reactformat=3, alignment=False, levellimit=None,
            freqlimit=0.35, verbose=False, step3="u", ignorewarn=False,
            HOME_DIR=None, write_to=None, priority=None,
            rfam=False, g4=False, M=1.8, B=-0.6, rbp=False,
            i=None, ff=None, c=None, config=None, s=None, seq=None,
            a=None, ali=None, algo=None, algorithm=None, rb=None,
            fl=None, freqlim=None, ll=None, levlim=None, tl=None,
            ol=None, cl=None, pl=None, pr=None, s3=None, msn=None,
            rf=None, eo=None, hr=None, ico=None, iw=None, ignore=None,
            t=None, bs=None, v=None, inputrestr=None):
    """Print SQUARNA predictions for the given input; same keyword surface and
    defaults as the reference's Predict (cli.py:416-430, docstring 431-600).
    Short synonyms (i, ff, c, s, a, algo, rb, fl, ll, tl, ol, cl, pl, pr, s3, msn,
    rf, eo, hr, ico, iw, t, bs, v) override their long forms when given."""
    opts = dict(inputfile=inputfile, fileformat=fileformat, inputseq=inputseq, configfile=configfile,
                alignment=alignment, algorithms=algorithms, rankby=rankby, freqlimit=freqlimit,
                levellimit=levellimit, toplim=toplim, outplim=outplim, conslim=conslim, poollim=poollim,
                priority=priority, step3=step3, maxstemnum=maxstemnum, reactformat=reactformat,
                evalonly=evalonly, hardrest=hardrest, interchainonly=interchainonly, ignorewarn=ignorewarn,
                threads=threads, byseq=byseq, verbose=verbose)
    given = locals()
    for short, long_ in _SYNONYMS:          # later entries win, as in the reference's if-chain (cli.py:602-664)
        if given[short] is not None:
            opts[long_] = given[short]
    inputfile, fileformat, inputseq, configfile = (opts[k] for k in ("inputfile", "fileformat", "inputseq", "configfile"))
    alignment, algorithms, rankby, freqlimit = (opts[k] for k in ("alignment", "algorithms", "rankby", "freqlimit"))
    levellimit, toplim, outplim, conslim, poollim = (opts[k] for k in ("levellimit", "toplim", "outplim", "conslim", "poollim"))
    priority, step3, maxstemnum, reactformat = (opts[k] for k in ("priority", "step3", "maxstemnum", "reactformat"))
    evalonly, hardrest, interchainonly, ignorewarn = (opts[k] for k in ("evalonly", "hardrest", "interchainonly", "ignorewarn"))
    threads, byseq, verbose = (opts[k] for k in ("threads", "byseq", "verbose"))

    if HOME_DIR is None:
        HOME_DIR = os.path.dirname(os.path.abspath(__file__))
    if write_to is None:
        write_to = sys.stdout
    if inputfile is not None and not os.path.exists(inputfile) and os.path.exists(os.path.join(HOME_DIR, inputfile)):
        inputfile = os.path.join(HOME_DIR, inputfile)

    assert os.path.exists(str(inputfile)) or inputseq, "Input file does not exist."
    assert fileformat in {'unknown', 'fasta', 'default', 'stockholm', 'clustal'}, \
        "Wrong fileformat, choose one of these: default,fasta,stockholm,clustal"

    configfileset = configfile is not None
    if not configfileset:
        configfile = os.path.join(HOME_DIR, "def.conf")
        priority = set('bppN,bppH1,bppH2'.split(',')) if priority is None else set(x for x in priority.split(',') if x)
    else:
        if not os.path.exists(configfile):
            for cand in (os.path.join(HOME_DIR, configfile + ".conf"), os.path.join(HOME_DIR, configfile)):
                if os.path.exists(cand):
                    configfile = cand
                    break
        assert os.path.exists(configfile), "Config file does not exist."
        priority = set() if priority is None else set(x for x in priority.split(',') if x)

    assert ''.join(sorted(inputformat.replace('x', ''))) in {"q", "fq", "qr", "qt", "qrt", "fqr", "fqt", "fqrt"}, \
        'Inappropriate inputformat value (subset of "fqrtx" with "q" being mandatory): {}'.format(inputformat)

    maxstemnumset = maxstemnum is not None
    if maxstemnumset:
        try:
            maxstemnum = int(float(maxstemnum))
            assert maxstemnum >= 0
        except Exception:
            raise ValueError("Inappropriate maxstemnum value (non-negative integer): {}".format(maxstemnum))
    try:
        threads = min(max(1, int(float(threads))), os.cpu_count())
    except Exception:
        raise ValueError("Inappropriate threads value (integer): {}".format(threads))
    try:
        M = float(M)
    except Exception:
        raise ValueError("Inappropriate M value (float): {}".format(M))
    try:
        B = float(B)
    except Exception:
        raise ValueError("Inappropriate B value (float): {}".format(B))
    try:
        algos = set(algorithms.upper())
        assert algos <= {'E', 'G', 'H', 'N'}
    except Exception:
        raise ValueError('Inappropriate algorithm value (should be subset of "eghn"): {}'.format(algorithms))
    assert rankby in {"r", "s", "rs", "dr", "ds", "drs"}, \
        'Inappropriate rankby value (r/s/rs/dr/ds/drs): {}'.format(rankby)

    outplimset = outplim is not None
    if outplimset:
        outplim = _positive_int(outplim, "outplim")
    toplim = _positive_int(toplim, "toplim")
    if not outplimset:
        outplim = toplim
    conslim = _positive_int(conslim, "conslim")
    poollim = _positive_int(poollim, "poollim")
    assert int(float(reactformat)) in {3, 10, 26}, "Inappropriate reactformat value (3/10/26): {}".format(reactformat)
    reactformat = int(float(reactformat))
    if levellimit is not None:
        try:
            levellimit = int(float(levellimit))
        except Exception:
            raise ValueError("Inappropriate levellimit value (integer): {}".format(levellimit))
    try:
        freqlimit = float(freqlimit)
        assert 0 <= freqlimit <= 1
    except Exception:
        raise ValueError("Inappropriate freqlimit value (float between 0.0 and 1.0): {}".format(freqlimit))
    try:
        step3 = step3.lower()
        assert step3 in {'u', 'i', '1', '2'}
    except Exception:
        raise ValueError("Inappropriate freqlimit value (float between 0.0 and 1.0): {}".format(step3))

    rankbydiff = "d" in rankby
    if "r" in rankby and "s" in rankby:
        rankby = (0, 2, 1)
    elif "r" in rankby:
        rankby = (2, 0, 1)
    elif "s" in rankby:
        rankby = (1, 2, 0)

    # `ent` / entropy: the runners print "sequence<TAB>entropy:<TAB>value" in place of the sequence line
    # (SQRNdbnseq.py:1313-1318; Predict hands it on at SQUARNA.py:883, 926 and 990)
    if rfam or g4 or rbp:
        raise NotImplementedError("rfam / g4 / rbp restraint discovery is outside the GPU hot path")

    if alignment and not configfileset:
        configfile = os.path.join(HOME_DIR, "ali.conf")
    paramsetnames, paramsets = ParseConfig(configfile)
    auto = None
    if not configfileset:
        auto = (ParseConfig(os.path.join(HOME_DIR, "500.conf")), ParseConfig(os.path.join(HOME_DIR, "1000.conf")))
    if maxstemnumset:
        for ps in paramsets:
            ps['maxstemnum'] = maxstemnum
        if auto:
            for _, sets in auto:
                for ps in sets:
                    ps['maxstemnum'] = maxstemnum

    if alignment:
        from .SQRNdbnali import RunSQRNdbnali
        objs, fmt, _single = ParseInput(inputseq, inputfile, inputformat, fmt=fileformat, ignore=ignorewarn,
                                        inputrestr=inputrestr, M=M, B=B)
        defReactivities, defRestraints, defReference = ParseInput(inputseq, inputfile, inputformat,
                                                                  returndefaults=True, fmt=fmt, ignore=ignorewarn,
                                                                  M=M, B=B)[0]
        objs = list(objs)
        N = len(objs[0][1])
        assert all(len(obj[1]) == N for obj in objs), 'The sequences are not aligned'
        try:
            if defReactivities:
                defReactivities = _resolve_reacts(defReactivities, N, M, B)
            assert not defReactivities or len(defReactivities) == N
        except Exception:
            raise ValueError('Inappropriate default reactivities line:\n {}'.format(defReactivities))
        assert not defRestraints or len(defRestraints) == N, \
            'Inappropriate default restraints line:\n {}'.format(defRestraints)
        assert not defReference or len(defReference) == N, \
            'Inappropriate default reference line:\n {}'.format(defReference)
        if levellimit is None:
            levellimit = 3 - int(N > 500)
        RunSQRNdbnali(objs, defReactivities, defRestraints, defReference, levellimit, freqlimit, verbose, step3,
                      paramsetnames, paramsets, threads, rankbydiff, rankby, hardrest, interchainonly, toplim,
                      outplim, conslim, reactformat, poollim, entropy=entropy, algos=algos, sink=write_to, M=M, B=B)
        return

    # single-sequence mode (cli.py:845-935).  byseq and pool-parallel modes print the same
    # text in the reference; both stream the input through batched GPU calls here.
    inputs, fmt, _single = ParseInput(inputseq, inputfile, inputformat, fmt=fileformat, ignore=ignorewarn,
                                      inputrestr=inputrestr, M=M, B=B)

    # Bulk lane: one greedy parameter set, pl=1, an input made of name + sequence lines only.  The whole file is
    # parsed, predicted and turned into text on buffers (csrc/sqrn_textio.cpp + the fast lane); any other shape
    # takes the per-entry path below, which prints the same text.
    algos_ = {a for a in algos} if algos else None
    if (inputfile and not inputseq and fmt in ("default", "fasta") and auto is None and not evalonly
            and len(paramsets) == 1 and (algos_ or set(paramsets[0]["algorithms"])) == {"G"}
            and not paramsets[0].get("bpp", 0) and poollim == 1 and not interchainonly
            and min(toplim, outplim, conslim) >= 1 and (fmt == "fasta" or inputformat.startswith("q"))
            and not entropy and os.environ.get("SQRN_NO_BULK") is None):
        def per_entry(entries):              # the few entries the bulk lane cannot print (> 30 pseudoknot levels)
            RunSQRNdbnseqBatch(entries, paramsetnames, paramsets, rankbydiff, rankby, hardrest, interchainonly,
                               toplim, outplim, conslim, reactformat, evalonly, poollim, sink=write_to,
                               algos=algos, priority=priority, rfam=None, levellimit=levellimit, entropy=entropy, M=M, B=B)
        if _bulk_lane(inputfile, fmt == "fasta", paramsetnames[0], paramsets[0], conslim, write_to, per_entry=per_entry):
            return

    def config_for(sequence):               # autoconfig by RAW (gapped) length, cli.py:870-878
        if auto is None or len(sequence) < 500:
            return 0
        return 2 if len(sequence) >= 1000 else 1

    tables = [(paramsetnames, paramsets)] + (list(auto) if auto else [])
    pending = []
    n_seen = n_printed = 0

    def flush():
        # entries of one flush share a config table; input order is preserved because a
        # change of table forces a flush
        if not pending:
            return
        names_, sets_ = tables[pending[0][0]]
        nonlocal n_printed
        n_printed += len(pending)
        RunSQRNdbnseqBatch([e[1] for e in pending], names_, sets_, rankbydiff, rankby, hardrest, interchainonly,
                           toplim, outplim, conslim, reactformat, evalonly, poollim, sink=write_to,
                           algos=algos, priority=priority, rfam=None, levellimit=levellimit, entropy=entropy, M=M, B=B,
                           header_on_error=not byseq)
        del pending[:]

    entries = iter(inputs)
    while True:
        try:
            entry = next(entries)
        except StopIteration:
            break
        except Exception:
            # a line the parser rejects: the reference streams its input (SQUARNA.py:866-885) and has printed every
            # entry before it; with byseq it prints in groups of threads * 10 entries (887-935): the full groups
            if byseq:
                group = max(int(threads), 1) * 10
                del pending[max(n_seen // group * group - n_printed, 0):]
            flush()
            raise
        n_seen += 1
        which = config_for(entry[1])
        if pending and (pending[0][0] != which or len(pending) >= BATCH_ENTRIES):
            flush()
        pending.append((which, entry))
    flush()


def _bulk_lane(path, multiline, psname, paramset, conslim, sink, device=None, slice_entries=131072, per_entry=None):
    """SQUARNA.py:845-935 for the plain shape of an input.  False: not that shape (nothing was written)."""
    import time
    import numpy as np
    from . import _lib
    from .SQRNdbnseq import get_context
    trace = os.environ.get("SQRN_TRACE") is not None
    t0 = time.perf_counter()
    with open(path, "rb") as fh:
        text = fh.read()
    t1 = time.perf_counter()
    parsed = _lib.text_parse(text, multiline)
    if parsed is None:
        return False
    sym, sym_off = _lib.text_ungap(parsed)                           # UnAlign (seq.py:236-255) on the whole buffer
    t2 = time.perf_counter()
    if int(np.diff(sym_off).max(initial=0)) > 16000:
        return False
    from .SQRNdbnseq import _resolve_devices
    devs = [device] if device is not None else _resolve_devices(None)
    if len(devs) > 1 and parsed.n >= 4096 * len(devs):
        # every visible GPU, one host thread each (the reference's Pool(threads) over sequences, SQUARNA.py:889)
        from .sharding import MultiGPU
        ctx = MultiGPU(contexts=[get_context(d) for d in devs])
    else:
        ctx = get_context(devs[0])
    try:
        dbn, scores, nst = ctx.fast_predict(paramset, sym, sym_off)
    except _lib.SqrnError:
        return False
    # sequences whose structure has more than 30 pseudoknot levels (n_stems = -1: the one-byte glyphs ran out) are
    # printed by the per-entry path, in their place; everything around them stays on the bulk formatter
    t3 = time.perf_counter()
    deep = np.flatnonzero(nst < 0).tolist()
    if deep and per_entry is None:
        return False
    binary = getattr(sink, "buffer", None)
    scratch = [[], []]                                               # two text buffers, reused by every other slice

    def emit(first, stop):
        # slice k + 1 is formatted (library threads) while a writer thread hands slice k to the file: both release the GIL
        writer = pending = None
        try:
            for k, lo in enumerate(range(first, stop, slice_entries)):
                count = min(slice_entries, stop - lo)
                block = _lib.text_format(parsed, lo, count, sym_off, dbn, scores, conslim, psname, scratch[k & 1])
                if binary is None:
                    sink.write(block.tobytes().decode("ascii"))
                    continue
                if pending is not None:
                    pending.result()                                 # (its buffer is the one the next slice will reuse)
                elif stop - lo > slice_entries:
                    from concurrent.futures import ThreadPoolExecutor
                    writer = ThreadPoolExecutor(1)
                    sink.flush()
                if writer is None:
                    sink.flush()
                    binary.write(memoryview(block))
                else:
                    pending = writer.submit(binary.write, memoryview(block))
            if pending is not None:
                pending.result()
        finally:
            if writer is not None:
                writer.shutdown(wait=True)

    at = 0
    for e in deep:
        emit(at, e)
        nb, nl = int(parsed.name_begin[e]), int(parsed.name_len[e])
        name = bytes(parsed.text[nb:nb + nl]).decode("ascii")
        seq = bytes(parsed.seq[int(parsed.seq_offsets[e]):int(parsed.seq_offsets[e + 1])]).decode("ascii")
        per_entry([(name, seq, None, None, None)])
        at = e + 1
    emit(at, parsed.n)
    if trace:
        print("[sqrn] bulk lane: read %.3f s, parse + ungap %.3f s, predict %.3f s, format + write %.3f s (%d entries)"
              % (t1 - t0, t2 - t1, t3 - t2, time.perf_counter() - t3, parsed.n), file=sys.stderr)
    return True


# --------------------------------------------------------------------- Main
_VALUE_OPTS = {"algo": "algorithms", "algos": "algorithms", "algorithm": "algorithms", "algorithms": "algorithms",
               "s": "inputseq", "seq": "inputseq", "sequence": "inputseq", "i": "inputfile", "input": "inputfile",
               "ff": "fileformat", "fileformat": "fileformat", "c": "configfile", "config": "configfile",
               "if": "inputformat", "inputformat": "inputformat", "msn": "maxstemnum", "maxstemnum": "maxstemnum",
               "t": "threads", "threads": "threads", "rb": "rankby", "rankby": "rankby", "tl": "toplim",
               "toplim": "toplim", "ol": "outplim", "outplim": "outplim", "cl": "conslim", "conslim": "conslim",
               "pl": "poollim", "poollim": "poollim", "pr": "priority", "priority": "priority",
               "rf": "reactformat", "reactformat": "reactformat", "ll": "levellimit", "levlim": "levellimit",
               "levellim": "levellimit", "levlimit": "levellimit", "levellimit": "levellimit",
               "fl": "freqlimit", "freqlim": "freqlimit", "freqlimit": "freqlimit", "frequencylim": "freqlimit",
               "frequencylimit": "freqlimit", "s3": "step3", "step3": "step3", "m": "M", "b": "B"}
_FLAG_OPTS = {"bs": "byseq", "byseq": "byseq", "eo": "evalonly", "evalonly": "evalonly", "hr": "hardrest",
              "hardrest": "hardrest", "ico": "interchainonly", "interchainonly": "interchainonly",
              "a": "alignment", "ali": "alignment", "alignment": "alignment", "v": "verbose", "verbose": "verbose",
              "iw": "ignorewarn", "ignore": "ignorewarn", "ent": "entropy", "entropy": "entropy", "rbp": "rbp",
              "rfam": "rfam", "g4": "g4"}
# "-key value" forms the reference rewrites to key=value / bare flags (cli.py:1073-1108)
_DASH_VALUE = {"algo", "algorithm", "algos", "algorithms", "b", "c", "config", "i", "input", "if", "inputformat",
               "rb", "rankby", "ff", "fileformat", "fl", "freqlim", "ll", "levlim", "tl", "toplim", "ol", "outplim",
               "cl", "conslim", "pl", "poollim", "pr", "priority", "s3", "step3", "m", "msn", "maxstemnum", "rf",
               "reactformat", "s", "seq", "sequence", "t", "threads"}
_DASH_FLAG = {"a", "ali", "alignment", "bs", "byseq", "ent", "entropy", "eo", "evalonly", "g4", "hr", "hardrest",
              "iw", "ignore", "ico", "interchainonly", "rbp", "rfam", "v", "verbose"}

USAGE = """
Usage:

SQUARNA i=inputfile [OPTIONS]

SQUARNA s=ACGUGUCAC [OPTIONS]

For further details read the help message:

SQUARNA --help
"""


def Main(argv=None):
    """console entry point (cli.py:994-1257): key=value options, bare flags and
    `-key value` forms; prints the input path, then calls Predict."""
    home = os.path.dirname(os.path.abspath(__file__))
    args = list(sys.argv[1:] if argv is None else argv)
    if not args:
        print(USAGE)
        sys.exit(1)
    if any(h in args for h in ("--help", "-help", "help", "--h", "-h", "h", "--H", "-H", "H")):
        with open(os.path.join(home, "USAGE.md")) as fh:
            print(fh.read())
        sys.exit(0)

    normal = []
    k = 0
    while k < len(args):
        a = args[k]
        bare = a.lstrip('-').lower()
        if a.startswith('-') and bare in _DASH_VALUE and a.lower() in ("-" + bare, "--" + bare):
            normal.append(a.lstrip('-') + '=' + args[k + 1])
            k += 1
        elif a.startswith('-') and bare in _DASH_FLAG and a.lower() in ("-" + bare, "--" + bare):
            normal.append(a.lstrip('-'))
        else:
            normal.append(a)
        k += 1

    kw = dict(inputfile=None, fileformat="unknown", inputseq=None, configfile=None, inputformat="qtrf",
              maxstemnum=None, threads=os.cpu_count(), byseq=False, algorithms="", entropy=False, rankby="r",
              evalonly=False, hardrest=False, interchainonly=False, toplim=5, outplim=None, conslim=1,
              poollim=100, reactformat=3, alignment=False, levellimit=None, freqlimit=0.35, verbose=False,
              step3="u", ignorewarn=False, priority=None, rfam=False, g4=False, rbp=False, M=1.8, B=-0.6)
    for a in normal:
        low = a.lower()
        key, sep, val = a.partition('=')
        if sep and key.lower() in _VALUE_OPTS:
            dest = _VALUE_OPTS[key.lower()]
            if dest == "algorithms" and not val:
                continue
            if dest in ("fileformat", "inputformat"):
                val = val.lower()
            elif dest == "rankby":
                val = ''.join(sorted(val.lower()))
            kw[dest] = val
        elif low in _FLAG_OPTS:
            kw[_FLAG_OPTS[low]] = True
        elif len(normal) == 1:
            if os.path.exists(a):
                kw["inputfile"] = a
            elif sum(low.count(x) for x in (GAPS | set("acgut"))) > len(a) / 2:
                kw["inputseq"] = a
            else:
                kw["inputfile"] = a
        else:
            print("Unrecognized option: {}".format(a))

    print(kw["inputfile"])
    Predict(HOME_DIR=home, write_to=None, **kw)


if __name__ == "__main__":
    Main()
