"""ctypes binding of the CPU oracle (oracle/libssc_oracle.so).

TEST INFRASTRUCTURE: imported only by tests/, __graft_entry__.smoke() and bench.py's
cpu_baseline leg.  It lives outside the product package (simuscop_b200/) on purpose: nothing
on the product path imports, links or executes anything under oracle/.
"""
import ctypes as C

import numpy as np

from simuscop_b200 import abi
from simuscop_b200.paths import ORACLE_LIB


class OraclePlan(C.Structure):
    _fields_ = [("prof", C.POINTER(abi.ProfileTables)), ("genome", C.c_void_p), ("genome_len", C.c_uint64),
                ("bins", C.c_void_p), ("n_bins", C.c_int64), ("segs", C.c_void_p), ("n_segs", C.c_int64),
                ("names", C.c_char_p), ("genome_first", C.c_uint64)]


_lib = None


def lib():
    global _lib
    if _lib is None:
        _lib = C.CDLL(ORACLE_LIB)
        _lib.ssco_generate.restype = C.c_int64
        _lib.ssco_generate.argtypes = [C.POINTER(OraclePlan), C.c_uint64, C.c_int64, C.c_int64,
                                       C.c_void_p, C.c_size_t, C.POINTER(C.c_size_t),
                                       C.c_void_p, C.c_size_t, C.POINTER(C.c_size_t),
                                       C.c_void_p, C.c_int64, C.POINTER(C.c_uint64)]
        _lib.ssco_philox.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
        _lib.ssco_draw_real.restype = C.c_double
        _lib.ssco_draw_real.argtypes = [C.c_uint32, C.c_double, C.c_double]
        _lib.ssco_draw_int.restype = C.c_long
        _lib.ssco_draw_int.argtypes = [C.c_uint32, C.c_long, C.c_long]
        _lib.ssco_rand_indx.restype = C.c_int
        _lib.ssco_rand_indx.argtypes = [C.c_void_p, C.c_int, C.c_uint32]
        _lib.ssco_set_draw_trace.restype = None
        _lib.ssco_set_draw_trace.argtypes = [C.c_void_p, C.c_int64] * 3
        _lib.ssco_draw_trace_counts.restype = None
        _lib.ssco_draw_trace_counts.argtypes = [C.c_void_p]
    return _lib


def philox(ctr, key):
    c = np.asarray(ctr, dtype=np.uint32)
    k = np.asarray(key, dtype=np.uint32)
    o = np.zeros(4, dtype=np.uint32)
    lib().ssco_philox(c.ctypes.data, k.ctypes.data, o.ctypes.data)
    return o


# draw_trace=True: what ssc_oracle.c records for the pairs in range, one structured array per table
FRAG_TRACE = np.dtype([("pair", "i8"), ("attempt", "i8"), ("x0", "i8"), ("x1", "i8"), ("pos", "i8"), ("want", "i8"),
                       ("len", "i8"), ("accepted", "i8")])
# kind: 0 = neither event test passed, 1 = the insertion test passed (k inserted bases, k may be 0), 2 = the deletion test passed
# (k deleted template bases before clipping at the read end); lenword: the length draw (0 when kind is 0)
SCAN_TRACE = np.dtype([("pair", "i8"), ("mate", "i8"), ("j", "i8"), ("x0", "i8"), ("x1", "i8"), ("kind", "i8"), ("k", "i8"),
                       ("lenword", "i8")])
# j: output position, m: read length after indels, subtab: 1 or 2 (subs_cdf1 / subs_cdf2), row: k-mer row (-1: the base passes
# through), ref / call: base indices (-1: N), qrow: ref * 4 + call (-1: N, its quality is drawn without a table)
BASE_TRACE = np.dtype([("pair", "i8"), ("mate", "i8"), ("j", "i8"), ("m", "i8"), ("subtab", "i8"), ("row", "i8"), ("bin", "i8"),
                       ("ref", "i8"), ("call", "i8"), ("u2", "i8"), ("qrow", "i8"), ("u3", "i8")])
_TRACE_DTYPES = (FRAG_TRACE, SCAN_TRACE, BASE_TRACE)


def generate(plan, seed, pair_lo=0, pair_hi=None, trace=False, genome=None, genome_first=0, draw_trace=False):
    """Run the oracle over a simuscop_b200.planfile.Plan. Returns (fq1, fq2, info).
    genome / genome_first: a window of the haplotype store (ASCII, store index of its first base) instead of plan.genome,
    for plans whose store is too large to hold as ASCII (bench-scale parity tests).
    draw_trace: info["frag"], info["scan"] and info["base"] hold every fragment attempt, scanned position and output base
    of the pairs in range (FRAG_TRACE, SCAN_TRACE, BASE_TRACE)."""
    if draw_trace:
        return _generate_traced(plan, seed, pair_lo, pair_hi, trace, genome, genome_first)
    L = lib()
    if pair_hi is None:
        pair_hi = plan.planned_pairs()
    prof = plan.profile_struct()
    op = OraclePlan()
    op.prof = C.pointer(prof)
    genome = np.ascontiguousarray(plan.genome if genome is None else genome)
    bins = np.ascontiguousarray(plan.bins)
    segs = np.ascontiguousarray(plan.segs)
    op.genome = genome.ctypes.data
    op.genome_len = genome.size
    op.genome_first = int(genome_first)
    op.bins = bins.ctypes.data
    op.n_bins = bins.size
    op.segs = segs.ctypes.data
    op.n_segs = segs.size
    op.names = plan.names
    npairs = max(0, pair_hi - pair_lo)
    rl = plan.hdr["read_length"]
    cap = int(npairs * (2 * rl * 2 + 400) + 4096)
    out1 = np.empty(cap, dtype=np.uint8)
    out2 = np.empty(cap if plan.paired else 1, dtype=np.uint8)
    l1, l2, nb = C.c_size_t(0), C.c_size_t(0), C.c_uint64(0)
    tr = np.zeros((npairs, 4), dtype=np.int64) if trace else None
    n = L.ssco_generate(C.byref(op), seed, pair_lo, pair_hi, out1.ctypes.data, out1.size, C.byref(l1),
                        out2.ctypes.data if plan.paired else None, out2.size if plan.paired else 0, C.byref(l2),
                        tr.ctypes.data if trace else None, npairs if trace else 0, C.byref(nb))
    if n == -3:
        raise RuntimeError("oracle: a fragment lies outside the genome window handed over")
    if n < 0:
        raise RuntimeError("oracle output buffer too small (%d)" % n)
    info = dict(emitted=int(n), bases=int(nb.value), trace=tr[:n] if trace else None)
    return out1[:l1.value].tobytes(), out2[:l2.value].tobytes() if plan.paired else b"", info


def _generate_traced(plan, seed, pair_lo, pair_hi, trace, genome, genome_first):
    L = lib()
    npairs = max(0, (plan.planned_pairs() if pair_hi is None else pair_hi) - pair_lo)
    caps = [4 * npairs + 64, 2 * npairs * plan.hdr["read_length"] + 64, 4 * npairs * plan.hdr["read_length"] + 64]
    for _ in range(2):
        bufs = [np.zeros(c, dtype=d) for c, d in zip(caps, _TRACE_DTYPES)]
        L.ssco_set_draw_trace(*[a for b in bufs for a in (b.ctypes.data, b.size)])
        try:
            f1, f2, info = generate(plan, seed, pair_lo, pair_hi, trace, genome, genome_first)
            counts = np.zeros(3, dtype=np.int64)
            L.ssco_draw_trace_counts(counts.ctypes.data)
        finally:
            L.ssco_set_draw_trace(None, 0, None, 0, None, 0)
        if all(n <= c for n, c in zip(counts, caps)):
            info.update(frag=bufs[0][:counts[0]], scan=bufs[1][:counts[1]], base=bufs[2][:counts[2]])
            return f1, f2, info
        caps = [int(n) for n in counts]
    raise RuntimeError("oracle draw trace: counts changed between two runs of the same plan")
