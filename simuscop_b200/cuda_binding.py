"""ctypes binding of libsimuscop_cuda.so (the C ABI of include/simuscop.h).

Plumbing for tests and bench.py only: every call goes to the CUDA library; a missing
library or a missing GPU raises -- there is no fallback path.
"""
import ctypes as C

import numpy as np

from . import abi
from .paths import LIB_CUDA

SYMBOLS = ["ssc_last_error", "ssc_version", "ssc_create", "ssc_destroy", "ssc_set_option", "ssc_set_profile",
           "ssc_genome_reserve", "ssc_genome_append", "ssc_genome_size", "ssc_reference_upload", "ssc_reference_upload_fasta", "ssc_reference_prefetch_fasta", "ssc_reference_adopt_prefetched", "ssc_genome_append_ref", "ssc_genome_poke", "ssc_genome_read", "ssc_gc_census", "ssc_set_plan", "ssc_generate",
           "ssc_generate_device", "ssc_read_shape", "ssc_generate_reads", "ssc_segment_name", "ssc_get_stats", "ssc_reset_stats",
           "ssc_table_lookup_host", "ssc_sub_lookup_host", "ssc_gzip_member_host", "ssc_issue_floor", "ssc_set_read_group",
           "ssc_bam_header"]

_lib = None


class SscError(RuntimeError):
    pass


def lib():
    global _lib
    if _lib is None:
        L = C.CDLL(LIB_CUDA)   # raises OSError when the extension is not built: no fallback
        L.ssc_last_error.restype = C.c_char_p
        L.ssc_create.argtypes = [C.c_int, C.POINTER(C.c_void_p)]
        L.ssc_destroy.argtypes = [C.c_void_p]
        L.ssc_set_option.argtypes = [C.c_void_p, C.c_char_p, C.c_int64]
        L.ssc_set_profile.argtypes = [C.c_void_p, C.POINTER(abi.ProfileTables)]
        L.ssc_genome_reserve.argtypes = [C.c_void_p, C.c_uint64]
        L.ssc_genome_append.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64, C.POINTER(C.c_uint64)]
        L.ssc_genome_size.argtypes = [C.c_void_p, C.POINTER(C.c_uint64)]
        L.ssc_reference_upload.argtypes = [C.c_void_p, C.c_char_p, C.c_uint64]
        L.ssc_reference_upload_fasta.argtypes = [C.c_void_p, C.c_int, C.c_uint64, C.c_uint64, C.c_uint64, C.c_uint32, C.c_uint32,
                                                 C.POINTER(C.c_uint64)]
        L.ssc_reference_prefetch_fasta.argtypes = [C.c_void_p, C.c_int, C.c_uint64, C.c_uint64, C.c_uint64, C.c_uint32, C.c_uint32]
        L.ssc_reference_adopt_prefetched.argtypes = [C.c_void_p, C.POINTER(C.c_uint64)]
        L.ssc_genome_append_ref.argtypes = [C.c_void_p, C.c_uint64, C.c_uint64, C.c_int32, C.POINTER(C.c_uint64)]
        L.ssc_genome_poke.argtypes = [C.c_void_p, C.c_void_p, C.c_char_p, C.c_int64]
        L.ssc_genome_read.argtypes = [C.c_void_p, C.c_uint64, C.c_uint64, C.c_void_p]
        L.ssc_gc_census.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p]
        L.ssc_set_plan.argtypes = [C.c_void_p, C.c_uint64, C.c_void_p, C.c_int64, C.c_void_p, C.c_int64,
                                   C.c_char_p, C.c_int64, C.POINTER(C.c_int64), C.POINTER(C.c_int64)]
        L.ssc_generate.argtypes = [C.c_void_p, C.c_int64, C.c_int64, abi.SINK_FN, C.c_void_p]
        L.ssc_generate_device.argtypes = [C.c_void_p, C.c_int64, C.c_int64, C.POINTER(C.c_uint64),
                                          C.POINTER(C.c_uint64), C.POINTER(C.c_uint64), C.POINTER(C.c_double)]
        L.ssc_read_shape.argtypes = [C.c_void_p, C.c_int64, C.c_int64, C.POINTER(C.c_int64), C.POINTER(C.c_int32),
                                     C.POINTER(C.c_int32)]
        L.ssc_generate_reads.argtypes = [C.c_void_p, C.c_int64, C.c_int64, C.POINTER(abi.ReadArrays), C.c_void_p,
                                         C.POINTER(C.c_int64)]
        L.ssc_segment_name.argtypes = [C.c_void_p, C.c_int32, C.c_char_p, C.c_int32]
        L.ssc_get_stats.argtypes = [C.c_void_p, C.POINTER(abi.Stats)]
        L.ssc_reset_stats.argtypes = [C.c_void_p]
        L.ssc_table_lookup_host.argtypes = [C.c_void_p, C.c_int, C.c_uint32]
        L.ssc_sub_lookup_host.argtypes = [C.c_void_p, C.c_uint32]
        L.ssc_gzip_member_host.argtypes = [C.c_char_p, C.c_uint32, C.c_char_p, C.c_size_t, C.c_void_p, C.c_size_t]
        L.ssc_gzip_member_host.restype = C.c_int64
        L.ssc_issue_floor.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int64, C.c_int, C.POINTER(C.c_double)]
        L.ssc_set_read_group.argtypes = [C.c_void_p, C.c_char_p]
        L.ssc_bam_header.argtypes = [C.c_char_p, C.c_void_p, C.c_size_t]
        L.ssc_bam_header.restype = C.c_int64
        _lib = L
    return _lib


def _ck(rc):
    if rc != 0:
        raise SscError("ssc error %d: %s" % (rc, lib().ssc_last_error().decode(errors="replace")))


def bam_header(read_group=None):
    """The header of a BAM stream of the "bam" option as one BGZF block (ssc_bam_header; needs no GPU): @HD, an @RG line
    with ID and SM = read_group when it is given, no references."""
    rg = read_group.encode() if isinstance(read_group, str) else read_group
    buf = C.create_string_buffer(1024)
    n = lib().ssc_bam_header(rg, buf, len(buf))
    if n <= 0:
        raise SscError("ssc_bam_header: %s" % lib().ssc_last_error().decode(errors="replace"))
    return buf.raw[:n]


def _read_views(reads, length, pair_id, segment, pos, frag):
    return dict(reads=reads, seq=reads[:, :, 0], qual=reads[:, :, 1], length=length, pair_id=pair_id, segment=segment, pos=pos,
                frag=frag)


class Generator:
    """One handle on one GPU."""

    def __init__(self, device=0):
        self.h = C.c_void_p()
        _ck(lib().ssc_create(device, C.byref(self.h)))
        self.device = device
        self.planned = 0
        self.emitted = 0
        self._keep = []

    def close(self):
        if self.h:
            lib().ssc_destroy(self.h)
            self.h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def set_option(self, key, value):
        _ck(lib().ssc_set_option(self.h, key.encode(), int(value)))

    def set_read_group(self, read_group):
        """RG:Z:<read_group> on every record of the "bam" output; None or "" removes the tag (ssc_set_read_group)."""
        rg = read_group.encode() if isinstance(read_group, str) else read_group
        _ck(lib().ssc_set_read_group(self.h, rg))

    def load_plan(self, plan, seed):
        """Upload profile tables, haplotype store and bins of a planfile.Plan."""
        prof = plan.profile_struct()
        _ck(lib().ssc_set_profile(self.h, C.byref(prof)))
        g = np.ascontiguousarray(plan.genome)
        _ck(lib().ssc_genome_reserve(self.h, g.size))
        first = C.c_uint64()
        _ck(lib().ssc_genome_append(self.h, g.ctypes.data, g.size, C.byref(first)))
        assert first.value == 0
        self.set_plan(plan.bins, plan.segs, plan.names, seed)

    def genome_read(self, start, n):
        """Decode store bases [start, start+n) back to upper-case ASCII (diagnostic)."""
        buf = C.create_string_buffer(int(n))
        _ck(lib().ssc_genome_read(self.h, int(start), int(n), buf))
        return buf.raw[:n]

    def genome_size(self):
        v = C.c_uint64()
        _ck(lib().ssc_genome_size(self.h, C.byref(v)))
        return v.value

    def gc_census(self, starts, lens):
        """G/C and non-ACGT base counts of haplotype-store intervals (ssc_gc_census)."""
        starts = np.ascontiguousarray(starts, dtype=np.int64)
        lens = np.ascontiguousarray(lens, dtype=np.int32)
        gc = np.zeros(len(starts), np.int32)
        nn = np.zeros(len(starts), np.int32)
        _ck(lib().ssc_gc_census(self.h, starts.ctypes.data, lens.ctypes.data, len(starts), gc.ctypes.data, nn.ctypes.data))
        return gc, nn

    def set_plan(self, bins, segs, names, seed):
        bins = np.ascontiguousarray(bins)
        segs = np.ascontiguousarray(segs)
        pp, ep = C.c_int64(), C.c_int64()
        _ck(lib().ssc_set_plan(self.h, seed, bins.ctypes.data, bins.size, segs.ctypes.data, segs.size,
                               names, len(names), C.byref(pp), C.byref(ep)))
        self.planned, self.emitted = pp.value, ep.value
        return self.planned, self.emitted

    def generate(self, lo=0, hi=None, sink=None, user=None):
        """Stream pairs [lo, hi) through the pinned host slabs. Without `sink` returns (fq1, fq2) bytes.  `sink`: a Python
        callable or a C function (an abi.SINK_FN instance, e.g. the file writer of libsimuscop_host) called with `user`."""
        if hi is None:
            hi = self.planned
        parts1, parts2 = [], []

        def collect(user, b1, l1, b2, l2, first, n):
            parts1.append(C.string_at(b1, l1))
            if b2:
                parts2.append(C.string_at(b2, l2))
            return 0
        cb = sink if isinstance(sink, abi.SINK_FN) else abi.SINK_FN(sink if sink is not None else collect)
        _ck(lib().ssc_generate(self.h, lo, hi, cb, user))
        if sink is None:
            return b"".join(parts1), b"".join(parts2)

    def generate_device(self, lo=0, hi=None):
        if hi is None:
            hi = self.planned
        b1, b2, nb, ms = C.c_uint64(), C.c_uint64(), C.c_uint64(), C.c_double()
        _ck(lib().ssc_generate_device(self.h, lo, hi, C.byref(b1), C.byref(b2), C.byref(nb), C.byref(ms)))
        return dict(bytes1=b1.value, bytes2=b2.value, bases=nb.value, device_ms=ms.value)

    def read_shape(self, lo=0, hi=None):
        """(pairs the range [lo, hi) emits, mates per pair, slot pitch in bytes) of the array output."""
        if hi is None:
            hi = self.planned
        n, m, p = C.c_int64(), C.c_int32(), C.c_int32()
        _ck(lib().ssc_read_shape(self.h, lo, hi, C.byref(n), C.byref(m), C.byref(p)))
        return n.value, m.value, p.value

    def empty_reads(self, n_pairs):
        """Uninitialised torch arrays for n_pairs pairs of array output on the handle's device (see generate_reads)."""
        import torch
        _, mates, pitch = self.read_shape(0, 0)
        dev = torch.device("cuda", self.device)
        n = max(int(n_pairs), 1)                     # the library takes no null pointers, also for an empty range
        reads = torch.empty((n, mates, 2, pitch), dtype=torch.uint8, device=dev)
        return _read_views(reads, torch.empty((n, mates), dtype=torch.int16, device=dev),
                           torch.empty(n, dtype=torch.int64, device=dev), torch.empty(n, dtype=torch.int32, device=dev),
                           torch.empty(n, dtype=torch.int32, device=dev), torch.empty(n, dtype=torch.int32, device=dev))

    def generate_reads(self, lo=0, hi=None, stream=None, out=None):
        """Pairs [lo, hi) as torch arrays on the handle's device, no FASTQ text and no host copy (ssc_generate_reads).  Returns a
        dict: reads [n, M, 2, pitch] uint8 (row 0 the bases, row 1 the qualities as FASTQ characters, zero past the length), seq
        and qual (its two rows), length [n, M] int16, pair_id [n] int64, segment / pos / frag [n] int32 (the read name is
        segment_name(segment) + pos + '#' + frag + '/mate').  The call is ordered after the work queued on `stream` (default: torch's
        current stream) and returns when the arrays are complete.  `out`: arrays of an earlier call or of empty_reads, with room
        for the range, written in place (the result views their first n rows)."""
        import torch
        if hi is None:
            hi = self.planned
        if out is None:
            out = self.empty_reads(self.read_shape(lo, hi)[0])
        a = out
        for k, dt in (("reads", torch.uint8), ("length", torch.int16), ("pair_id", torch.int64), ("segment", torch.int32),
                      ("pos", torch.int32), ("frag", torch.int32)):
            if a[k].dtype != dt or not a[k].is_contiguous() or not a[k].is_cuda:
                raise ValueError("generate_reads: out[%r] must be a contiguous CUDA tensor of %s" % (k, dt))
        if stream is None:
            stream = torch.cuda.current_stream(torch.device("cuda", self.device))
        st = abi.ReadArrays(a["reads"].data_ptr(), a["length"].data_ptr(), a["pair_id"].data_ptr(), a["segment"].data_ptr(),
                            a["pos"].data_ptr(), a["frag"].data_ptr(), min(a["reads"].shape[0], a["length"].shape[0],
                            a["pair_id"].shape[0], a["segment"].shape[0], a["pos"].shape[0], a["frag"].shape[0]),
                            a["reads"].shape[-1])
        n = C.c_int64()
        _ck(lib().ssc_generate_reads(self.h, lo, hi, C.byref(st), C.c_void_p(stream.cuda_stream), C.byref(n)))
        k = n.value
        return _read_views(a["reads"][:k], a["length"][:k], a["pair_id"][:k], a["segment"][:k], a["pos"][:k], a["frag"][:k])

    def segment_name(self, i):
        """Read-name prefix "@<popu>#<chr>#" of segment i of the plan (the `segment` array of generate_reads)."""
        buf = C.create_string_buffer(80)
        _ck(lib().ssc_segment_name(self.h, int(i), buf, len(buf)))
        return buf.value

    def issue_floor(self, mode, read_length, n_pairs, reps=3):
        """Mean launch time (ms) of the issue-rate microbenchmark (ssc_issue_floor)."""
        ms = C.c_double()
        _ck(lib().ssc_issue_floor(self.h, mode, read_length, n_pairs, reps, C.byref(ms)))
        return ms.value

    def stats(self):
        s = abi.Stats()
        _ck(lib().ssc_get_stats(self.h, C.byref(s)))
        return {k: getattr(s, k) for k, _ in abi.Stats._fields_}

    def reset_stats(self):
        _ck(lib().ssc_reset_stats(self.h))
