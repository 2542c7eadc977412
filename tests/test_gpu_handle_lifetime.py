"""Handle lifetime: the device memory a handle allocates is freed with the handle, and a call that fails frees what it
allocated before it failed.

Both tests read the device's free memory (torch.cuda.mem_get_info) and assume that the process has the GPU to itself."""
import ctypes as C
import hashlib
import os

import numpy as np
import pytest

import helpers
from simuscop_b200 import cuda_binding, planfile

pytestmark = pytest.mark.gpu

MiB = 1 << 20
SSC_ERR_INVALID = 1


def free_bytes():
    import torch
    torch.cuda.synchronize(0)
    torch.cuda.empty_cache()
    return torch.cuda.mem_get_info(0)[0]


def test_rejected_issue_floor_frees_its_scratch(built):
    """ssc_issue_floor allocates its scratch before it refuses mode 1 with 4,194,304 pairs, whose two blob files do not fit
    32-bit cursors.  2,000 refused calls leave the free device memory as it was after the first."""
    L = cuda_binding.lib()
    g = cuda_binding.Generator(0)
    try:
        ms = C.c_double()

        def refused():
            return L.ssc_issue_floor(g.h, 1, 151, 1 << 22, 1, C.byref(ms)) == SSC_ERR_INVALID

        assert refused(), L.ssc_last_error()
        assert b"32-bit blob cursors" in L.ssc_last_error()
        before = free_bytes()
        assert all(refused() for _ in range(2000))
        lost = before - free_bytes()
        assert lost <= 4 * MiB, "%d bytes of device memory lost over 2000 refused calls" % lost
    finally:
        g.close()


def write_fasta(path, n, cols=60, seed=3):
    """One record of n random ACGT bases in lines of `cols`; returns the arguments of ssc_reference_upload_fasta after fd."""
    seq = np.frombuffer(b"ACGT", np.uint8)[np.random.default_rng(seed).integers(0, 4, n)].tobytes()
    head = b">chrA\n"
    with open(path, "wb") as f:
        f.write(head + b"".join(seq[i:i + cols] + b"\n" for i in range(0, n, cols)))
    return len(head), n + (n - 1) // cols, n, cols, cols + 1


def one_round(plan, seed, fasta):
    """Creates a handle, runs every output mode and one FASTA upload, prefetch and adoption on it, and destroys it.  Returns a
    digest of everything it generated."""
    L = cuda_binding.lib()
    h = hashlib.sha256()
    g = cuda_binding.Generator(0)
    try:
        g.set_option("batch_pairs", 1024)            # many batches: both buffer sets and the mover in use
        g.load_plan(plan, seed)
        for opts in ({}, {"gzip": 1, "bgzf": 1}, {"interleave": 1}):
            for k, v in opts.items():
                g.set_option(k, v)
            for part in g.generate():
                h.update(part)
            dev = g.generate_device()
            h.update(b"%d %d %d" % (dev["bytes1"], dev["bytes2"], dev["bases"]))
            for k in opts:
                g.set_option(k, 0)
        a = g.generate_reads()
        for k in ("reads", "length", "pair_id", "segment", "pos", "frag"):
            h.update(a[k].cpu().numpy().tobytes())
        del a
        other = C.c_uint64()
        fd = os.open(fasta[0], os.O_RDONLY)
        try:
            cuda_binding._ck(L.ssc_reference_upload_fasta(g.h, fd, *fasta[1], C.byref(other)))
            cuda_binding._ck(L.ssc_reference_prefetch_fasta(g.h, fd, *fasta[1]))
            cuda_binding._ck(L.ssc_reference_adopt_prefetched(g.h, C.byref(other)))
        finally:
            os.close(fd)
        assert other.value == 0
    finally:
        g.close()
    return h.hexdigest()


def test_handles_free_what_they_allocate(built, tmp_path):
    """Three rounds, each of which creates a handle on a small PE XTen plan, runs plain, gzip + BGZF, interleaved and
    device-resident generation, array output and a FASTA prefetch, and destroys the handle: the free device memory after
    round 3 is within 4 MiB of that after round 1, and every round generates the same bytes."""
    scn = helpers.build_scenario("pe_xten", str(tmp_path))
    plan = planfile.read_plan(helpers.plan_dumps(scn, "life")[0])
    path = str(tmp_path / "chrA.fa")
    fasta = (path, write_fasta(path, 100000))
    digests = [one_round(plan, scn["seed"], fasta)]
    after1 = free_bytes()
    digests += [one_round(plan, scn["seed"], fasta) for _ in range(2)]
    after3 = free_bytes()
    assert digests[1:] == digests[:1] * 2
    assert abs(after3 - after1) <= 4 * MiB, "free device memory after round 1: %d, after round 3: %d" % (after1, after3)
