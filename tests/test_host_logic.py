"""Host-side logic on CPU: C-ABI symbols, exact threshold tables, plan parity of the C++ front end,
pair-ID sharding (gloo, world size 2)."""
import ctypes as C
import hashlib
import json
import os
import subprocess
import sys

import numpy as np
import pytest

import helpers
from oracle import binding as oracle_binding
from simuscop_b200 import cuda_binding, paths, planfile, sharding, synth, testdata

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def _declared(header):
    import re
    txt = open(os.path.join(paths.ROOT, "include", header)).read()
    return sorted(set(re.findall(r"\b(ss[ch]_[a-z0-9_]+)\s*\(", txt)) - {"ssc_sink_fn"})


def test_cuda_library_exports_every_declared_symbol(built):
    L = C.CDLL(paths.LIB_CUDA)
    names = _declared("simuscop.h")
    assert "ssc_generate" in names and len(names) >= 14
    for n in names:
        assert hasattr(L, n), n
    assert sorted(cuda_binding.SYMBOLS) == names


def test_host_library_exports_every_declared_symbol(built):
    L = C.CDLL(paths.LIB_HOST)
    for n in _declared("simuscop_host.h"):
        assert hasattr(L, n), n


def test_no_gpu_fails_loudly(built):
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    with pytest.raises(cuda_binding.SscError) as e:
        cuda_binding.Generator(0)
    assert "no CPU fallback" in str(e.value)


def test_threshold_tables_reproduce_randindx_at_every_boundary(built, tmp_path):
    """u32 thresholds == FP64 randIndx for draws at and around every table boundary, on real profile rows."""
    import gzip
    p = str(tmp_path / "p.plan")
    with gzip.open(os.path.join(GOLD, "pe_tiny.plan.gz"), "rb") as f, open(p, "wb") as g:
        g.write(f.read())
    plan = planfile.read_plan(p)
    L = cuda_binding.lib()
    O = oracle_binding.lib()
    rng = np.random.default_rng(5)
    t = plan.tables
    Q = plan.hdr["n_qual"]
    rows = [t["ins_cdf"], t["del_cdf"], t["isize_cdf"]]
    qual = t["quality_cdf"].reshape(-1, Q)
    rows += [qual[i] for i in rng.integers(0, qual.shape[0], 12)]
    rows += [np.zeros(5), np.array([0.0, 0.0, 1.0, 1.0]), np.array([1e-17, 0.5, 0.5, 0.9]), np.array([0.3, 0.2, 0.9, 0.8])]
    for cdf in rows:
        cdf = np.ascontiguousarray(cdf, dtype=np.float64)
        us = {0, 1, 2, 0xFFFFFFFF, 0xFFFFFFFE, 0x80000000}
        for c in np.unique(cdf):
            # u such that r(u) is closest to c, and its neighbours
            u0 = int(min(max((float(c) - 2.2204e-16) / (1 - 2.2204e-16) * 4294967296.0, 0), 4294967295))
            us.update(max(0, min(0xFFFFFFFF, u0 + d)) for d in range(-3, 4))
        us.update(int(x) for x in rng.integers(0, 1 << 32, 200, dtype=np.uint64))
        for u in us:
            assert L.ssc_table_lookup_host(cdf.ctypes.data, cdf.size, u) == O.ssco_rand_indx(cdf.ctypes.data, cdf.size, u), (u, cdf[:6])
    sub = t["subs_cdf1"].reshape(-1, 4)
    for i in list(rng.integers(0, sub.shape[0], 40)) + [0, sub.shape[0] - 1]:
        cdf = np.ascontiguousarray(sub[i])
        us = {0, 1, 0xFFFFFFFF, 0xFFFFFFFE}
        for c in cdf:
            u0 = int(min(max((float(c) - 2.2204e-16) / (1 - 2.2204e-16) * 4294967296.0, 0), 4294967295))
            us.update(max(0, min(0xFFFFFFFF, u0 + d)) for d in range(-2, 3))
        us.update(int(x) for x in rng.integers(0, 1 << 32, 50, dtype=np.uint64))
        for u in us:
            assert L.ssc_sub_lookup_host(cdf.ctypes.data, u) == O.ssco_rand_indx(cdf.ctypes.data, 4, u)


@pytest.mark.parametrize("name", ["pe_xten", "se_gaiix", "pe_tiny", "pe_variants", "pe_wes", "se_tumor", "pe_ploidy3", "se_ploidy1", "pe_iupac"])
def test_host_plan_matches_golden_hashes(name, built, workdir):
    """Tables, haplotypes (SNP/SNV/indel/CNV), bins and read counts of the C++ front end, byte for byte."""
    scn = helpers.build_scenario(name, workdir)
    ours = helpers.plan_dumps(scn, "ours")
    gold = json.load(open(os.path.join(GOLD, "golden.json")))[name]
    assert len(ours) == len(gold["samples"])
    for pf, s in zip(ours, gold["samples"]):
        assert hashlib.sha256(open(pf, "rb").read()).hexdigest() == s["plan_sha256"]


def _outcome(scn, tag):
    """Exit code, last message and plan sha256 of the front end on `scn`, as stored for the reference in tests/golden/fuzz.json."""
    d = scn["dir"]
    cfg = os.path.join(d, "cfg_%s.txt" % tag)
    synth.write_config(cfg, output=os.path.join(d, "out_" + tag), **scn["kw"])
    return helpers.plan_outcome(paths.SIMUREADS, cfg, os.path.join(d, "p_" + tag), scn["seed"], d)


@pytest.mark.parametrize("seed", helpers.FUZZ_VARIATION_SEEDS)
def test_host_plan_equals_the_instrumented_reference_on_random_variation_sets(seed, built, workdir):
    """Plan-construction fuzz (CPU only): random CNV / insertion / deletion / SNV files, ploidy 1..3, PE and SE.  The plan dump of the
    C++ front end (tables, rand()-phased haplotypes, bins, read counts) must equal the instrumented reference's dump byte for byte
    (its sha256, tests/golden/fuzz.json)."""
    scn = helpers.build_random_variation_scenario(seed, workdir)
    gold = helpers.golden_entry(scn["name"])
    rc, msg, plans = _outcome(scn, "ours")
    assert rc == gold["returncode"] == 0, msg
    assert plans == gold["plan_sha256"] and plans, (seed, open(scn["kw"]["variation"]).read())


@pytest.mark.parametrize("seed", helpers.FUZZ_JOB_SEEDS)
def test_host_plan_equals_the_instrumented_reference_on_random_jobs(seed, built, workdir):
    """The same fuzz over the other inputs: multi-chromosome genomes, capture targets, SNP files on both strands, tumour mixtures
    with per-population variations (seeds chosen to cover every mode)."""
    scn, mode = helpers.build_random_job_scenario(seed, workdir)
    gold = helpers.golden_entry(scn["name"])
    rc, msg, plans = _outcome(scn, "ours")
    assert rc == gold["returncode"] == 0, (mode, msg)
    assert plans == gold["plan_sha256"] and plans, (seed, mode)


@pytest.mark.parametrize("gen,seed", helpers.EDGE_CASES)
def test_host_plan_equals_the_instrumented_reference_on_edge_case_inputs(gen, seed, built, workdir):
    """One seed per kind of helpers.build_edge_variation_scenario (53: an input both programs reject with the same message) and of
    helpers.build_edge_input_scenario (capture targets, SNP files, abundance files): the reference's exit code, and its last
    message on a rejected input or its plan dumps otherwise."""
    scn, kind = (helpers.build_edge_variation_scenario if gen == "variation" else helpers.build_edge_input_scenario)(seed, workdir)
    gold = helpers.golden_entry(scn["name"])
    rc, msg, plans = _outcome(scn, "ours")
    assert rc == gold["returncode"], (kind, rc, gold["returncode"], msg, gold.get("message"))
    if rc != 0:
        assert msg == gold["message"], kind
    else:
        assert plans == gold["plan_sha256"] and plans, kind


def test_unphaseable_haploid_gain_is_rejected_not_spun_on(built, tmp_path):
    """ploidy 1 with a copy-number gain whose major copy number is smaller than the copy number: the reference never leaves the
    loop at Segment.cpp:183-189 (it looks for a second haplotype index); the replacement reports the segment and exits."""
    d = str(tmp_path)
    synth.make_genome(os.path.join(d, "ref.fa"), [300000], seed=3, names=["chr20"])
    with open(os.path.join(d, "variations.txt"), "w") as f:
        f.write("c\ttest\tchr20\t100001\t200000\t4\t3\n")
    data = testdata.materialize(os.path.join(d, "data"))
    cfg = os.path.join(d, "cfg.txt")
    synth.write_config(cfg, output=os.path.join(d, "out"), ref=os.path.join(d, "ref.fa"), profile=os.path.join(data, testdata.PROFILES["XTen"]),
                       layout="PE", coverage=1, insertSize=300, threads=1, verbose=0, name="test", ploidy=1,
                       variation=os.path.join(d, "variations.txt"))
    r = subprocess.run([paths.SIMUREADS, cfg], env=dict(os.environ, SIMUSCOP_PLAN_ONLY="1", SIMUSCOP_DUMP_PLAN=os.path.join(d, "plan"), SIMUSCOP_SEED="1"), capture_output=True,
                       text=True, timeout=120)
    assert r.returncode == 1 and "cannot be phased with ploidy 1" in r.stderr, r.stderr[-500:]


def test_cli_argument_and_config_errors(built, tmp_path):
    r = subprocess.run([paths.SIMUREADS], capture_output=True, text=True)
    assert r.returncode == 1 and "configuration file is required" in r.stderr
    r = subprocess.run([paths.SIMUREADS, "a", "b"], capture_output=True, text=True)
    assert r.returncode == 1 and "too many input arguments" in r.stderr
    cfg = tmp_path / "c.txt"
    cfg.write_text("ref = x.fa\nprofile = p\nname = t\noutput = o\ncoverage = 1\nbogus = 1\n")
    r = subprocess.run([paths.SIMUREADS, str(cfg)], capture_output=True, text=True)
    assert r.returncode == 1 and 'unrecognized item "bogus"' in r.stderr
    cfg.write_text("ref = x.fa\nname = t\noutput = o\ncoverage = 1\n")
    r = subprocess.run([paths.SIMUREADS, str(cfg)], capture_output=True, text=True)
    assert r.returncode == 1 and "sequencing profile must be specified" in r.stderr


def test_config_matrix_behaves_like_the_reference(built, tmp_path):
    """Config grammar and validation (lib/config/Config.cpp:46-99 and the checks of simuReads.cpp): for a matrix of missing keys,
    bad values, missing input files and formatting variants (helpers.config_matrix), the replacement CLI exits with the
    reference's code and last message, and on success dumps the reference's plan byte for byte (tests/golden/fuzz.json).  Where
    the reference dies of an uncaught exception (insertSize below the read length: std::bad_array_new_length, SIGABRT) the
    replacement reports the problem and exits 1."""
    wd = str(tmp_path)
    gold = helpers.golden_entry("config_matrix")
    cases, aborts = helpers.config_matrix(wd)
    assert sorted(label for label, _ in cases) == sorted(gold["cases"])

    def run(text):
        cfg = os.path.join(wd, "c_ours.txt")
        with open(cfg, "w") as f:
            f.write(text)
        return helpers.plan_outcome(paths.SIMUREADS, cfg, os.path.join(wd, "p_ours"), 1, wd)

    for label, text in cases:
        want = gold["cases"][label]
        rc, msg, plans = run(text)
        assert rc == want["returncode"], (label, rc, want, msg)
        if rc != 0:
            assert msg == want["message"], (label, msg, want["message"])
        else:
            assert plans == want["plan_sha256"] and plans, label
    # the reference aborts here; the replacement says why
    rc, msg, _ = run(aborts)
    assert gold["insert_size_below_read_length"]["returncode"] < 0 and rc == 1 and "insert size" in msg


def test_shard_ranges_partition():
    for planned in (0, 1, 7, 1000, 298013245):
        for world in (1, 2, 3, 8):
            rs = [sharding.shard_range(planned, r, world) for r in range(world)]
            assert rs[0][0] == 0 and rs[-1][1] == planned
            assert all(a[1] == b[0] for a, b in zip(rs[:-1], rs[1:]))
            assert max(h - l for l, h in rs) - min(h - l for l, h in rs) <= 1


_WORKER = r"""
import os, sys, gzip
sys.path.insert(0, sys.argv[1]); sys.path.insert(0, os.path.join(sys.argv[1], "tests"))
import torch, torch.distributed as dist
from oracle import binding as oracle_binding
from simuscop_b200 import planfile, sharding
dist.init_process_group("gloo")
rank, world = dist.get_rank(), dist.get_world_size()
plan = planfile.read_plan(sys.argv[2])
lo, hi = sharding.shard_range(plan.planned_pairs(), rank, world)
f1, f2, info = oracle_binding.generate(plan, 7, lo, hi)
out = [None] * world
dist.all_gather_object(out, (lo, hi, f1, f2))
if rank == 0:
    w1, w2, _ = oracle_binding.generate(plan, 7)
    out.sort()
    assert b"".join(o[2] for o in out) == w1 and b"".join(o[3] for o in out) == w2
    open(sys.argv[3], "w").write("ok %d" % world)
dist.barrier()
dist.destroy_process_group()
"""


def test_two_rank_sharding_concatenates_to_single_rank_output(built, tmp_path):
    """world_size 2 over gloo: each rank generates its pair-ID range (with the CPU checker standing in for a
    GPU); the shards in rank order are byte-identical to the unsharded output."""
    import gzip
    p = str(tmp_path / "p.plan")
    with gzip.open(os.path.join(GOLD, "pe_tiny.plan.gz"), "rb") as f, open(p, "wb") as g:
        g.write(f.read())
    w = tmp_path / "worker.py"
    w.write_text(_WORKER)
    flag = str(tmp_path / "ok.txt")
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2",
                        "--master-addr", "127.0.0.1", "--master-port", "29517", str(w), paths.ROOT, p, flag],
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-3000:]
    assert open(flag).read() == "ok 2"


def test_gzip_member_host_mirror_inflates(built):
    """The device gzip encoder's tables and algebra on the host (ssc_gzip_member_host: Huffman code fitted to a sample,
    dynamic block header, bit packing, lane-strided CRC-32 combination): zlib must accept every member."""
    import ctypes as C
    import gzip
    import random
    L = cuda_binding.lib()
    rnd = random.Random(7)

    def fastq(n):
        rec = []
        for i in range(n):
            ln = rnd.choice([151, 150, 149, 152, 96])
            rec.append("@test#chr%d#%d#%d/1\n%s\n+\n%s\n" % (rnd.randint(1, 22), rnd.randint(0, 999999), i + 1,
                       "".join(rnd.choice("ACGT") for _ in range(ln)), "".join(rnd.choice("FFFFFFF:A<,#") for _ in range(ln))))
        return "".join(rec).encode()
    sample = fastq(100)
    members = []
    for n, cut in ((1, 0), (2, 1), (32, 2), (33, 3), (64, 0)):
        d = fastq(n)
        d = d[:len(d) - cut] if cut else d
        buf = C.create_string_buffer(2 * len(d) + 1024)
        m = L.ssc_gzip_member_host(d, len(d), sample, len(sample), buf, len(buf))
        assert m > 0
        assert gzip.decompress(buf.raw[:m]) == d
        members.append((d, buf.raw[:m]))
    assert gzip.decompress(b"".join(z for _, z in members)) == b"".join(d for d, _ in members)
    noise = bytes(rnd.randrange(256) for _ in range(4099))          # every byte value stays encodable
    buf = C.create_string_buffer(4 * len(noise))
    m = L.ssc_gzip_member_host(noise, len(noise), sample, len(sample), buf, len(buf))
    assert gzip.decompress(buf.raw[:m]) == noise


def test_gzip_member_host_stores_what_coding_would_expand(built):
    """A member whose Huffman code (fitted to the sample) would be longer than its bytes + 23 is one stored block: gzip header,
    0x01, LEN, NLEN, the bytes, CRC-32, ISIZE -- what zlib does, and what the device encoder does too.  Inputs: noise, bytes
    absent from the sample (codes of 14-15 bits; up to the largest blob, 32 x 612 bytes), and 1..15 bytes (no or one full
    word pair, less than the block header).  Members that coding does not expand stay coded (BTYPE 2)."""
    import ctypes as C
    import random
    import struct
    import zlib
    L = cuda_binding.lib()
    rnd = random.Random(11)
    sample = b"".join(b"@normal#chr1#%d#%d/1\n%s\n+\n%s\n" % (rnd.randint(0, 99999), i + 1,
                                                              bytes(rnd.choice(b"ACGT") for _ in range(151)),
                                                              bytes(rnd.choice(b"FFF:,") for _ in range(151)))
                      for i in range(64))
    absent = bytes(sorted(set(range(256)) - set(sample)))
    assert len(absent) > 200

    def member(d):
        buf = C.create_string_buffer(len(d) + 4096)
        m = L.ssc_gzip_member_host(d, len(d), sample, len(sample), buf, len(buf))
        assert m > 0
        return buf.raw[:m]

    def stored(d):
        n = len(d)
        return (b"\x1f\x8b\x08\x00\x00\x00\x00\x00\x00\xff" + struct.pack("<BHH", 1, n, n ^ 0xFFFF) + d +
                struct.pack("<II", zlib.crc32(d), n))
    expanding = [bytes(rnd.randrange(256) for _ in range(4099)), absent * 3, (absent * 100)[:32 * 612],
                 b"@" + absent[:63] + b"\n" + bytes(rnd.choice(b"!\"#$%&'()*+,-./0123456") for _ in range(8000)),
                 absent[:1], absent[:7], bytes(absent[:5]) * 3, sample[:1], sample[100:107]]   # short: a ~60-byte table
    for d in expanding:
        z = member(d)
        assert z == stored(d) and len(z) == len(d) + 23, len(d)
        assert zlib.decompressobj(wbits=31).decompress(z) == d
    for d in [sample[:4096], sample[:1001], sample[5:613]]:
        z = member(d)
        assert len(z) <= len(d) + 23 and (z[10] >> 1) & 3 == 2 and zlib.decompressobj(wbits=31).decompress(z) == d
    assert len(member(sample[:4096])) < 4096 // 2
    buf = C.create_string_buffer(len(expanding[0]) + 22)                      # one byte short of the stored member
    assert L.ssc_gzip_member_host(expanding[0], len(expanding[0]), sample, len(sample), buf, len(buf)) == 0


def test_file_writer_sink_writes_ordered_slabs(built, tmp_path):
    """The output side of the drop-in CLI (ssh_writer_*, the role of SeqWriter::write): slabs handed to the sink in order end
    up back to back in the files, whatever the number of pwrite workers, for paired and single-end layouts."""
    import numpy as np
    from simuscop_b200 import abi, host_binding
    hl = host_binding.lib()
    hl.ssh_writer_open.argtypes = [C.c_char_p, C.c_char_p, C.c_int, C.POINTER(C.c_void_p)]
    hl.ssh_writer_sink.restype = C.c_void_p
    hl.ssh_writer_close.argtypes = [C.c_void_p, C.POINTER(C.c_uint64), C.POINTER(C.c_uint64)]
    sink = C.cast(hl.ssh_writer_sink(), abi.SINK_FN)
    rng = np.random.default_rng(3)
    for threads, paired, mode in ((1, True, None), (5, True, None), (3, False, None), (5, True, "mmap"), (3, False, "mmap"),
                                  (5, True, "hybrid"), (2, True, "hybrid"), (4, False, "hybrid")):
        # default: one pwrite stream per file; SIMUSCOP_WRITER_MODE=mmap: the pool copies 8 MiB chunks into mappings of the
        # files; hybrid: a stream per file from the front, the other threads through mappings from the back
        os.environ.pop("SIMUSCOP_WRITER_MODE", None)
        if mode:
            os.environ["SIMUSCOP_WRITER_MODE"] = mode
        p1, p2 = str(tmp_path / ("w%d%s_1.fq" % (threads, mode))), str(tmp_path / ("w%d%s_2.fq" % (threads, mode)))
        w = C.c_void_p()
        assert hl.ssh_writer_open(p1.encode(), p2.encode() if paired else None, threads, C.byref(w)) == 0
        want1, want2 = b"", b""
        for n in (0, 1, 17, (8 << 20) - 1, (8 << 20) + 5, 20 << 20):          # around the 8 MiB chunk size of the pool
            a = rng.integers(0, 256, n, dtype=np.uint8).tobytes()
            b = rng.integers(0, 256, n // 2 + 3, dtype=np.uint8).tobytes() if paired else b""
            assert sink(w, a, len(a), b if paired else None, len(b), 0, 0) == 0
            want1 += a; want2 += b
        b1, b2 = C.c_uint64(), C.c_uint64()
        assert hl.ssh_writer_close(w, C.byref(b1), C.byref(b2)) == 0
        assert (b1.value, b2.value) == (len(want1), len(want2))
        assert open(p1, "rb").read() == want1
        if paired:
            assert open(p2, "rb").read() == want2
        else:
            assert not os.path.exists(p2)
    os.environ.pop("SIMUSCOP_WRITER_MODE", None)
    assert hl.ssh_writer_open(str(tmp_path / "no" / "such" / "dir.fq").encode(), None, 2, C.byref(C.c_void_p())) != 0


@pytest.mark.parametrize("kind,seed", [("scenario", "pe_variants"), ("scenario", "se_tumor"), ("scenario", "pe_ploidy3"), ("scenario", "pe_iupac")] +
                         [("fuzz", s) for s in (11, 12, 13, 14, 15, 16, 21, 22, 23)] + [("edge", s) for s in (0, 1, 3, 5, 6, 7, 14, 17)])
def test_splice_lists_equal_haplotype_strings(kind, seed, built, workdir):
    """Segments with insertion / deletion variants are assembled on the device from splice lists (runs of the reference slice
    + inserted literals, substitutions mapped onto the surviving runs).  Materialised on the host, every such list must give
    the haplotype string of the string construction -- which the plan-dump tests pin against the instrumented reference --
    for CNV gains / losses with tandem copies, homo- and heterozygous indels and SNVs, SNPs, indels at segment edges and
    inside CNVs, triploid genomes, tumour populations."""
    from simuscop_b200 import host_binding
    if kind == "scenario":
        scn = helpers.build_scenario(seed, workdir)
    elif kind == "fuzz":
        scn = helpers.build_random_variation_scenario(seed, workdir)
    else:
        scn, _ = helpers.build_edge_variation_scenario(seed, workdir)
    cfg = os.path.join(scn["dir"], "cfg_splice.txt")
    synth.write_config(cfg, output=os.path.join(scn["dir"], "out_splice"), **scn["kw"])
    hl = host_binding.lib()
    hl.ssh_selftest_splices.argtypes = [C.c_void_p, C.POINTER(C.c_int64), C.POINTER(C.c_int64)]
    # (a config the front end rejects exits the process, like the reference: run the check in a child)
    code = ("import ctypes as C, sys; sys.path.insert(0, %r); from simuscop_b200 import host_binding as hb; j = hb.Job(%r, %d); "
            "hl = hb.lib(); hl.ssh_selftest_splices.argtypes = [C.c_void_p, C.POINTER(C.c_int64), C.POINTER(C.c_int64)]; "
            "n, k = C.c_int64(), C.c_int64(); bad = hl.ssh_selftest_splices(j.j, C.byref(n), C.byref(k)); print('RESULT', bad, n.value, k.value)"
            % (paths.ROOT, cfg, scn["seed"]))
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, cwd=scn["dir"])
    if r.returncode != 0:
        pytest.skip("input rejected by the front end (as by the reference): %s" % r.stderr.strip().split("\n")[-1][:120])
    bad, n, k = [int(x) for x in [l for l in r.stdout.splitlines() if l.startswith("RESULT")][0].split()[1:]]
    assert bad == 0 and n > 0, (bad, n, k)


def test_bench_count_bases_streams_exactly(tmp_path):
    """bench.py's reference arm counts the emitted bases of multi-GB FASTQ files in constant memory: the streaming count must
    equal the naive one, also when a buffer boundary cuts a line."""
    import gzip
    import bench
    data = gzip.open(os.path.join(GOLD, "pe_tiny_1.fq.gz")).read()
    p = tmp_path / "a.fq"
    p.write_bytes(data * 3)
    want = 3 * sum(len(x) for x in data.split(b"\n")[1::4])
    assert bench.count_bases([str(p)]) == want
    real_open = open

    class Tiny:                                # 1000-byte reads: every kind of boundary position occurs
        def __init__(self, f): self.f = f
        def read(self, n): return self.f.read(min(n, 1000))
        def __enter__(self): return self
        def __exit__(self, *a): self.f.close()
    import builtins
    old = builtins.open
    builtins.open = lambda path, mode="r", *a, **k: Tiny(real_open(path, mode, *a, **k)) if str(path) == str(p) else real_open(path, mode, *a, **k)
    try:
        assert bench.count_bases([str(p)]) == want
    finally:
        builtins.open = old
