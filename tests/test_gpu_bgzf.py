"""BGZF output (ssc_set_option "bgzf" with "gzip", SIMUSCOP_BGZF): every gzip member of the device encoder written as a BGZF
block, so htslib readers decompress the files in parallel and seek in them through the .gzi block index.

On one handle and range, each check compares four outputs: plain, plain with "bgzf" alone (no effect), gzip and gzip + bgzf,
the two compressed ones with the one Huffman table fitted after the plan was set.  Every BGZF stream is walked block by block:
the header is exact, the blocks tile the stream, none exceeds 64 KiB, each inflates on its own to whole FASTQ records (in
two-file PE, block k of both files to the same pairs), each equals the gzip member of the same ticket with FLG = FEXTRA and the
8-byte BC field, and the blocks concatenate to the plain bytes, which equal the oracle's.  The CLI files end with the EOF block
and every .gzi entry points at a block that inflates to the bytes at its uncompressed offset."""
import gzip
import os
import shutil
import struct
import subprocess
import zlib

import pytest

import helpers
from simuscop_b200 import planfile
from test_gpu_interleave import cli, interleave
from test_gpu_output_side import TICKET, bases, expanding_cases, split_members  # noqa: F401 (fixtures)
from test_gpu_plan_edges import load, profiles  # noqa: F401 (fixtures)

pytestmark = pytest.mark.gpu

HEADER = bytes.fromhex("1f8b08040000000000ff060042430200")
BGZF_EOF = bytes.fromhex("1f8b08040000000000ff0600424302001b0003000000000000000000")
BGZF_STORED_EXTRA = 31
assert len(HEADER) == 16


def to_bgzf(member):
    assert member[:4] == b"\x1f\x8b\x08\x00"
    return member[:3] + b"\x04" + member[4:10] + b"\x06\x00BC\x02\x00" + struct.pack("<H", len(member) + 8 - 1) + member[10:]


def walk(z):
    """The blocks of a BGZF stream: every header exactly HEADER + BSIZE, the blocks tile the stream, none over 65 536 bytes."""
    out, at = [], 0
    while at < len(z):
        assert z[at:at + 16] == HEADER, "block header at byte %d: %s" % (at, z[at:at + 18].hex())
        n = struct.unpack_from("<H", z, at + 16)[0] + 1
        assert 28 <= n <= 65536 and at + n <= len(z), (at, n, len(z))
        out.append(z[at:at + n])
        at += n
    return out


def inflate(block):
    d = zlib.decompressobj(wbits=31)
    raw = d.decompress(block)
    assert d.eof and not d.unused_data
    assert struct.unpack_from("<I", block, len(block) - 4)[0] == len(raw)
    return raw


def headers(raw):
    """The header lines of a run of whole FASTQ records (asserts that it is one)."""
    assert raw.startswith(b"@") and raw.endswith(b"\n")
    lines = raw.split(b"\n")[:-1]
    assert len(lines) % 4 == 0 and all(x == b"+" for x in lines[2::4])
    assert all(len(s) == len(q) for s, q in zip(lines[1::4], lines[3::4]))
    return lines[0::4]


def same_pairs(h1, h2):
    assert len(h1) == len(h2)
    for a, b in zip(h1, h2):
        assert a[:-1] == b[:-1] and a[-1:] == b"1" and b[-1:] == b"2", (a, b)


def check_range(g, lo=0, hi=None, want=None):
    """The four outputs of pairs [lo, hi) on handle g (plan loaded); want: the oracle's plain bytes.  Leaves gzip and bgzf off.
    Returns [[raw bytes of each block] per stream] and [[block] per stream]."""
    g.set_option("gzip", 0)
    g.set_option("bgzf", 0)
    plain = g.generate(lo, hi)
    if want is not None:
        assert plain == want
    g.set_option("bgzf", 1)
    assert g.generate(lo, hi) == plain                     # without gzip the option changes nothing
    g.set_option("gzip", 1)
    g.set_option("bgzf", 0)
    gz = g.generate(lo, hi)
    g.set_option("bgzf", 1)
    g.reset_stats()
    bg = g.generate(lo, hi)
    st = g.stats()
    assert st["gz_bytes"] == len(bg[0]) + len(bg[1]) and st["fastq_bytes"] == len(plain[0]) + len(plain[1])
    d = g.generate_device(lo, hi)
    assert (d["bytes1"], d["bytes2"]) == (len(bg[0]), len(bg[1])), d
    raws, blocks = [], []
    for f in range(2):
        if not plain[f]:
            assert bg[f] == b""
            continue
        bl, members = walk(bg[f]), split_members(gz[f])
        assert len(bl) == len(members), (len(bl), len(members))
        rs = []
        for j, (b, m) in enumerate(zip(bl, members)):
            assert b == to_bgzf(m), "file %d, block %d of %d bytes" % (f + 1, j, len(b))
            raw = inflate(b)
            headers(raw)
            if (b[18] >> 1) & 3 == 0:                    # stored
                assert b[18] == 1 and len(b) == len(raw) + BGZF_STORED_EXTRA
            rs.append(raw)
        assert b"".join(rs) == plain[f]
        raws.append(rs)
        blocks.append(bl)
    if len(raws) == 2:                                   # block k of _1 and of _2: the same pairs
        for r1, r2 in zip(*raws):
            same_pairs(headers(r1), headers(r2))
    g.set_option("gzip", 0)
    g.set_option("bgzf", 0)
    return raws, blocks


def scenario(name, workdir):
    scn = helpers.build_scenario(name, workdir)
    return planfile.read_plan(helpers.plan_dumps(scn, "bgzf")[0]), scn


SCENARIOS = {"pe_xten": ("pe_xten", {}), "pe_xten_interleaved": ("pe_xten", {"interleave": 1}),
             "pe_xten_batch256": ("pe_xten", {"batch_pairs": 256}), "se_gaiix": ("se_gaiix", {}),
             "pe_tiny": ("pe_tiny", {}), "pe_tiny_interleaved_batch256": ("pe_tiny", {"interleave": 1, "batch_pairs": 256})}


@pytest.mark.parametrize("name", SCENARIOS)
def test_parity_scenarios(name, built, workdir):
    """Two-file PE, SE, interleaved PE, and 256 pairs per batch (many batches: blocks of 8 tickets a batch), over the whole
    plan and over a range that starts and ends inside a ticket."""
    from oracle import binding as oracle_binding
    from simuscop_b200 import cuda_binding
    key, options = SCENARIOS[name]
    plan, scn = scenario(key, workdir)
    o1, o2, _ = oracle_binding.generate(plan, scn["seed"])
    g = cuda_binding.Generator(0)
    try:
        for k, v in options.items():
            g.set_option(k, v)
        g.load_plan(plan, scn["seed"])
        ilv = options.get("interleave") and plan.paired
        want = (interleave(o1, o2)[0], b"") if ilv else (o1, o2)
        raws, _ = check_range(g, want=want)
        assert len(raws) == (1 if ilv or not plan.paired else 2)
        if ilv:
            for r in raws[0]:                              # a block holds whole pairs, mate 1 then mate 2
                h = headers(r)
                same_pairs(h[0::2], h[1::2])
        if "batch_pairs" in options:
            assert len(raws[0]) >= 2 * (g.planned // options["batch_pairs"])
        P = g.planned
        check_range(g, TICKET + 5, P - 37)
        assert g.stats()["gen_kernel"] == 1
    finally:
        g.close()


@pytest.mark.parametrize("mode", ["xten", "xten_interleaved", "k3_160"])
def test_expanding_blocks_are_stored(mode, expanding_cases):  # noqa: F811
    """Tickets whose Huffman code would expand them: stored blocks of raw + 31 bytes, equal to the gzip member with the field
    inserted; interleaved, longer than any two-file block could be, and still below 64 KiB."""
    from simuscop_b200 import cuda_binding
    case = expanding_cases("k3_160" if mode == "k3_160" else "xten")
    g = cuda_binding.Generator(0)
    try:
        ilv = mode.endswith("interleaved")
        if ilv:
            g.set_option("interleave", 1)
        load(g, case)
        o1, o2 = case["o"]
        _, blocks = check_range(g, want=(interleave(o1, o2)[0], b"") if ilv else (o1, o2))
        stored = [b for bl in blocks for b in bl if (b[18] >> 1) & 3 == 0]
        assert len(stored) >= 64
        if ilv:
            assert max(len(b) for b in stored) > 20480 + BGZF_STORED_EXTRA
    finally:
        g.close()


# ---------------------------------------------------------------------------------------------------------------------------
# CLI
# ---------------------------------------------------------------------------------------------------------------------------
def check_file(data, plain, gzi):
    """A CLI output: BGZF blocks, the EOF block last, inflating to `plain`; gzi (bytes or None): the block index."""
    assert data.endswith(BGZF_EOF) and gzip.decompress(data) == plain
    blocks = walk(data)
    assert blocks[-1] == BGZF_EOF and all(len(b) > 28 for b in blocks[:-1])
    if gzi is None:
        return
    starts, c, u = [], 0, 0
    for b in blocks[:-1]:
        starts.append((c, u))
        c += len(b)
        u += struct.unpack_from("<I", b, len(b) - 4)[0]
    (n,) = struct.unpack_from("<Q", gzi)
    assert len(gzi) == 8 + 16 * n and n == len(blocks) - 2
    entries = [struct.unpack_from("<QQ", gzi, 8 + 16 * k) for k in range(n)]
    assert entries == starts[1:]
    for c, u in entries:
        blk = data[c:c + struct.unpack_from("<H", data, c + 16)[0] + 1]
        raw = inflate(blk)
        assert raw == plain[u:u + len(raw)]
        headers(raw)


CLI_CASES = {"pe": ("pe_tiny", {}), "interleaved": ("pe_tiny", {"SIMUSCOP_INTERLEAVE": "1"}), "se": ("se_gaiix", {})}


@pytest.mark.parametrize("name", CLI_CASES)
def test_cli_files(name, built, workdir):
    """SIMUSCOP_BGZF=1 (without SIMUSCOP_GZIP): <name>.fq.gz + <name>.fq.gz.gzi per stream, equal in content to the plain run."""
    key, env = CLI_CASES[name]
    scn = helpers.build_scenario(key, workdir)
    r, out = cli(scn, "bgzf_plain_" + name, **env)
    assert r.returncode == 0, r.stderr[-3000:]
    plain = {f: helpers.read_file(os.path.join(out, f)) for f in os.listdir(out)}
    r, out = cli(scn, "bgzf_" + name, SIMUSCOP_BGZF="1", **env)
    assert r.returncode == 0, r.stderr[-3000:]
    want = sorted([f + ".gz" for f in plain] + [f + ".gz.gzi" for f in plain])
    assert sorted(os.listdir(out)) == want and len(plain) == (2 if name == "pe" else 1)
    for f, p in plain.items():
        check_file(helpers.read_file(os.path.join(out, f + ".gz")), p, helpers.read_file(os.path.join(out, f + ".gz.gzi")))


def test_cli_stdout(built, workdir):
    """SIMUSCOP_STDOUT=1 SIMUSCOP_BGZF=1: the interleaved BGZF stream with its EOF block on standard output, and no index."""
    scn = helpers.build_scenario("pe_tiny", workdir)
    r, out = cli(scn, "bgzf_so_plain", SIMUSCOP_STDOUT="1")
    assert r.returncode == 0
    plain = r.stdout
    r, out = cli(scn, "bgzf_so", SIMUSCOP_STDOUT="1", SIMUSCOP_BGZF="1")
    assert r.returncode == 0, r.stderr[-3000:]
    check_file(r.stdout, plain, None)
    assert not os.path.exists(out) or os.listdir(out) == []


@pytest.mark.parametrize("devices", ["0,0,0", "0,1"])
def test_cli_several_handles(devices, built, workdir):
    """Batches of 256 pairs over several handles (one GPU three times, or two GPUs): the slabs pass the writer's turnstile in
    batch order, the files inflate to the one-handle run's bytes and the index offsets are global over the file."""
    import torch
    if devices == "0,1" and torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    scn = helpers.build_scenario("pe_tiny", workdir)
    tag = "bgzf_dev" + devices.replace(",", "")
    r, one = cli(scn, tag + "_one", SIMUSCOP_BGZF="1")
    assert r.returncode == 0
    r, out = cli(scn, tag, SIMUSCOP_BGZF="1", SIMUSCOP_DEVICES=devices, SIMUSCOP_BATCH_PAIRS="256")
    assert r.returncode == 0, r.stderr[-3000:]
    for f in ("test_1.fq.gz", "test_2.fq.gz"):
        plain = gzip.decompress(helpers.read_file(os.path.join(one, f)))
        data = helpers.read_file(os.path.join(out, f))
        check_file(data, plain, helpers.read_file(os.path.join(out, f + ".gzi")))
        pairs = len(plain.split(b"\n")) // 4
        assert len(walk(data)) - 1 >= -(-pairs // 256)                   # at least one block per batch


@pytest.mark.skipif(not (shutil.which("bgzip") or shutil.which("samtools")), reason="bgzip / samtools not installed")
def test_htslib_reads_the_files(built, workdir):
    """Where htslib's tools are installed: bgzip -t and a parallel bgzip -d accept the file, samtools fqidx indexes it."""
    scn = helpers.build_scenario("se_gaiix", workdir)
    r, out = cli(scn, "bgzf_hts_plain")
    assert r.returncode == 0
    plain = helpers.read_file(os.path.join(out, "test.fq"))
    r, out = cli(scn, "bgzf_hts", SIMUSCOP_BGZF="1")
    assert r.returncode == 0
    path = os.path.join(out, "test.fq.gz")
    if shutil.which("bgzip"):
        assert subprocess.run(["bgzip", "-t", path], capture_output=True).returncode == 0
        d = subprocess.run(["bgzip", "-d", "-@4", "-c", path], capture_output=True)
        assert d.returncode == 0 and d.stdout == plain
    if shutil.which("samtools"):
        assert subprocess.run(["samtools", "fqidx", path], capture_output=True).returncode == 0
        rec = plain.split(b"\n")[40:44]
        name = rec[0][1:].split()[0].decode()
        q = subprocess.run(["samtools", "fqidx", path, name], capture_output=True)
        assert q.returncode == 0 and q.stdout.split(b"\n")[0].split()[0] == rec[0].split()[0]
