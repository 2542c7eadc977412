"""The BGZF side of the file writer (ssh_writer_bgzf), without a GPU: slabs of BGZF blocks end up back to back in the files,
each stream ends with the 28-byte BGZF EOF block, each .gzi holds the start of every block after the first with the running
ISIZE sum (htslib's bgzf_index_dump layout), and a slab that is not whole BGZF blocks makes the sink and the close fail.

The blocks are the host mirror's gzip members (ssc_gzip_member_host) with the BGZF extra field inserted, which is how the
device encoder's "bgzf" blocks relate to its "gzip" members."""
import ctypes as C
import gzip
import os
import random
import struct
import zlib

import pytest

from simuscop_b200 import abi, cuda_binding, host_binding

BGZF_EOF = bytes.fromhex("1f8b08040000000000ff0600424302001b0003000000000000000000")
SSC_ERR_INVALID, SSC_ERR_STATE, SSC_ERR_SINK = 1, 3, 5


def fastq(rnd, n, mate=1):
    return b"".join(b"@bgzf#chr%d#%d#%d/%d\n%s\n+\n%s\n" % (rnd.randint(1, 22), rnd.randint(0, 999999), i + 1, mate,
                                                           bytes(rnd.choice(b"ACGT") for _ in range(151)),
                                                           bytes(rnd.choice(b"FF:,#") for _ in range(151)))
                    for i in range(n))


def to_bgzf(member):
    """A gzip member (10-byte header, no FLG bits) as a BGZF block: FLG = FEXTRA and XLEN 6, 'B' 'C', SLEN 2, BSIZE inserted."""
    assert member[:4] == b"\x1f\x8b\x08\x00"
    return member[:3] + b"\x04" + member[4:10] + b"\x06\x00BC\x02\x00" + struct.pack("<H", len(member) + 8 - 1) + member[10:]


@pytest.fixture(scope="module")
def blocks(built):
    """Two streams of BGZF blocks (coded and stored) of 1..32 records each: [(raw, block)] per stream."""
    L = cuda_binding.lib()
    rnd = random.Random(5)
    sample = fastq(rnd, 64)
    out = []
    for mate in (1, 2):
        s = []
        for n in [1, 32, 7, 32, 32, 2, 17, 32, 5, 32, 32, 1]:
            raw = fastq(rnd, n, mate)
            if n == 7:                        # bytes the sample lacks: a stored block
                raw = raw.translate(bytes.maketrans(b"ACGT", b"\x90\x91\x92\x93"))
            buf = C.create_string_buffer(len(raw) + 4096)
            m = L.ssc_gzip_member_host(raw, len(raw), sample, len(sample), buf, len(buf))
            assert m > 0
            s.append((raw, to_bgzf(buf.raw[:m])))
        assert any(b[18] == 1 for _, b in s) and any((b[18] >> 1) & 3 == 2 for _, b in s)   # stored and coded blocks
        out.append(s)
    return out


def writer_lib():
    hl = host_binding.lib()
    hl.ssh_writer_open.argtypes = [C.c_char_p, C.c_char_p, C.c_int, C.POINTER(C.c_void_p)]
    hl.ssh_writer_open_fd.argtypes = [C.c_int, C.POINTER(C.c_void_p)]
    hl.ssh_writer_bgzf.argtypes = [C.c_void_p, C.c_char_p, C.c_char_p]
    hl.ssh_writer_sink.restype = C.c_void_p
    hl.ssh_writer_close.argtypes = [C.c_void_p, C.POINTER(C.c_uint64), C.POINTER(C.c_uint64)]
    return hl, C.cast(hl.ssh_writer_sink(), abi.SINK_FN)


def slabs_of(stream, cuts):
    """The blocks of a stream cut into slabs at the given block indices (an empty slab where two cuts meet)."""
    data = [b for _, b in stream]
    bounds = [0] + list(cuts) + [len(data)]
    return [b"".join(data[a:b]) for a, b in zip(bounds, bounds[1:])]


def expected_index(stream):
    entries, c, u = [], 0, 0
    for j, (raw, blk) in enumerate(stream):
        if j:
            entries.append((c, u))
        c += len(blk)
        u += len(raw)
    return struct.pack("<Q", len(entries)) + b"".join(struct.pack("<QQ", a, b) for a, b in entries)


def check_stream(path, index, stream):
    data = open(path, "rb").read()
    assert data == b"".join(b for _, b in stream) + BGZF_EOF
    assert gzip.decompress(data) == b"".join(r for r, _ in stream)
    if index:
        gzi = open(index, "rb").read()
        assert gzi == expected_index(stream)
        (n,) = struct.unpack_from("<Q", gzi)
        assert n == len(stream) - 1
        for k in range(n):                # every entry: a block that inflates on its own to the bytes at its offset
            c, u = struct.unpack_from("<QQ", gzi, 8 + 16 * k)
            blk = data[c:c + struct.unpack_from("<H", data, c + 16)[0] + 1]
            assert zlib.decompressobj(wbits=31).decompress(blk) == stream[k + 1][0]
            assert u == sum(len(r) for r, _ in stream[:k + 1])


@pytest.mark.parametrize("threads", [1, 4])
def test_two_files_and_their_indexes(threads, blocks, tmp_path):
    """PE: both files are their blocks and the EOF block, whatever the slab cuts; both indexes are exact."""
    hl, sink = writer_lib()
    p1, p2 = str(tmp_path / "r_1.fq.gz"), str(tmp_path / "r_2.fq.gz")
    w = C.c_void_p()
    assert hl.ssh_writer_open(p1.encode(), p2.encode(), threads, C.byref(w)) == 0
    assert hl.ssh_writer_bgzf(w, (p1 + ".gzi").encode(), (p2 + ".gzi").encode()) == 0
    s1, s2 = slabs_of(blocks[0], [1, 1, 4, 9]), slabs_of(blocks[1], [1, 1, 4, 9])
    for a, b in zip(s1, s2):
        assert sink(w, a, len(a), b, len(b), 0, 0) == 0
    b1, b2 = C.c_uint64(), C.c_uint64()
    assert hl.ssh_writer_close(w, C.byref(b1), C.byref(b2)) == 0
    assert (b1.value, b2.value) == (sum(map(len, s1)) + 28, sum(map(len, s2)) + 28)
    check_stream(p1, p1 + ".gzi", blocks[0])
    check_stream(p2, p2 + ".gzi", blocks[1])


def test_single_file_without_index_and_one_slab(blocks, tmp_path):
    hl, sink = writer_lib()
    p = str(tmp_path / "se.fq.gz")
    w = C.c_void_p()
    assert hl.ssh_writer_open(p.encode(), None, 2, C.byref(w)) == 0
    assert hl.ssh_writer_bgzf(w, None, b"x.gzi") == SSC_ERR_INVALID          # no second file to index
    assert hl.ssh_writer_bgzf(w, None, None) == 0
    assert hl.ssh_writer_bgzf(w, None, None) == SSC_ERR_STATE
    (a,) = slabs_of(blocks[0], [])
    assert sink(w, a, len(a), None, 0, 0, 0) == 0
    assert hl.ssh_writer_close(w, None, None) == 0
    check_stream(p, None, blocks[0])
    assert os.listdir(tmp_path) == ["se.fq.gz"]


def test_descriptor(blocks, tmp_path):
    """A writer on a descriptor (standard output in the CLI) appends the EOF block too, and may keep an index."""
    hl, sink = writer_lib()
    p = str(tmp_path / "fd.fq.gz")
    fd = os.open(p, os.O_WRONLY | os.O_CREAT | os.O_TRUNC, 0o644)
    try:
        w = C.c_void_p()
        assert hl.ssh_writer_open_fd(fd, C.byref(w)) == 0
        assert hl.ssh_writer_bgzf(w, (p + ".gzi").encode(), None) == 0
        for a in slabs_of(blocks[1], [3, 6, 6, 11]):
            assert sink(w, a, len(a), None, 0, 0, 0) == 0
        assert hl.ssh_writer_close(w, None, None) == 0
    finally:
        os.close(fd)
    check_stream(p, p + ".gzi", blocks[1])


def test_bgzf_only_before_the_first_slab(blocks, tmp_path):
    hl, sink = writer_lib()
    w = C.c_void_p()
    assert hl.ssh_writer_open(str(tmp_path / "late.fq.gz").encode(), None, 1, C.byref(w)) == 0
    a = blocks[0][0][1]
    assert sink(w, a, len(a), None, 0, 0, 0) == 0
    assert hl.ssh_writer_bgzf(w, None, None) == SSC_ERR_STATE
    assert hl.ssh_writer_close(w, None, None) == 0
    assert open(str(tmp_path / "late.fq.gz"), "rb").read() == a      # a plain writer: no EOF block


def bad_slabs(blocks):
    """Slabs that are not whole BGZF blocks: a truncated block, a plain gzip member, a BSIZE past the slab, a bad subfield."""
    good = blocks[0][1][1]
    member = good[:3] + b"\x00" + good[4:10] + good[18:]
    bsize_long = good[:16] + struct.pack("<H", len(good)) + good[18:]
    sub = good[:12] + b"BD" + good[14:]
    return {"truncated": good + good[:-1], "gzip_member": good + member, "bsize_past_slab": bsize_long,
            "subfield": sub, "short": good[:20]}


@pytest.mark.parametrize("kind", ["truncated", "gzip_member", "bsize_past_slab", "subfield", "short"])
@pytest.mark.parametrize("paired", [False, True])
def test_malformed_slab_fails(kind, paired, blocks, tmp_path):
    """The sink returns non-zero, takes no further slab, writes nothing of the bad slab, and the close reports the failure
    without appending the EOF block."""
    hl, sink = writer_lib()
    p1, p2 = str(tmp_path / "bad_1.fq.gz"), str(tmp_path / "bad_2.fq.gz")
    w = C.c_void_p()
    assert hl.ssh_writer_open(p1.encode(), p2.encode() if paired else None, 2, C.byref(w)) == 0
    assert hl.ssh_writer_bgzf(w, (p1 + ".gzi").encode(), (p2 + ".gzi").encode() if paired else None) == 0
    g1, g2 = blocks[0][0][1], blocks[1][0][1]
    assert sink(w, g1, len(g1), g2 if paired else None, len(g2) if paired else 0, 0, 0) == 0
    bad = bad_slabs(blocks)[kind]
    if paired:                            # the bad slab in file 2: file 1's good slab of the same call is not written either
        assert sink(w, g1, len(g1), bad, len(bad), 0, 0) != 0
    else:
        assert sink(w, bad, len(bad), None, 0, 0, 0) != 0
    assert sink(w, g1, len(g1), g2 if paired else None, len(g2) if paired else 0, 0, 0) != 0
    assert hl.ssh_writer_close(w, None, None) == SSC_ERR_SINK
    assert open(p1, "rb").read() == g1
    if paired:
        assert open(p2, "rb").read() == g2
