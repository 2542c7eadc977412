"""ssc_bam_header (no GPU): the header of the "bam" output's BAM stream as one stored BGZF block.

The block inflates with zlib to "BAM\\1", l_text, the @HD line (plus @RG with ID and SM when a read group is given) and n_ref = 0;
its BGZF fields (BSIZE, CRC-32, ISIZE) are right; bad read groups are refused and a short buffer gets 0."""
import ctypes as C
import struct
import zlib

import pytest

from simuscop_b200 import cuda_binding

BGZF_HEADER = bytes.fromhex("1f8b08040000000000ff060042430200")


@pytest.fixture(autouse=True)
def _library(built):
    return built


def expected_raw(rg):
    text = b"@HD\tVN:1.6\tSO:unsorted\tGO:query\n"
    if rg:
        text += b"@RG\tID:%s\tSM:%s\n" % (rg, rg)
    return b"BAM\x01" + struct.pack("<I", len(text)) + text + struct.pack("<I", 0)


def raw_call(rg, cap):
    buf = C.create_string_buffer(max(cap, 1))
    n = cuda_binding.lib().ssc_bam_header(rg, buf, cap)
    return n, buf.raw[:max(n, 0)]


@pytest.mark.parametrize("rg", [None, b"", b"A", b"sample_0.300+p2_0.250", b"!" + bytes(range(0x23, 0x7f))[:62] + b"~"])
def test_header_block(rg):
    raw = expected_raw(rg)
    blk = cuda_binding.bam_header(rg)
    assert len(blk) == len(raw) + 31
    assert blk[:16] == BGZF_HEADER and struct.unpack_from("<H", blk, 16)[0] == len(blk) - 1
    n = len(raw)
    assert blk[18:23] == bytes([1, n & 255, n >> 8, ~n & 255, (~n >> 8) & 255])        # one final stored block
    crc, isize = struct.unpack_from("<II", blk, len(blk) - 8)
    assert crc == zlib.crc32(raw) and isize == len(raw)
    d = zlib.decompressobj(wbits=31)
    assert d.decompress(blk) == raw and d.eof and not d.unused_data


def test_read_group_of_64_bytes():
    rg = bytes(range(0x21, 0x61))
    assert len(rg) == 64
    assert zlib.decompress(cuda_binding.bam_header(rg), wbits=31) == expected_raw(rg)


@pytest.mark.parametrize("rg", [b"a b", b"tab\t", b"x" * 65, b"\x7f", "é".encode()])
def test_bad_read_groups_are_refused(rg):
    assert raw_call(rg, 4096)[0] == -1
    with pytest.raises(cuda_binding.SscError):
        cuda_binding.bam_header(rg)


def test_short_buffer():
    full = len(cuda_binding.bam_header(b"rg1"))
    assert raw_call(b"rg1", full - 1)[0] == 0
    assert raw_call(b"rg1", 0)[0] == 0
    n, blk = raw_call(b"rg1", full)
    assert n == full and blk == cuda_binding.bam_header(b"rg1")
