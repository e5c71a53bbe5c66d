"""BGZF inputs for the tests of the CRC32 / ISIZE check: byte edits of `synth_bam.bam_bytes` output at known blocks, and
the 200k-read BAM of tests/_bam_bench.py.  The block table is read here on its own (bam_bytes writes the `BC` subfield
first), not with the reader under test."""
import struct


def block_offsets(raw):
    """File offset and size of every BGZF block of `raw`, in order."""
    out, p = [], 0
    while p < len(raw):
        bsize = struct.unpack_from("<H", raw, p + 16)[0] + 1
        out.append((p, bsize))
        p += bsize
    return out


def flip_payload(raw, k, at=100):
    """Byte `at` of block k's DEFLATE payload inverted.  For a stored (level 0) block, `at` >= 5 lands in the data."""
    b = bytearray(raw)
    p, _ = block_offsets(raw)[k]
    b[p + 18 + at] ^= 0xff
    return bytes(b)


def flip_crc(raw, k):
    """One byte of block k's CRC32 field inverted."""
    b = bytearray(raw)
    p, bsize = block_offsets(raw)[k]
    b[p + bsize - 8] ^= 0xff
    return bytes(b)


def set_isize(raw, k, isize):
    b = bytearray(raw)
    p, bsize = block_offsets(raw)[k]
    struct.pack_into("<I", b, p + bsize - 4, isize)
    return bytes(b)


def bench_bam(copies=10):
    """(BGZF bytes, primers) of tests/_bam_bench.py's input: 20 000 reads of make_alignments(seed=5) repeated `copies`
    times under distinct names, in blocks of 60 000 inflated bytes (10 copies: 200k reads, about 5 000 blocks)."""
    from fslr_b200 import synth_bam as sb
    refs, recs, primers = sb.make_alignments(20000, seed=5, p_unmapped=0.0)
    enc = [sb.encode_record(*r) for r in recs]
    big = [e[:36] + b"%02x" % c + e[38:] for c in range(copies) for e in enc]    # the first two name characters: the copy
    return sb.bam_bytes(refs, big), primers
