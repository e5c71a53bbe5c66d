"""CPU tests of the host BGZF readers (mapping_info.inflate_bgzf, mapping_info.bgzf_header_prefix,
cluster.get_chromosome_lengths): a block whose inflated bytes do not match its CRC32 or ISIZE is refused with a
ValueError naming the block and its file offset, as htslib refuses it; valid files read as before."""
import gzip
import json
import os
import re

import numpy as np
import pytest

from tests import bgzf_cases as bc

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CASES_DIR = os.path.join(ROOT, "tests", "golden", "bam_cases")


def _bam(level, block=4000):
    from fslr_b200 import synth_bam as sb
    refs, recs, _ = sb.make_alignments(300, seed=5, p_unmapped=0.0)
    return sb.bam_bytes(refs, [sb.encode_record(*r) for r in recs], block=block, level=level)


def _msg(kind, raw, k):
    return re.escape("%s mismatch in BGZF block %d (file offset %d)" % (kind, k, bc.block_offsets(raw)[k][0]))


def _readers(raw, tmp_path):
    from fslr_b200 import cluster, mapping_info as mi
    path = tmp_path / "t.bam"
    path.write_bytes(raw)
    return {"inflate_bgzf": lambda: mi.inflate_bgzf(raw),
            "inflate_bgzf_threads": lambda: mi.inflate_bgzf(raw, threads=4),
            "inflate_bgzf_path": lambda: mi.inflate_bgzf(str(path)),
            "bgzf_header_prefix": lambda: mi.bgzf_header_prefix(raw),
            "get_chromosome_lengths": lambda: cluster.get_chromosome_lengths(str(path))}


@pytest.mark.parametrize("kind,level", [("payload", 0), ("crc", 1), ("crc", 6), ("isize", 1)])
def test_corrupt_header_block_is_refused_by_every_reader(tmp_path, kind, level):
    """Block 0 holds the BAM header, so all three readers inflate it."""
    raw = _bam(level)
    if kind == "payload":
        bad, want = bc.flip_payload(raw, 0, at=300), _msg("CRC32", raw, 0)       # a stored block: still inflates cleanly
    elif kind == "crc":
        bad, want = bc.flip_crc(raw, 0), _msg("CRC32", raw, 0)
    else:
        bad, want = bc.set_isize(raw, 0, 3999), _msg("ISIZE", raw, 0)
    for name, read in _readers(bad, tmp_path).items():
        with pytest.raises(ValueError, match=want):
            read()


def test_record_block_issue_case(tmp_path):
    """117 stored blocks; one payload bit flipped in block 3 inflates to a stream that differs in one byte."""
    from fslr_b200 import mapping_info as mi
    raw = _bam(0)
    assert len(bc.block_offsets(raw)) == 117
    b = bytearray(raw)
    b[bc.block_offsets(raw)[3][0] + 18 + 200] ^= 0x04
    for threads in (1, 8):
        with pytest.raises(ValueError, match=_msg("CRC32", raw, 3)):
            mi.inflate_bgzf(bytes(b), threads=threads)
    mi.bgzf_header_prefix(bytes(b))                                               # the header blocks are intact
    bad = bc.flip_crc(bc.flip_crc(raw, 9), 4)                                     # two bad blocks: the first is named
    with pytest.raises(ValueError, match=_msg("CRC32", raw, 4)):
        mi.inflate_bgzf(bad, threads=8)
    eof = bytearray(raw)
    eof[-8] = 1                                                                   # the EOF marker's CRC32 must be 0
    with pytest.raises(ValueError, match=_msg("CRC32", raw, 116)):
        mi.inflate_bgzf(bytes(eof))
    with pytest.raises(ValueError, match=_msg("ISIZE", raw, 116)):
        mi.inflate_bgzf(bc.set_isize(raw, 116, 1))


@pytest.mark.parametrize("name", sorted(json.load(open(os.path.join(CASES_DIR, "cases.json")))))
def test_valid_bams_read_as_before(name):
    """The stored fixtures: the stream gzip inflates, the header parsed from it, the reference lengths."""
    from fslr_b200 import cluster, mapping_info as mi
    path = os.path.join(CASES_DIR, name + ".bam")
    raw = open(path, "rb").read()
    want = np.frombuffer(gzip.decompress(raw), dtype=np.uint8)
    got = mi.inflate_bgzf(raw)
    assert np.array_equal(got, want) and np.array_equal(mi.inflate_bgzf(path, threads=1), want)
    refs, first = mi.parse_bam_header(want)
    assert mi.bgzf_header_prefix(raw) == (refs, first)
    assert cluster.get_chromosome_lengths(path) == dict(refs)
