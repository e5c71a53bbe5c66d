"""The device BAM route (fslrc_bam_open_bgzf) refuses a BGZF block whose inflated bytes do not match the CRC32 of its
trailer (k_bgzf_crc), as htslib does and as the oracle's gzip-based reader does; the host-inflate route names the same
block; the context stays usable; valid files give the bytes they gave before."""
import gzip
import re

import pytest

from tests import bgzf_cases as bc

pytestmark = pytest.mark.gpu


def _valid(level, block=4000):
    from fslr_b200 import synth_bam as sb
    refs, recs, primers = sb.make_alignments(300, seed=5, p_unmapped=0.0)
    return sb.bam_bytes(refs, [sb.encode_record(*r) for r in recs], block=block, level=level), primers


def _eof_crc(raw):
    b = bytearray(raw)
    b[-8] = 0x5a                                                                  # the EOF marker (ISIZE 0) with CRC32 != 0
    return bytes(b)


# name: (level, corruption, index of the first bad block); the BAM header sits in block 0, which is never touched here
CASES = {
    "stored_payload_byte": (0, lambda r: bc.flip_payload(r, 3, at=200), 3),      # inflates cleanly, one byte differs
    "level1_crc_field": (1, lambda r: bc.flip_crc(r, 5), 5),
    "level6_crc_field": (6, lambda r: bc.flip_crc(r, 7), 7),
    "eof_block_crc": (1, _eof_crc, -1),
    "two_bad_blocks": (0, lambda r: bc.flip_payload(bc.flip_crc(r, 9), 2, at=50), 2),   # the first is named
}


def _msg(raw, k):
    k = k % len(bc.block_offsets(raw))
    return re.escape("CRC32 mismatch in BGZF block %d (file offset %d)" % (k, bc.block_offsets(raw)[k][0]))


@pytest.mark.parametrize("case", sorted(CASES))
def test_corrupt_block_is_refused(tmp_path, case):
    from fslr_b200 import _native, mapping_info as mi
    from oracle import mapping_info_oracle as mo
    level, corrupt, k = CASES[case]
    good, primers = _valid(level)
    bad = corrupt(good)
    assert len(bad) == len(good) and bad != good
    path, ok = str(tmp_path / "bad.bam"), str(tmp_path / "ok.bam")
    open(path, "wb").write(bad)
    open(ok, "wb").write(good)
    want = _msg(good, k)
    with pytest.raises(_native.FslrError, match=want):
        mi.read_bam_table(path, None, primers)
    with pytest.raises(_native.FslrError, match=want):                           # the same bytes from memory
        mi.read_bam_table(bad, None, primers)
    with pytest.raises(ValueError, match=want):                                  # host-inflate route: the same block
        mi.read_bam_table(path, None, primers, device_inflate=False)
    with pytest.raises(gzip.BadGzipFile, match="CRC check failed"):             # the oracle (stub pysam reads through gzip)
        mo.mapping_rows(path, None, primers, "9.9")
    # the context that refused the file opens the next one
    expect = mo.mapping_tsv(mo.mapping_rows(ok, None, primers, "9.9")).encode()
    t = mi.read_bam_table(ok, None, primers)
    try:
        assert t.mappings_bed_bytes("9.9").tobytes() == expect
    finally:
        t.close()


def test_pipeline_writes_nothing_for_a_corrupt_bam(tmp_path):
    from fslr_b200 import _native, pipeline
    good, primers = _valid(0)
    bam = tmp_path / "s.bwa_dodi.bam"
    bam.write_bytes(bc.flip_payload(good, 3, at=200))
    csv = tmp_path / "primers.csv"
    csv.write_text("primer_name,primer_seq\n" + "".join("%s,%s\n" % kv for kv in primers.items()))
    base = str(tmp_path / "s")
    with pytest.raises(_native.FslrError, match=_msg(good, 3)):
        pipeline.main(["--bam", str(bam), "--primers-csv", str(csv), "--primers", ",".join(primers), "--out-base", base])
    assert not (tmp_path / "s.mappings.bed").exists()


def test_bench_size_bam(tmp_path):
    """About 5 000 blocks of 60 000 inflated bytes, so nearly every lane of k_bgzf_crc has a full 2048-byte segment: the
    device route gives the host-inflate route's bytes; a flipped byte in the last block before the EOF marker is refused."""
    from fslr_b200 import _native, mapping_info as mi
    raw, primers = bc.bench_bam(10)
    path = str(tmp_path / "big.bam")
    open(path, "wb").write(raw)
    a = mi.read_bam_table(path, None, primers, device_inflate=False)
    try:
        want = a.mappings_bed_bytes("9.9").tobytes()
    finally:
        a.close()
    b = mi.read_bam_table(path, None, primers)
    try:
        assert b.mappings_bed_bytes("9.9").tobytes() == want
    finally:
        b.close()
    k = len(bc.block_offsets(raw)) - 2
    with pytest.raises(_native.FslrError, match=_msg(raw, k)):
        mi.read_bam_table(bc.flip_crc(raw, k), None, primers)
