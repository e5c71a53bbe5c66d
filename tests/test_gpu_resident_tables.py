"""Device-resident tables (engine.ResidentTable: tsv.ParsedBed, mapping_info.BamTable).  The library context holds one table
of each kind, so a handle whose table a later open replaced must refuse every call: its device columns are gone, and the
context's entry points now describe the newer table."""
import json
import os

import pytest

pytestmark = pytest.mark.gpu

CASES_DIR = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden", "bam_cases")
CASES = json.load(open(os.path.join(CASES_DIR, "cases.json")))


def test_a_stale_bam_table_refuses_qnames():
    """qnames() of a replaced BamTable raises like its other methods.  The newer table has more reads than the stale one:
    reading its names into arrays sized for the stale table would write past them."""
    from fslr_b200 import mapping_info as mi
    old = mi.read_bam_table(os.path.join(CASES_DIR, "one_read.bam"), None, CASES["one_read"]["primers"])
    new = mi.read_bam_table(os.path.join(CASES_DIR, "basic.bam"), None, CASES["basic"]["primers"])
    try:
        assert new.n_reads > old.n_reads
        with pytest.raises(RuntimeError, match="stale BamTable"):
            old.qnames()
        old.close()                                                      # must not free the newer table
        names = new.qnames()
        assert len(names) == new.n_reads and len(set(names)) == new.n_reads
    finally:
        new.close()
    closed = mi.read_bam_table(os.path.join(CASES_DIR, "one_read.bam"), None, CASES["one_read"]["primers"])
    closed.close()
    with pytest.raises(RuntimeError, match="BamTable is closed"):
        closed.qnames()
