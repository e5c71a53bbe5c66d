"""TEST INFRASTRUCTURE ONLY — the edges of the similarity graph from the CPU oracle (oracle/fslr_oracle.c).

The oracle's literal loop adds an edge where cluster.py:220-221 does, but does not report it.  Rather than keep a second
copy of that loop, this module compiles the unmodified oracle source with one statement inserted after the edge count
(`st->edges++; edges++;`): it records (query_key, other read, jaccard), in the order the reference adds them.  The
result is a separate library under tests/_build; everything else of the oracle is the same code, and
tests/test_oracle_edges.py checks that its ids and counters equal those of oracle.oracle_cluster.
"""
import ctypes as C
import os
import subprocess

import numpy as np

from oracle import oracle as orc

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SRC = os.path.join(ROOT, "oracle", "fslr_oracle.c")
BUILD = os.path.join(ROOT, "tests", "_build")
ANCHOR = "st->edges++; edges++;"

PREFIX = r"""
#include <stdint.h>
#include <stdlib.h>
static int32_t *g_r1, *g_r2; static double *g_j; static int64_t g_n, g_cap;
static void record_edge(int32_t a, int32_t b, double j) {
    if (g_n == g_cap) {
        g_cap = g_cap ? 2 * g_cap : 1024;
        g_r1 = (int32_t *)realloc(g_r1, g_cap * 4); g_r2 = (int32_t *)realloc(g_r2, g_cap * 4);
        g_j = (double *)realloc(g_j, g_cap * 8);
    }
    g_r1[g_n] = a; g_r2[g_n] = b; g_j[g_n] = j; g_n++;
}
void oracle_edges_reset(void) { g_n = 0; }
int64_t oracle_edges_get(const int32_t **r1, const int32_t **r2, const double **j) { *r1 = g_r1; *r2 = g_r2; *j = g_j; return g_n; }
"""

_lib = None


def _load():
    global _lib
    if _lib is None:
        os.makedirs(BUILD, exist_ok=True)
        so = os.path.join(BUILD, "liboracle_edges.so")
        if not os.path.exists(so) or os.path.getmtime(so) < max(os.path.getmtime(SRC), os.path.getmtime(__file__)):
            text = open(SRC).read()
            if text.count(ANCHOR) != 1:
                raise RuntimeError("oracle/fslr_oracle.c: the edge statement %r is not there exactly once" % ANCHOR)
            src = os.path.join(BUILD, "oracle_edges.c")
            with open(src, "w") as f:
                f.write(PREFIX + text.replace(ANCHOR, ANCHOR + " record_edge(qk, o->rid, j);"))
            # the oracle's own flags (oracle/Makefile): no FMA contraction, so the doubles are the reference's
            subprocess.check_call(["gcc", "-O2", "-fPIC", "-shared", "-Wall", "-Wno-unused-variable", "-ffp-contract=off",
                                   "-o", so, src])
        lib = C.CDLL(so)
        lib.fslr_oracle_cluster.restype = C.c_int
        lib.fslr_oracle_cluster.argtypes = [C.POINTER(orc._In), C.c_void_p, C.c_void_p, C.POINTER(orc._Stats)]
        lib.oracle_edges_reset.restype = None
        lib.oracle_edges_get.restype = C.c_int64
        lib.oracle_edges_get.argtypes = [C.POINTER(C.POINTER(C.c_int32)), C.POINTER(C.POINTER(C.c_int32)),
                                         C.POINTER(C.POINTER(C.c_double))]
        _lib = lib
    return _lib


def oracle_cluster_edges(table, params, order=None):
    """oracle.oracle_cluster plus the edges: returns (cluster, n_reads, stats, (read1 int32, read2 int32, jaccard
    float64)), the edges as (query_key, other read, jaccard similarity) in read ids, in the order cluster.py adds them."""
    lib = _load()
    keep = []

    def p(a, dt):
        a = np.ascontiguousarray(a, dtype=dt)
        keep.append(a)
        return a.ctypes.data

    cut = np.asarray(params.jaccard_cutoffs, dtype=np.float64)
    masked = params.chrom_masked if params.chrom_masked is not None else np.zeros(table.n_chrom, np.uint8)
    a = orc._In(table.n_rows, table.n_reads, p(table.read_id, np.int32), p(table.chrom, np.int32),
                p(table.rstart, np.int32), p(table.rend, np.int32), p(table.aln_size, np.int32),
                p(table.qstart, np.int32), p(table.qend, np.int32), p(table.n_alignments, np.int32),
                table.n_chrom, p(table.chrom_len, np.int64), p(masked, np.uint8),
                int(params.mask_subtelomere), int(params.subtel),
                p(order, np.int64) if order is not None else None,
                params.overlap, params.qlen_diff, params.n_alignment_diff,
                p(cut, np.float64), len(cut), int(params.edge_threshold))
    out_c = np.empty(table.n_reads, dtype=np.int32)
    out_n = np.empty(table.n_reads, dtype=np.int32)
    st = orc._Stats()
    lib.oracle_edges_reset()
    rc = lib.fslr_oracle_cluster(C.byref(a), out_c.ctypes.data, out_n.ctypes.data, C.byref(st))
    if rc != 0:
        raise ZeroDivisionError("oracle: invalid table (code %d): zero aln_size / qlen2 / n_alignments" % rc)
    r1, r2, j = C.POINTER(C.c_int32)(), C.POINTER(C.c_int32)(), C.POINTER(C.c_double)()
    n = lib.oracle_edges_get(C.byref(r1), C.byref(r2), C.byref(j))
    edges = (np.ctypeslib.as_array(r1, (n,)).copy() if n else np.zeros(0, np.int32),
             np.ctypeslib.as_array(r2, (n,)).copy() if n else np.zeros(0, np.int32),
             np.ctypeslib.as_array(j, (n,)).copy() if n else np.zeros(0, np.float64))
    stats = {k: int(getattr(st, k)) for k, _ in orc._Stats._fields_}
    return out_c, out_n, stats, edges
