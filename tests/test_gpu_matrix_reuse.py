"""A destroyed matrix is parked and handed to the next hx_create of the same shape; nothing that one use of it set up
may carry over to the next use."""
import os
import subprocess
import sys
import textwrap

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
pytestmark = pytest.mark.gpu

# The verdict of the sortedness pre-pass is read back by ingest_totals() only after an ingestion launch ran it.  A
# reused handle must not remember that its previous user ran one: the zeroed flag word would read as "not sorted",
# the process would note that it has met unsorted reads, and every later short-read launch would queue the
# counting-sort fallback (k_flag_not + 11 k_l2_* launches instead of one k1_pairs_red).
_SCRIPT = textwrap.dedent("""
    import numpy as np
    from gretel_b200 import synth
    from gretel_b200.hansel import Hansel, REF_SYMBOLS, REF_UNSYMBOLS
    N, R, mk = 2000, 100_000, 12
    rank, off, codes = synth.random_packed(np.random.default_rng(7), N, R, mk, sort=True)

    def ingest():
        h = Hansel.init_matrix(REF_SYMBOLS, REF_UNSYMBOLS, N, band_w=mk - 1)
        totals = h.ingest_packed(rank, off, codes)
        n = h.launch_count()
        h.close()
        return totals, n

    first = ingest()
    h = Hansel.init_matrix(REF_SYMBOLS, REF_UNSYMBOLS, N, band_w=mk - 1)   # the parked handle of the first use
    h.ingest_totals()                                                        # nothing ingested
    h.close()
    third = ingest()
    print("launches", first[1], third[1])
    assert third == first, (first, third)
""")


def test_reused_matrix_does_not_inherit_the_prepass_verdict():
    env = dict(os.environ)
    env.pop("HX_NO_MATRIX_CACHE", None)          # the matrix cache must be on
    env.pop("HX_HOST_PIPELINE", None)
    env["PYTHONPATH"] = ROOT + os.pathsep + env.get("PYTHONPATH", "")
    # a fresh process: whether unsorted reads have been met is remembered for the whole process
    out = subprocess.run([sys.executable, "-c", _SCRIPT], capture_output=True, text=True, timeout=280, cwd=ROOT,
                         env=env)
    assert out.returncode == 0, out.stdout[-2000:] + out.stderr[-2000:]
