"""The SNP table of the command line goes to the sys.stdout of the call, wherever sys.stdout pointed when
gretel_b200.cmd was first imported (a caller or test harness that swaps sys.stdout later still gets it)."""
import io
import sys

from gretel_b200 import cmd


class _Counts:
    def get_counts_at(self, i):
        return {"A": 1, "total": 1}


def test_snp_table_writes_to_current_stdout(monkeypatch):
    buf = io.StringIO()
    monkeypatch.setattr(sys, "stdout", buf)
    cmd.snp_table(_Counts(), {"N": 2, "snp_rev": [3, 7]})
    lines = buf.getvalue().split("\n")
    assert lines[0].split("\t") == ["i", "pos", "gap", "A", "C", "G", "T", "N", "-", "_", "tot"]
    assert lines[1:4] == ["0\t0\t0\t1\t0\t0\t0\t0\t0\t0\t1", "1\t3\t3\t1\t0\t0\t0\t0\t0\t0\t1",
                          "2\t7\t4\t1\t0\t0\t0\t0\t0\t0\t1"]
