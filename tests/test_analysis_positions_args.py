"""CPU: argument handling and the positions file of `analysis --positions FILE --batches K` (host/analysis.cpp).  Every
case here is rejected before a device is needed."""
import os
import subprocess

import pytest

from takzero_b200 import build as tz_build


def run(args):
    tz_build.build()
    exe = os.path.join(os.path.dirname(tz_build.LIB), "bin", "analysis")
    return subprocess.run([exe, *args], capture_output=True, text=True, timeout=120)


@pytest.mark.parametrize("args", [
    ["--positions", "{f}"],                                  # no --batches
    ["--batches", "2"],                                      # no --positions
    ["--positions", "{f}", "--batches", "0"],
    ["--positions", "{f}", "--batches", "2", "--example"],
    ["--positions", "{f}", "--batches", "2", "--tps", "x4/x4/x4/x4 1 1"],
    ["--positions", "{f}", "--batches", "2", "--board", "9"],
    ["--positions", "{f}", "--batches", "2", "--batch-size", "0"],
])
def test_bad_arguments_are_rejected(tmp_path, args):
    f = tmp_path / "positions.txt"
    f.write_text("x4/x4/x4/x4 1 1\n")
    out = run(["--board", "4"] + [a.format(f=f) for a in args])
    assert out.returncode == 2, out.stderr
    assert out.stdout == ""


@pytest.mark.parametrize("text,line", [
    ("x4/x4/x4/x4 1 1\nx4/x4/x4/x5 1 1\n", 2),       # a row of five squares on 4x4
    ("x4/x4/x4/x4 1 1\n\n  \nnot tps\n", 4),           # blank lines count, and are skipped
    ("x4/x4/x4/x4 1 1\nx4/x4/x4 1 1\n", 2),            # three rows
])
def test_a_bad_tps_line_is_rejected_with_its_number(tmp_path, text, line):
    f = tmp_path / "positions.txt"
    f.write_text(text)
    out = run(["--board", "4", "--positions", str(f), "--batches", "1"])
    assert out.returncode == 2
    assert f"line {line} is not valid TPS" in out.stderr
    assert out.stdout == ""


def test_a_missing_or_empty_file_is_rejected(tmp_path):
    out = run(["--board", "4", "--positions", str(tmp_path / "missing.txt"), "--batches", "1"])
    assert out.returncode == 2 and "cannot read" in out.stderr
    f = tmp_path / "empty.txt"
    f.write_text("\n\n")
    out = run(["--board", "4", "--positions", str(f), "--batches", "1"])
    assert out.returncode == 2 and "no position" in out.stderr
