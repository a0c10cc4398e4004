"""compare_paired without a GPU: pairs-file parsing, the argument errors raised before any device call,
and registration as a command."""
import argparse
import os

import numpy as np
import pytest


def _args(argv):
    from splicedice_b200 import compare_paired
    p = argparse.ArgumentParser()
    compare_paired.add_parser(p)
    return p.parse_args(argv)


def test_pairs_file_blank_lines_crlf_and_extra_fields(tmp_path):
    from splicedice_b200 import compare_paired
    f = tmp_path / "pairs.txt"
    f.write_bytes(b"s0\ts1\r\n\n   \r\ns 3\ts2\tpatient 7\tnote\ns5\ts4\r\n\ns6\ts7")
    assert compare_paired.read_pairs(str(f)) == [("s0", "s1"), ("s 3", "s2"), ("s5", "s4"), ("s6", "s7")]


@pytest.mark.parametrize("text,needle", [("s0\ts1\ns2\n", "pairs.txt:2"), ("s0\ts1\n\ns2\t\n", "pairs.txt:3"),
                                         ("\ts1\n", "pairs.txt:1"), ("s0 s1\n", "pairs.txt:1")])
def test_malformed_lines_name_the_file_and_line(tmp_path, text, needle):
    from splicedice_b200 import compare_paired
    f = tmp_path / "pairs.txt"
    f.write_text(text)
    with pytest.raises(ValueError) as e:
        compare_paired.read_pairs(str(f))
    assert needle in str(e.value)


@pytest.mark.parametrize("pairs,needle", [
    ([("s0", "s1"), ("s2", "s1")], "'s1' is listed twice"),
    ([("s0", "s1"), ("s1", "s2")], "'s1' is listed twice"),
    ([("s0", "s0")], "'s0' is listed twice"),
    ([("s0", "s9")], "'s9' is not a column of the PS table"),
    ([], "no pairs"),
])
def test_pair_errors(pairs, needle):
    from splicedice_b200 import compare_paired
    with pytest.raises(ValueError) as e:
        compare_paired.pair_columns([f"s{i}" for i in range(8)], pairs)
    assert needle in str(e.value)


def test_pair_columns_follow_the_header():
    from splicedice_b200 import compare_paired
    c1, c2 = compare_paired.pair_columns(["a", "b", "c", "d", "e"], [("d", "a"), ("c", "e")])
    assert c1.dtype == c2.dtype == np.int32
    assert c1.tolist() == [3, 2] and c2.tolist() == [0, 4]


def test_cli_errors_come_before_any_device_call(golden_dir, tmp_path):
    """The checks run on the host: they raise ValueError here, where a device call would fail otherwise."""
    from splicedice_b200 import compare_paired
    tsv = os.path.join(golden_dir, "cli_8x", "expected", "ref_allPS.tsv")
    cases = [("s0\ts1\ns2\n", "pairs.txt:2"), ("s0\ts1\ns2\ts0\n", "'s0'"), ("s0\tnope\n", "'nope'"),
             ("\n", "no pairs")]
    for text, needle in cases:
        (tmp_path / "pairs.txt").write_text(text)
        out = tmp_path / "cmp.tsv"
        with pytest.raises(ValueError) as e:
            compare_paired.run_with(_args(["-p", tsv, "--pairs", str(tmp_path / "pairs.txt"), "-o", str(out)]))
        assert needle in str(e.value)
        assert not out.exists()


def test_registered_as_a_command():
    from splicedice_b200 import __main__ as cli
    from splicedice_b200 import compare_paired
    assert cli.COMMANDS["compare_paired"] is compare_paired
    a = _args(["-p", "x_allPS.npz", "--pairs", "pairs.txt"])
    assert (a.ps, a.pairs, a.output, a.device) == ("x_allPS.npz", "pairs.txt", "compare_paired.tsv", 0)
    a = _args(["--ps", "x_allPS.tsv", "--pairs", "p.txt", "--output", "o.tsv", "--device", "1"])
    assert (a.ps, a.pairs, a.output, a.device) == ("x_allPS.tsv", "p.txt", "o.tsv", 1)


def test_header():
    from splicedice_b200 import compare_paired
    assert compare_paired.HEADER == "event\tn\tmean1\tmean2\tdelta\tW\tpvalue\tcorrected\n"
