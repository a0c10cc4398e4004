"""compare_conditions without a GPU: groups-file parsing, group order, the argument errors raised before
any device call, and registration as a command."""
import argparse
import os

import pytest


def _args(argv):
    from splicedice_b200 import compare_conditions
    p = argparse.ArgumentParser()
    compare_conditions.add_parser(p)
    return p.parse_args(argv)


def test_manifest_groups_by_its_last_field(golden_dir):
    from splicedice_b200 import compare_conditions
    path = os.path.join(golden_dir, "cli_8x", "input", "manifest.txt")
    names, members = compare_conditions.read_groups(path)
    assert names == ["cond0", "cond1"]
    assert members == [["s0", "s2", "s4", "s6"], ["s1", "s3", "s5", "s7"]]


def test_two_column_file_blank_lines_crlf_and_first_appearance_order(tmp_path):
    from splicedice_b200 import compare_conditions
    f = tmp_path / "g.txt"
    f.write_bytes(b"s3\tliver\r\n\n   \r\ns0\tbrain\r\ns 1\tliver\ns9\tinput/s9.bed\tm\tkidney\n\ns2\tbrain")
    names, members = compare_conditions.read_groups(str(f))
    assert names == ["liver", "brain", "kidney"]
    assert members == [["s3", "s 1"], ["s0", "s2"], ["s9"]]


@pytest.mark.parametrize("text,needle", [("s0\tA\ns1\n", "g.txt:2"), ("s0\tA\n\ns1\t\n", "g.txt:3"),
                                         ("s0\tA\ns1\t \n", "g.txt:2")])
def test_malformed_lines_name_the_file_and_line(tmp_path, text, needle):
    from splicedice_b200 import compare_conditions
    f = tmp_path / "g.txt"
    f.write_text(text)
    with pytest.raises(ValueError) as e:
        compare_conditions.read_groups(str(f))
    assert needle in str(e.value)


@pytest.mark.parametrize("names,members,needle", [
    (["A", "B"], [["s0", "s1"], ["s2", "s1"]], "'s1' is listed twice"),
    (["A", "B"], [["s0", "s0"], ["s2"]], "'s0' is listed twice"),
    (["A", "B"], [["s0"], ["s9"]], "'s9' is not a column of the PS table"),
    (["A"], [["s0", "s1"]], "at least two"),
    ([], [], "at least two"),
])
def test_group_errors(names, members, needle):
    from splicedice_b200 import compare_conditions
    with pytest.raises(ValueError) as e:
        compare_conditions.group_columns([f"s{i}" for i in range(8)], names, members)
    assert needle in str(e.value)


def test_group_columns_follow_the_header():
    from splicedice_b200 import compare_conditions
    cols = compare_conditions.group_columns(["a", "b", "c", "d", "e"], ["x", "y", "z"], [["d", "a"], ["c"], ["e"]])
    assert [c.tolist() for c in cols] == [[3, 0], [2], [4]]


def test_header_names_the_groups_in_order():
    from splicedice_b200 import compare_conditions
    assert compare_conditions.header(["liver", "brain"]) == "event\tH\tpvalue\tcorrected\tmean_liver\tmean_brain\n"


def test_cli_errors_come_before_any_device_call(golden_dir, tmp_path):
    """The checks run on the host: they raise ValueError here, where a device call would fail otherwise."""
    from splicedice_b200 import compare_conditions
    tsv = os.path.join(golden_dir, "cli_8x", "expected", "ref_allPS.tsv")
    cases = [("s0\tA\ns1\n", "g.txt:2"), ("s0\tA\ns1\tB\ns0\tB\n", "'s0'"), ("s0\tA\nnope\tB\n", "'nope'"),
             ("s0\tA\ns1\tA\n", "at least two"), ("\n", "at least two")]
    for text, needle in cases:
        (tmp_path / "g.txt").write_text(text)
        out = tmp_path / "cmp.tsv"
        with pytest.raises(ValueError) as e:
            compare_conditions.run_with(_args(["-p", tsv, "-g", str(tmp_path / "g.txt"), "-o", str(out)]))
        assert needle in str(e.value)
        assert not out.exists()


def test_registered_as_a_command():
    from splicedice_b200 import __main__ as cli
    from splicedice_b200 import compare_conditions
    assert cli.COMMANDS["compare_conditions"] is compare_conditions
    a = _args(["-p", "x_allPS.npz", "-g", "manifest.txt"])
    assert (a.ps, a.groups, a.output, a.device) == ("x_allPS.npz", "manifest.txt", "compare_conditions.tsv", 0)
    a = _args(["--ps", "x_allPS.tsv", "--groups", "g.txt", "--output", "o.tsv", "--device", "1"])
    assert (a.ps, a.groups, a.output, a.device) == ("x_allPS.tsv", "g.txt", "o.tsv", 1)
