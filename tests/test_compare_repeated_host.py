"""compare_repeated without a GPU: blocks-file parsing and every refusal, the argument errors raised before
any device call (in the CLI, in sd_friedman_rows and in ops.friedman_rows), and registration as a command."""
import argparse
import os

import numpy as np
import pytest


def _args(argv):
    from splicedice_b200 import compare_repeated
    p = argparse.ArgumentParser()
    compare_repeated.add_parser(p)
    return p.parse_args(argv)


def test_blocks_file_blank_lines_crlf_and_skipped_subjects(tmp_path):
    from splicedice_b200 import compare_repeated
    f = tmp_path / "blocks.txt"
    f.write_bytes(b"\n  \r\nbase\t4 weeks\t12 weeks\r\ns0\ts1\ts2\r\n\n   \r\ns 3\t\ts5\ns6\ts7\ts8\n\t\t\ns12\t\t\ns9\ts10\ts11")
    names, subjects, skipped = compare_repeated.read_blocks(str(f))
    assert names == ["base", "4 weeks", "12 weeks"]
    assert subjects == [["s0", "s1", "s2"], ["s6", "s7", "s8"], ["s9", "s10", "s11"]]
    assert skipped == [["s 3", "", "s5"], ["s12", "", ""]]


@pytest.mark.parametrize("text,needle", [
    ("A\tB\tC\ns0\ts1\n", "blocks.txt:2: expected 3"),
    ("A\tB\tC\ns0\ts1\ts2\n\ns3\ts4\ts5\ts6\n", "blocks.txt:4: expected 3"),
    ("\nA\tB\tC\n\ns0 s1 s2\n", "blocks.txt:4: expected 3"),
    ("A\tB\n", "blocks.txt:1: the header names 2 condition(s)"),
    ("\n\nA\n", "blocks.txt:3: the header names 1 condition(s)"),
    ("A\t\tC\ns0\ts1\ts2\n", "blocks.txt:1: empty condition name"),
    ("A\tB\t \ns0\ts1\ts2\n", "blocks.txt:1: empty condition name"),
    ("A\tB\tA\ns0\ts1\ts2\n", "blocks.txt:1: a condition is named twice"),
    ("A\tB\tC\n", "no subject"),
    ("A\tB\tC\ns0\t\ts2\n\n", "no subject"),
    ("\n \n", "no header"),
])
def test_malformed_files_name_the_file_and_line(tmp_path, text, needle):
    from splicedice_b200 import compare_repeated
    f = tmp_path / "blocks.txt"
    f.write_text(text)
    with pytest.raises(ValueError) as e:
        compare_repeated.read_blocks(str(f))
    assert needle in str(e.value)


def test_two_conditions_point_to_compare_paired(tmp_path):
    from splicedice_b200 import compare_repeated
    f = tmp_path / "blocks.txt"
    f.write_text("before\tafter\ns0\ts1\n")
    with pytest.raises(ValueError, match="compare_paired"):
        compare_repeated.read_blocks(str(f))


@pytest.mark.parametrize("subjects,skipped,needle", [
    ([["s0", "s1", "s2"], ["s3", "s1", "s4"]], [], "'s1' is listed twice"),
    ([["s0", "s1", "s0"]], [], "'s0' is listed twice"),
    ([["s0", "s1", "s2"], ["s3", "s4", "s9"]], [], "'s9' is not a column of the PS table"),
    ([["s0", "s1", "s2"]], [["s3", "", "s1"]], "'s1' is listed twice"),          # a skipped line reuses a sample
    ([["s0", "s1", "s2"]], [["s3", "", "s3"]], "'s3' is listed twice"),
    ([["s0", "s1", "s2"]], [["", "s9", ""]], "'s9' is not a column of the PS table"),  # a typo on a skipped line
])
def test_block_errors(subjects, skipped, needle):
    from splicedice_b200 import compare_repeated
    with pytest.raises(ValueError) as e:
        compare_repeated.block_columns([f"s{i}" for i in range(8)], subjects, skipped)
    assert needle in str(e.value)


def test_skipped_lines_get_no_columns():
    from splicedice_b200 import compare_repeated
    cols = compare_repeated.block_columns([f"s{i}" for i in range(8)], [["s4", "s0", "s2"]], [["s1", "", "s3"]])
    assert cols.tolist() == [[4, 0, 2]]


def test_block_columns_follow_the_header():
    from splicedice_b200 import compare_repeated
    cols = compare_repeated.block_columns(["a", "b", "c", "d", "e", "f"], [["d", "a", "f"], ["c", "e", "b"]])
    assert cols.dtype == np.int32 and cols.tolist() == [[3, 0, 5], [2, 4, 1]]


def test_header_names_the_conditions_in_order():
    from splicedice_b200 import compare_repeated
    assert (compare_repeated.header(["base", "wk4", "wk12"])
            == "event\tn\tQ\tpvalue\tcorrected\tmean_base\tmean_wk4\tmean_wk12\n")


def test_cli_errors_come_before_any_device_call(golden_dir, tmp_path):
    """The checks run on the host: they raise ValueError here, where a device call would fail otherwise."""
    from splicedice_b200 import compare_repeated
    tsv = os.path.join(golden_dir, "cli_8x", "expected", "ref_allPS.tsv")
    cases = [("A\tB\tC\ns0\ts1\n", "blocks.txt:2"), ("A\tB\tC\ns0\ts1\ts2\ns3\ts4\ts0\n", "'s0'"),
             ("A\tB\tC\ns0\ts1\tnope\n", "'nope'"), ("A\tB\ns0\ts1\n", "compare_paired"),
             ("A\tB\tC\ns0\t\ts2\n", "no subject"), ("A\tB\tC\ns0\ts1\ts2\ns3\t\ts0\n", "'s0'"),
             ("A\tB\tC\ns0\ts1\ts2\nnope\ts3\t\n", "'nope'")]
    for text, needle in cases:
        (tmp_path / "blocks.txt").write_text(text)
        out = tmp_path / "cmp.tsv"
        with pytest.raises(ValueError) as e:
            compare_repeated.run_with(_args(["-p", tsv, "--blocks", str(tmp_path / "blocks.txt"), "-o", str(out)]))
        assert needle in str(e.value)
        assert not out.exists()


def test_registered_as_a_command():
    from splicedice_b200 import __main__ as cli
    from splicedice_b200 import compare_repeated
    assert cli.COMMANDS["compare_repeated"] is compare_repeated
    assert "compare_repeated" in cli.__doc__
    a = _args(["-p", "x_allPS.npz", "--blocks", "blocks.txt"])
    assert (a.ps, a.blocks, a.output, a.device) == ("x_allPS.npz", "blocks.txt", "compare_repeated.tsv", 0)
    a = _args(["--ps", "x_allPS.tsv", "--blocks", "b.txt", "--output", "o.tsv", "--device", "1"])
    assert (a.ps, a.blocks, a.output, a.device) == ("x_allPS.tsv", "b.txt", "o.tsv", 1)


@pytest.mark.parametrize("args,needle", [
    (dict(k=2), "n_conditions = 2 outside [3, 256]"),
    (dict(k=257), "n_conditions = 257 outside [3, 256]"),
    (dict(nb=0), "n_blocks = 0"),
    (dict(nb=5462, k=3), "n_blocks = 5462"),
    (dict(nb=64, k=257), "n_conditions = 257"),
    (dict(dtype=2), "dtype"),
    (dict(row_end=11), "row range"),
    (dict(row_begin=-1), "row range"),
    (dict(J=-1), "negative"),
    (dict(ld_mean=3), "ld too small"),
    (dict(ld_stats=1), "ld too small"),
    (dict(ld_ps=7), "ld too small"),
    (dict(null=True), "null pointer"),
])
def test_native_argument_errors_without_a_device(args, needle):
    """sd_friedman_rows checks its arguments before any CUDA call: SD_ERR_INVALID and the message."""
    from splicedice_b200 import native
    native.load()
    a = dict(J=10, S=8, ld_ps=8, dtype=native.SD_RANKSUM_F32, k=4, nb=2, row_begin=0, row_end=10, ld_mean=4,
             ld_stats=2, null=False)
    a.update(args)
    fake = None if a["null"] else 16                     # never dereferenced: every check fails first
    with pytest.raises(native.NativeCallError) as e:
        native.call("sd_friedman_rows", a["J"], a["S"], 16, a["ld_ps"], a["dtype"], a["k"], a["nb"], fake,
                    a["row_begin"], a["row_end"], 16, 16, a["ld_mean"], 16, a["ld_stats"], None)
    assert e.value.code == native.SD_ERR_INVALID and needle in str(e.value)


def test_empty_row_range_is_a_no_op_without_a_device():
    from splicedice_b200 import native
    native.load()
    native.call("sd_friedman_rows", 10, 8, None, 8, native.SD_RANKSUM_F64, 3, 2, None, 4, 4, None, None, 3, None, 2,
                None)


def test_ops_refuses_without_cuda():
    import torch
    from splicedice_b200 import native, ops
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    with pytest.raises(native.NativeLibraryError):
        ops.friedman_rows(torch.zeros((4, 8)), np.arange(6).reshape(2, 3))
