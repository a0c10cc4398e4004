"""compare_groups without a GPU: group-file parsing, the argument errors raised before any device call,
and the TSV / NPZ readers agreeing on sample and event names and order."""
import argparse
import os

import numpy as np
import pytest


def _args(argv):
    from splicedice_b200 import compare_groups
    p = argparse.ArgumentParser()
    compare_groups.add_parser(p)
    return p.parse_args(argv)


def test_group_files_manifest_blank_lines_and_carriage_returns(tmp_path):
    from splicedice_b200 import compare_groups
    f = tmp_path / "g.txt"
    f.write_bytes(b"s0\tinput/s0.junc.bed\tmeta0\tcond0\r\n\n   \r\ns2\r\ns 4\n\ns6\tx")
    assert compare_groups.read_samples(str(f)) == ["s0", "s2", "s 4", "s6"]
    (tmp_path / "empty.txt").write_text("\n\n")
    assert compare_groups.read_samples(str(tmp_path / "empty.txt")) == []


@pytest.mark.parametrize("g1,g2,needle", [
    (["s0", "s9"], ["s1"], "'s9' is not a column"),
    (["s0", "s1"], ["s2", "s1"], "'s1' is in both groups"),
    (["s0", "s2", "s0"], ["s1"], "'s0' is listed twice in group 1"),
    (["s0"], ["s1", "s3", "s1"], "'s1' is listed twice in group 2"),
    ([], ["s1"], "group 1 lists no samples"),
    (["s0"], [], "group 2 lists no samples"),
])
def test_group_errors_name_the_sample(g1, g2, needle):
    from splicedice_b200 import compare_groups
    samples = [f"s{i}" for i in range(8)]
    with pytest.raises(ValueError) as e:
        compare_groups.group_columns(samples, g1, g2)
    assert needle in str(e.value)


def test_group_columns_follow_the_header_order():
    from splicedice_b200 import compare_groups
    c1, c2 = compare_groups.group_columns(["a", "b", "c", "d", "e"], ["d", "a"], ["c"])
    assert c1.tolist() == [3, 0] and c2.tolist() == [2]


def test_cli_errors_come_before_any_device_call(golden_dir, tmp_path):
    """The checks run on the host: they raise ValueError here, where a device call would fail otherwise."""
    from splicedice_b200 import compare_groups
    tsv = os.path.join(golden_dir, "cli_8x", "expected", "ref_allPS.tsv")
    cases = [("s0\nnope\n", "s1\n", "'nope'"), ("s0\ns1\n", "s1\n", "'s1'"), ("\n", "s1\n", "group 1")]
    for g1, g2, needle in cases:
        (tmp_path / "a.txt").write_text(g1)
        (tmp_path / "b.txt").write_text(g2)
        out = tmp_path / "cmp.tsv"
        with pytest.raises(ValueError) as e:
            compare_groups.run_with(_args(["-p", tsv, "-g1", str(tmp_path / "a.txt"), "-g2", str(tmp_path / "b.txt"),
                                           "-o", str(out)]))
        assert needle in str(e.value)
        assert not out.exists()


def test_npz_and_tsv_readers_agree(golden_dir, tmp_path):
    from splicedice_b200 import compare_groups
    tsv = os.path.join(golden_dir, "cli_8x_lownan", "expected", "ref_allPS.tsv")
    samples, events, ps = compare_groups.read_ps(tsv)
    lines = open(tsv).read().splitlines()
    assert samples == lines[0].split("\t")[1:] and events == [l.split("\t")[0] for l in lines[1:]]
    assert ps.dtype == np.float64 and ps.shape == (len(events), len(samples)) and np.isnan(ps).any()
    npz = str(tmp_path / "x_allPS.npz")
    # the layout quant --npz writes (SPLICEDICE.writeNpz)
    np.savez(npz, cols=np.array(samples), rows=np.array(events), data=ps.astype(np.float32))
    s2, e2, ps2 = compare_groups.read_ps(npz)
    assert s2 == samples and e2 == events
    assert ps2.dtype == np.float32
    np.testing.assert_array_equal(ps2, ps.astype(np.float32))


def test_registered_as_a_command():
    from splicedice_b200 import __main__ as cli
    from splicedice_b200 import compare_groups
    assert cli.COMMANDS["compare_groups"] is compare_groups
    a = _args(["-p", "x_allPS.tsv", "-g1", "a.txt", "-g2", "b.txt"])
    assert (a.ps, a.group1, a.group2, a.output, a.device) == ("x_allPS.tsv", "a.txt", "b.txt", "compare_groups.tsv", 0)
