"""``python -m splicedice_b200 <command>``: the hot-path commands of the splicedice CLI
(quant, counts_to_ps, pairwise, ir_table) with the reference's flags, compare_groups (a rank-sum
test per event between two sample groups), compare_conditions (a Kruskal-Wallis test per event
across any number of sample groups), compare_paired (a signed-rank test per event between matched
sample pairs) and compare_repeated (a Friedman test per event across conditions measured on the same
subjects), running on a B200.
The remaining reference commands (BAM readers, the other downstream statistics) are out of scope."""
import argparse

from . import (compare_conditions, compare_groups, compare_paired, compare_repeated, counts_to_ps, ir_table,
               pairwise_fisher, quant)

COMMANDS = {
    "quant": quant,
    "counts_to_ps": counts_to_ps,
    "pairwise": pairwise_fisher,
    "ir_table": ir_table,
    "compare_groups": compare_groups,
    "compare_conditions": compare_conditions,
    "compare_paired": compare_paired,
    "compare_repeated": compare_repeated,
}


def main(argv=None):
    parser = argparse.ArgumentParser(prog="splicedice_b200", description=__doc__)
    sub = parser.add_subparsers(dest="command")
    for name, module in COMMANDS.items():
        cmd = sub.add_parser(name)
        module.add_parser(cmd)
        cmd.set_defaults(main=module.run_with)
    args = parser.parse_args(argv)
    if hasattr(args, "main"):
        args.main(args)
    else:
        parser.print_usage()


if __name__ == "__main__":
    main()
