"""`python -m ractip_b200`: the reference's command line (src/ractip.ggo) over the many-pair front end."""
import argparse
import sys

from .frontend import constraint_line, format_result, input_pairs, predict
from .ip import default_ip_opts
from .stage import ProbabilityStage, RpError, default_opts

RP_ERR_ARG = 1


def main(argv=None) -> int:
    ap = argparse.ArgumentParser(prog="python -m ractip_b200", description=__doc__)
    ap.add_argument("fasta", nargs="+", help="one FASTA file with two records, or two files")
    ap.add_argument("-a", "--alpha", type=float, default=0.7)
    ap.add_argument("-b", "--beta", type=float, default=0.0)
    ap.add_argument("-t", "--fold-th", type=float, default=0.5)
    ap.add_argument("-u", "--hybridize-th", type=float, default=0.1)
    ap.add_argument("-s", "--acc-th", type=float, default=0.003)
    ap.add_argument("--acc-max", action="store_true")
    ap.add_argument("--acc-max-ss", action="store_true")
    ap.add_argument("--acc-num", type=int, default=1)
    ap.add_argument("--max-w", type=int, default=15)
    ap.add_argument("--min-w", type=int, default=5)
    ap.add_argument("--zscore", type=int, default=0, choices=[0, 1, 2, 12])
    ap.add_argument("--num-shuffling", type=int, default=1000)
    ap.add_argument("--seed", type=int, default=1)
    ap.add_argument("--allow-isolated", action="store_true")
    ap.add_argument("-e", "--show-energy", action="store_true")
    ap.add_argument("-c", "--use-constraint", action="store_true",
                    help="constrain the probabilities by the records' structure lines (.x()[]; ? and space as .)")
    ap.add_argument("-P", "--param-file", default=None)
    ap.add_argument("--no-pk", action="store_true")
    ap.add_argument("--duplex", action="store_true")
    ap.add_argument("--no-bl", action="store_true")
    ap.add_argument("--all-pairs", action="store_true", help="every record of the first file against every record of the second")
    ap.add_argument("--device", type=int, default=0)
    args = ap.parse_args(argv)
    if len(args.fasta) > 2:
        ap.error("at most two FASTA files")
    try:
        pairs = input_pairs(args.fasta[0], args.fasta[1] if len(args.fasta) > 1 else None, args.all_pairs)
        if args.use_constraint:
            for a, b in pairs:
                constraint_line(a), constraint_line(b)
    except ValueError as e:   # the reference prints the message and exits 1 (src/ractip.cpp:1684-1697)
        print(e)
        return 1
    # option mapping of RactIP::parse_options (src/ractip.cpp:1474-1498)
    opts = default_opts(max_w=max(1, args.max_w), min_w=args.min_w, th_ss=args.fold_th, th_hy=args.hybridize_th,
                        th_ac=args.acc_th, use_pf_duplex=int(args.duplex))
    ipo = default_ip_opts(alpha=args.alpha, beta=args.beta, th_ss=args.fold_th, th_hy=args.hybridize_th,
                          th_ac=args.acc_th, max_w=args.max_w, min_w=args.min_w, acc_max=int(args.acc_max),
                          acc_max_ss=int(args.acc_max_ss), acc_num=args.acc_num, in_pk=int(not args.no_pk),
                          stacking=int(not args.allow_isolated))
    stage = ProbabilityStage(device=args.device, use_bl=not args.no_bl, param_file=args.param_file)
    try:
        for r in predict(stage, pairs, opts, ipo, args.show_energy, args.zscore, args.num_shuffling, args.seed,
                         use_constraint=args.use_constraint):
            print(format_result(r, args.show_energy))
    except RpError as e:
        if not (args.use_constraint and e.code == RP_ERR_ARG):
            raise
        print(e)   # a malformed structure line is an input error like the others
        return 1
    finally:
        stage.close()
    return 0


if __name__ == "__main__":
    sys.exit(main())
