"""Command line of runCBO.py (reference: src/ArgumentParser.py): same flags, defaults and seeding."""
from argparse import ArgumentParser as _ArgParser

from numpy import random


class ArgumentParser:
    FLAGS = [
        ("--initial_num_obs_samples", 100, int, "initial number of observational samples"),
        ("--num_interventions", 10, int, "size of the initial interventional dataset"),
        ("--type_cost", 1, int, "cost per node: fix_equal = 1, fix_different = 2, fix_different_variable = 3, fix_equal_variable = 4"),
        ("--num_additional_observations", 20, int, "additional observations collected for every decision"),
        ("--num_trials", 40, int, "number of BO trials"),
        ("--name_index", 0, int, "index of the interventional dataset used"),
        ("--seed", 9, int, "seed of the experiment"),
        ("--exploration_set", "MIS", str, "exploration set"),
        ("--causal_prior", False, bool, "do not specify to leave it False (any non-empty value enables it, as in the reference)"),
        ("--experiment", "complete_graph", str, "experiment"),
        ("--task", "min", str, "min or max"),
    ]

    def __init__(self):
        self.parser = _ArgParser(description="Causal Bayesian Optimisation (CBO) on the B200 acquisition sweep.")
        for flag, default, kind, text in self.FLAGS:
            self.parser.add_argument(flag, default=default, type=kind, help=text)
        # build-specific, optional
        self.parser.add_argument("--grid_points", default=100, type=int, help="candidate grid points per dimension")
        self.parser.add_argument("--device", default="cuda:0", type=str, help="CUDA device of the sweep")
        self.parser.add_argument("--refine_acquisition", action="store_true",
                                 help="refine each exploration set's grid maximum off the grid with on-device gradients "
                                      "(the reference's L-BFGS polish); off: the grid argmax")
        self.parser.add_argument("--optimize_surrogates", action="store_true",
                                 help="fit each exploration set's GP variance and lengthscale by marginal likelihood on the "
                                      "device at every refit (the reference's models[i].optimize(), whose result it discards); "
                                      "off: the reference's fixed variance 1 and lengthscale 1")

    def parse(self, verbose=False, argv=None):
        args = self.parser.parse_args(argv)
        random.seed(args.seed)
        if verbose is True:
            print("================================== Parsed arguments ==================================")
            for key in ["exploration_set", "initial_num_obs_samples", "num_interventions", "type_cost", "num_trials",
                        "causal_prior", "experiment", "task"]:
                print(key, getattr(args, key))
            print("======================================================================================")
            print()
        return args
