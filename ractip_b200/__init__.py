"""ractip_b200 -- B200-native probability stage for RactIP (McCaskill inside/outside,
two-strand co-fold / duplex partition functions, unpaired-window accessibilities).

The arithmetic lives in hand-written sm_100a CUDA kernels behind the C ABI of
include/ractip_prob.h (libractip_prob.so, built in-tree by ractip_b200/build.py).
Importing this package never falls back to a CPU implementation: using the stage
without the built library or without a GPU raises.
"""
from .stage import (DeviceBatch, PairProbabilities, PairRecords, ProbabilityStage, RpError,
                    bp_offsets, default_model, default_opts, dot_bracket, joint_structure, sample_opts, shape_deigan,
                    zscore_shuffles)

from .ip import (IPModel, JointPrediction, default_ip_opts, energy_of_duplex, energy_of_structure,  # noqa: E402
                 solve_joint, solve_ss, zscore_statistic)

from .frontend import (FastaRecord, PairResult, format_result, input_pairs, load_fasta, parse_fasta,  # noqa: E402
                       predict, read_shape)

__all__ = ["FastaRecord", "PairResult", "format_result", "input_pairs", "load_fasta", "parse_fasta", "predict", "read_shape", "IPModel", "JointPrediction", "default_ip_opts", "energy_of_duplex", "energy_of_structure",
           "solve_joint", "solve_ss", "zscore_statistic", "DeviceBatch", "PairProbabilities", "PairRecords", "ProbabilityStage", "RpError",
           "bp_offsets", "default_model", "default_opts", "dot_bracket", "joint_structure", "sample_opts", "shape_deigan",
           "zscore_shuffles"]
