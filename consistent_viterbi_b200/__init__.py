"""consistent_viterbi_b200 -- B200-native (sm_100a) hot path of consistent-viterbi.

The package directory uses an underscore (Python cannot import a hyphenated
name); it holds only what the hot path needs: csrc/ (CUDA kernels + the C ABI of
include/cv_b200.h) and the host-side mirror of the reference's solver interface.
"""
from . import _lib
from ._lib import CvError
from .hmm import HMM
from .viterbi import decode, decode_batch, decode_batch_f32, decode_batch_kbest, decode_batch_narrow, decode_kbest
from .posterior import loglik_batch, posterior_batch, score
from .cp import CPSolver, CpDistGroup, Solver, cfn_tables, cp_solve_arrays, plan_cuts
from .superseq import Constraints, SuperSequence, load_sequences, load_tags

__all__ = ["HMM", "decode", "decode_batch", "decode_batch_narrow", "decode_batch_f32", "decode_batch_kbest", "decode_kbest", "loglik_batch", "posterior_batch", "score", "CPSolver", "Solver", "cp_solve_arrays", "CpDistGroup", "plan_cuts", "cfn_tables", "Constraints",
           "SuperSequence", "load_sequences", "load_tags", "CvError", "_lib"]
