"""lasso_b200 — B200-native (sm_100a) accelerator for the a16z/Lasso prover hot path.

Host-side mirror of the reference's surface for that path (names follow the Rust items):

    DensifiedRepresentation.from_lookup_indices(ctx, indices, log_m)     src/lasso/densified.rs:22
        (indices: a host array, or a CUDA tensor read in place on the device)
    DensifiedRepresentation.commit(gens)                                 src/lasso/densified.rs:78
    SparsePolyCommitmentGens.new(ctx, label, c, s, num_memories, log_m)  src/lasso/surge.rs:32
    SparsePolynomialEvaluationProof.prove(ctx, strategy, dense, r, gens, ...)   src/lasso/surge.rs:119

Everything runs through the C-ABI shared library (include/lasso_b200.h); there is no CPU fallback:
importing works without a GPU, but creating a Context raises.
"""
from .api import (  # noqa: F401
    AND, IDX_I32, IDX_I64, IDX_U32, IDX_U64, LT, OR, RANGE_CHECK, XOR,
    Context, DensifiedRepresentation, LassoError, MsmJob, SparsePolyCommitmentGens, SparsePolynomialEvaluationProof,
    Strategy, bind_bot, bind_top, commit_rows, eq_evals, gather_lookup_polys, gens_points_needed, lib,
    library_path, materialize_subtables, msm, sample_generators, sumcheck_bind_round_arbitrary, sumcheck_round_arbitrary,
    sumcheck_round_cubic,
)
