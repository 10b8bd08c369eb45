"""valida_b200 — B200-native STARK prover backend for Valida's Machine::prove() hot path.

Host-side mirror of the reference's prover-facing interface (StarkConfig / UnivariatePcsWithLde /
Machine::prove) over the C ABI in include/valida_b200.h.  There is no CPU fallback: constructing a
Context without a CUDA device raises.
"""
from .api import (  # noqa: F401
    BABYBEAR_P,
    Context,
    DeviceMatrix,
    ProverData,
    Radix2Dft,
    TwoAdicFriPcs,
    MachineTraces,
    VgpuError,
    StarkConfig,
    prove_machine,
    verify_machine,
    verify_machines,
    last_verify_batch_phases,
    VerificationError,
    last_prove_phases,
    fib_program,
    generate_permutation_trace,
    quotient,
    lib,
    lib_path,
    run_program,
    run_program_log,
    VmLog,
    comm_unique_id,
    comm_init_local,
    run_ranks,
    shard_range,
    split_column_plan,
    tree_share,
)
