"""llama2.zig_b200 — B200 (sm_100a) drop-in for llama2.zig's `transformer()` hot path.

The product is the C-ABI shared library built from ``csrc/`` (``lib/libllama2_b200.so``,
declared in ``include/llama2_b200.h``).  This package is only the thin Python host used by
the tests and ``bench.py``: a ctypes binding whose names mirror the reference's own functions
(`transformer`, `matmul`, `rmsnorm`, `softmax`, `vector_weighted_sum_rows`;
/root/reference/src/main.zig:285-713) so the parity tests read like the reference's tests.

There is no CPU fallback anywhere in this package: if the CUDA library is missing or no
sm_100 device is present, calls raise `L2BError`.

The directory name contains a dot, so import it through the root alias module
``llama2_zig_b200`` (``import llama2_zig_b200 as l2b``).
"""
from .binding import (  # noqa: F401
    L2BError,
    L2BConfig,
    L2BShard,
    Transformer,
    checkpoint_floats,
    comm_unique_id,
    lib_path,
    load_library,
    matmul,
    rmsnorm,
    softmax,
    synth_checkpoint_host,
    vector_weighted_sum_rows,
    attention_head,
    fused_matmul,
    sample_prep,
    exported_symbols,
    forward_batch,
    generate_argmax_batch,
)
from .checkpoint import Checkpoint, read_checkpoint, MODEL_SHAPES  # noqa: F401

__all__ = [
    "L2BError", "L2BConfig", "L2BShard", "Transformer", "checkpoint_floats", "comm_unique_id",
    "lib_path", "load_library", "matmul", "rmsnorm", "softmax", "synth_checkpoint_host",
    "vector_weighted_sum_rows", "attention_head", "fused_matmul", "sample_prep", "exported_symbols", "forward_batch",
    "generate_argmax_batch", "Checkpoint",
    "read_checkpoint", "MODEL_SHAPES",
]
