"""CPU oracle for the TaxI2 pairwise-distance path.  TEST INFRASTRUCTURE ONLY.

Only tests/, __graft_entry__.smoke() and bench.py's CPU-baseline legs may import this package.
The product package (taxi2_b200) never does; it fails loudly when its CUDA library is missing.
See oracle/taxi_oracle.c for what is restated and the parity status ("tie-breaking unpinned").
"""
from .oracle import (  # noqa: F401
    align,
    align_count_pairs,
    build,
    count,
    count_pairs,
    max_threads,
    metrics,
    metrics_batch,
    uses_gotoh,
)
