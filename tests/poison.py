"""Poison the library's reused device result buffers before a host-form call under test.

The host forms (pair lists, rectangles, both orientations, gapped strings) write into the context's
own device buffers and download them.  Those buffers only grow and are reused from call to call, so a
pair a kernel leaves unwritten would come back holding whatever an earlier call left in its slot --
often the right answer, when two kernels are compared on the same inputs.  `poison` first fills
`npairs` slots with the result of one pair of identical sequences of `length` bases: every slot then
holds a count `same == length` (and a score of length x match), which no pair of shorter sequences
can reach.  It loads set 0; the caller reloads its own sets afterwards."""
from __future__ import annotations

import numpy as np


def poison(engine, npairs: int, length: int) -> None:
    seq = (b"ACGT" * (length // 4 + 1))[:length]
    engine.load([seq], 0)
    zero = np.zeros(max(int(npairs), 1), dtype=np.int32)
    got = engine.align_pairs(zero, zero)
    assert (got["counts"][:, 0] == length).all()
