"""Host-side pin of tests/test_sag_widths_gpu.py's case table: every row is a shape the native SAGPool steps accept,
with the head backward layout (narrow: k_head_bwd's per-CTA gradient row; wide: k_head_delta + K3's reductions) the
row claims, and every fallback case is refused.  The workspace queries are pure host functions of the shape, so a change
to HEAD_SMEM or to the step layouts fails here, on any machine, and names the GPU rows that have to move."""
import ctypes

import pytest

from test_sag_widths_gpu import FALLBACK, LARGE, PAIRS, ROWS

QUERIES = ("tsg_sag_nll_step_workspace_bytes", "tsg_sag_classify_workspace_bytes", "tsg_sag_triplet_step_workspace_bytes")


def _queries(H, C):
    # num_graphs = 1, as PackedSAGNet._head_fits asks: the answer depends on the head's shape, not on the batch
    from tsg import _lib
    shape = _lib.SagShape(1, 89, H, 0)
    head = _lib.SagHead(C, 1, 0.0, 0.0, 0.0, 0)
    return {q: getattr(_lib.lib, q)(ctypes.byref(shape), ctypes.byref(head)) for q in QUERIES}


def _k3_head_bytes(H):
    # K3's reduction workspace for lin1's weight gradient: only the wide layout reserves it (and it is the largest of the
    # three layers' reductions)
    from tsg import _lib
    return _lib.lib.tsg_linear_bwd_weight_workspace_bytes(H, 2 * H)


ACCEPTED = [(r[0], r[1], r[-1]) for r in ROWS] + [(r[2], r[3], r[-1]) for r in LARGE]


@pytest.mark.parametrize("H,C,head", ACCEPTED)
def test_every_row_is_accepted_with_the_head_layout_it_claims(H, C, head):
    from tsg import _lib
    q = _queries(H, C)
    assert all(v > 0 for v in q.values()), f"nhid {H}, C {C} is no longer accepted ({q}): move the row in test_sag_widths_gpu.py"
    assert _lib.lib.tsg_embed_bwd_weight_workspace_bytes(89, H) > 0, "the 89-label table no longer fits the embed kernels"
    wide = q["tsg_sag_nll_step_workspace_bytes"] >= _k3_head_bytes(H)
    assert wide == (head == "wide"), (f"nhid {H}, C {C} now takes the {'wide' if wide else 'narrow'} head backward, "
                                      f"the row says {head}: move it in test_sag_widths_gpu.py")


@pytest.mark.parametrize("H,C", [(r[0], r[1]) for r in FALLBACK])
def test_every_fallback_case_is_refused(H, C):
    assert list(_queries(H, C).values()) == [0, 0, 0], f"nhid {H}, C {C} is now accepted: it is no fallback case any more"


@pytest.mark.parametrize("H,c_narrow,c_wide", PAIRS)
def test_each_pair_sits_on_both_sides_of_the_head_switch(H, c_narrow, c_wide):
    """One class more moves the pair's head from k_head_bwd to k_head_delta + K3: the wide row's NLL workspace holds K3's
    reduction workspace for lin1 (at least tsg_linear_bwd_weight_workspace_bytes(H, 2H)); the narrow row's does not (its
    k_head_bwd gradient rows are far smaller, so the literal difference of the two is a little below that size)."""
    narrow = _queries(H, c_narrow)["tsg_sag_nll_step_workspace_bytes"]
    wide = _queries(H, c_wide)["tsg_sag_nll_step_workspace_bytes"]
    k3 = _k3_head_bytes(H)
    assert 0 < narrow < k3 <= wide, (H, c_narrow, narrow, c_wide, wide, k3)
