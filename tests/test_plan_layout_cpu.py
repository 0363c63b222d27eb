"""Where a planned-step workspace puts its arrays (host only, no GPU).

The plan of step k+1 runs on its own stream in one slot while the float kernels of step k read the
other slot and the step state.  The sharded step's local batch changes every step, so two steps in
flight may have different batches: whatever the two batches, no array of one slot may overlap an
array of the other slot or of the step state.
"""

import ctypes

import pytest

from spotlight_b200 import _lib


def layout(lib, ws_bytes, batch, U, I, D):
    a = _lib.MfStepArgs()
    a.num_users, a.num_items, a.dim, a.batch = U, I, D, batch
    a.fused_workspace_bytes = ws_bytes
    out = (ctypes.c_int64 * 300)()
    n = lib.slb_mf_fused_layout(ctypes.byref(a), out, 100)
    assert 0 < n <= 100, (n, _lib.load().slb_last_error())
    return [tuple(out[3 * k:3 * k + 3]) for k in range(n)]


def overlap(x, y):
    return x[1] < y[2] and y[1] < x[2]


@pytest.mark.parametrize('U, I, D, cap', [(500_000, 100_000, 64, 262144), (1000, 300, 8, 4096),
                                          (3 * 4096 + 5, 2 * 4096 + 17, 128, 1000)])
def test_slots_never_overlap_across_batches(U, I, D, cap):
    lib = _lib.load()
    need = lib.slb_mf_fused_workspace_bytes(cap, U, I, D)
    ws_bytes = int(need * 1.25) + 4096               # as ops.workspace sizes it
    batches = sorted({1, 2, 3, cap // 4, cap // 2 + 1, cap - 300, cap - 1, cap, cap + 1, cap + 300})
    layouts = {m: layout(lib, ws_bytes, m, U, I, D) for m in batches if m > 0}
    for m, arrays in layouts.items():
        assert {g for g, _, _ in arrays} == {0, 1, 2}, 'an array of the layout belongs to no group'
        assert all(0 <= b <= e <= ws_bytes for _, b, e in arrays)
        spans = sorted(arrays, key=lambda t: t[1])
        assert all(x[2] <= y[1] for x, y in zip(spans, spans[1:])), 'arrays of one layout overlap'
    for m1, l1 in layouts.items():
        for m2, l2 in layouts.items():
            clash = [(x, y) for x in l1 for y in l2 if x[0] != y[0] and overlap(x, y)]
            assert not clash, (m1, m2, clash[:3])


def test_batch_above_capacity_is_refused():
    lib = _lib.load()
    U, I, D, cap = 1000, 300, 8, 4096
    ws_bytes = lib.slb_mf_fused_workspace_bytes(cap, U, I, D)
    assert len(layout(lib, ws_bytes, cap, U, I, D)) > 0
    a = _lib.MfStepArgs()
    a.num_users, a.num_items, a.dim, a.batch = U, I, D, cap + 64
    a.fused_workspace_bytes = ws_bytes
    out = (ctypes.c_int64 * 300)()
    assert lib.slb_mf_fused_layout(ctypes.byref(a), out, 100) < 0
