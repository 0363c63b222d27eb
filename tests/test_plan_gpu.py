"""The planned step's integer plan (csrc/mf_v2.cuh), checked array by array.

The plan groups one minibatch's interactions by row: the user segments (members ascending by
interaction b), then the item segments (members ascending by term t, where term 2b is item[b] and
2b+1 is neg[b]).  Its output is restated here with a stable torch argsort and compared exactly; the
float kernels' bit-exactness rests on this contract.
"""

import ctypes

import numpy as np
import pytest
import torch

from spotlight_b200 import _lib, ops

pytestmark = pytest.mark.gpu

SCAN_TILE = 4096            # rows per scan tile (segindex.cuh SEG_SCAN_TILE)


def _cap(dim):
    """Members above which a row is "hot" (seg_sort_cap(lpr_for_dim(dim)) in the library)."""
    lpr = dim // 4
    lpr = 32 if lpr >= 32 else 1 << (lpr - 1).bit_length()
    return 128 if lpr >= 8 else (64 if lpr >= 4 else 16 * lpr)


class Planner(object):
    """One planned-step workspace of capacity `cap_batch`; builds plans through phase bit 1."""

    def __init__(self, U, I, dim, cap_batch, dev):
        self.lib = _lib.load()
        self.U, self.I, self.dim, self.cap_batch, self.dev = U, I, dim, cap_batch, dev
        small = torch.zeros((1, dim), device=dev)
        one = torch.zeros((1, 1), device=dev)
        self.keep = [small, one]
        ids = torch.zeros(cap_batch, dtype=torch.int64, device=dev)
        self.args = a = ops.mf_step_args(small, small, one, one, ids, ids, ids, 'bpr', 1, batch=cap_batch)
        a.num_users, a.num_items, a.dim = U, I, dim       # the plan reads ids only, never the tables
        a.grad_mode = _lib.GRAD_COMPACT
        a.opt, a.lr, a.eps = _lib.OPT_ADAGRAD, 0.1, 1e-10
        a.state_Wu = a.state_Wi = a.state_bu = a.state_bi = small.data_ptr()
        self.loss = torch.zeros(1, device=dev)
        a.loss_out = self.loss.data_ptr()
        need = self.lib.slb_mf_fused_workspace_bytes(cap_batch, U, I, dim)
        assert need > 0
        self.fws = torch.zeros(need, dtype=torch.uint8, device=dev)
        a.fused_workspace, a.fused_workspace_bytes = self.fws.data_ptr(), need
        wneed = self.lib.slb_mf_step_workspace_bytes(cap_batch, 1, a.loss, U, I)
        self.ws = torch.zeros(wneed, dtype=torch.uint8, device=dev)
        a.workspace, a.workspace_bytes = self.ws.data_ptr(), wneed

    def build(self, users, items, negs, slot=0):
        """Enqueues the plan of (users, items, negs) in `slot` on the current stream."""
        a = self.args
        # one workspace sized for cap_batch serves every smaller batch, as a sharded step's local
        # batch does
        a.users, a.items, a.negs = users.data_ptr(), items.data_ptr(), negs.data_ptr()
        a.batch = users.numel()
        try:
            _lib.check(self.lib.slb_mf_train_step_phases(ctypes.byref(a), 1 | (slot << 8), ops._stream()), 'plan')
        finally:
            a.batch = self.cap_batch

    def plan(self, users, items, negs, slot=0):
        """Builds the plan of (users, items, negs) in `slot` and returns its arrays (host numpy)."""
        self.build(users, items, negs, slot)
        return self.copy(users.numel(), slot)

    def copy_async(self, B, slot):
        """Device copies of the plan in `slot` (built over B interactions), on the current stream."""
        dev, R = self.dev, self.U + self.I
        i32 = dict(dtype=torch.int32, device=dev)
        out = dict(totals=torch.empty(4, **i32), seg_row=torch.empty(3 * B + 1, **i32),
                   seg_start=torch.empty(3 * B + 2, **i32), sid=torch.empty(R, **i32),
                   long_list=torch.empty(3 * B // 16 + 2, **i32), mu=torch.empty((B, 4), **i32),
                   mi=torch.empty((2 * B, 2), **i32))
        p = ops._ptr
        a = self.args
        a.batch = B
        try:
            _lib.check(self.lib.slb_mf_plan_copy(ctypes.byref(a), slot, B, p(out['totals']), p(out['seg_row']),
                                                 p(out['seg_start']), p(out['sid']), p(out['long_list']),
                                                 p(out['mu']), p(out['mi']), ops._stream()), 'plan_copy')
        finally:
            a.batch = self.cap_batch
        return out

    def copy(self, B, slot):
        out = self.copy_async(B, slot)
        torch.cuda.synchronize()
        return {k: v.cpu().numpy() for k, v in out.items()}


def expected(users, items, negs, U, I, cap):
    """The plan restated: stable argsorts of the user ids and of the item ids over terms 2b / 2b+1."""
    B = users.numel()
    terms = torch.stack([items, negs], 1).reshape(-1) + U          # row of term t
    cnt = torch.bincount(torch.cat([users, terms]), minlength=U + I)
    seg_row = torch.nonzero(cnt).reshape(-1)
    lens = cnt[seg_row]
    seg_start = torch.cat([torch.zeros(1, dtype=torch.int64, device=users.device), torch.cumsum(lens, 0)])
    sid = torch.full((U + I,), -1, dtype=torch.int64, device=users.device)
    sid[seg_row] = torch.arange(seg_row.numel(), device=users.device)
    ou = torch.argsort(users, stable=True)
    mu = torch.stack([ou, items[ou], negs[ou], torch.zeros_like(ou)], 1)
    ot = torch.argsort(terms, stable=True)
    mi = torch.stack([ot, sid[users[ot // 2]]], 1)
    hot = torch.nonzero(lens > cap).reshape(-1)
    n = lambda t: t.cpu().numpy()  # noqa: E731
    return dict(totals=np.array([seg_row.numel(), 3 * B, int((seg_row < U).sum()), hot.numel()]),
                seg_row=n(seg_row), seg_start=n(seg_start), sid=n(sid), hot=n(hot), mu=n(mu), mi=n(mi))


def check(got, exp):
    nseg, _, _, nlong = exp['totals']
    assert np.array_equal(got['totals'], exp['totals'])
    assert np.array_equal(got['seg_row'][:nseg], exp['seg_row'])
    assert np.array_equal(got['seg_start'][:nseg + 1], exp['seg_start'])
    assert np.array_equal(got['sid'][exp['seg_row']], exp['sid'][exp['seg_row']])
    assert np.array_equal(np.sort(got['long_list'][:nlong]), exp['hot'])
    assert np.array_equal(got['mu'], exp['mu'])
    assert np.array_equal(got['mi'], exp['mi'])


def run(planner, users, items, negs, slot=0):
    got = planner.plan(users, items, negs, slot)
    check(got, expected(users, items, negs, planner.U, planner.I, _cap(planner.dim)))
    return got


@pytest.fixture(scope='module')
def dev():
    if not torch.cuda.is_available():
        pytest.skip('needs a CUDA device')
    return torch.device('cuda:0')


def _ids(g, hi, n, dev):
    return torch.randint(0, hi, (n,), generator=g, device=dev)


def test_plan_bench_shape(dev):
    U, I, B = 1_000_000, 100_000, 524288
    pl = Planner(U, I, 64, B, dev)
    g = torch.Generator(device=dev).manual_seed(3)
    for slot in (0, 1):
        got = run(pl, _ids(g, U, B, dev), _ids(g, I, B, dev), _ids(g, I, B, dev), slot)
        assert got['totals'][3] == 0        # uniform ids: no row above the cap


def test_plan_zipf_hot_rows(dev):
    U, I, B = 50_000, 20_000, 200_000
    rs = np.random.RandomState(5)
    items = torch.from_numpy(np.minimum(rs.zipf(1.3, B) - 1, I - 1)).to(dev)
    negs = torch.from_numpy(rs.randint(0, I, B)).to(dev)
    users = torch.from_numpy(rs.randint(0, U, B)).to(dev)
    users[rs.choice(B, 3000, replace=False)] = 777           # one hot user row
    for dim in (64, 8):
        pl = Planner(U, I, dim, B, dev)
        got = run(pl, users, items, negs)
        hot = got['seg_row'][got['long_list'][:got['totals'][3]]]
        assert 777 in hot and (hot >= U).sum() >= 5


def test_plan_short_batch_and_one(dev):
    U, I, cap_batch = 300_000, 40_000, 65536
    pl = Planner(U, I, 64, cap_batch, dev)
    g = torch.Generator(device=dev).manual_seed(11)
    run(pl, _ids(g, U, cap_batch, dev), _ids(g, I, cap_batch, dev), _ids(g, I, cap_batch, dev), 0)
    run(pl, _ids(g, U, 12345, dev), _ids(g, I, 12345, dev), _ids(g, I, 12345, dev), 1)     # short last batch
    for slot in (0, 1):
        got = run(pl, _ids(g, U, 1, dev), _ids(g, I, 1, dev), _ids(g, I, 1, dev), slot)      # B = 1
        assert got['totals'][1] == 3


def test_plan_edge_rows(dev):
    # user and item rows at both ends of their ranges and on both sides of scan-tile boundaries
    U, I = 3 * SCAN_TILE + 5, 2 * SCAN_TILE + 17
    pl = Planner(U, I, 32, 4096, dev)
    R = U + I
    edge = [0, U - 1, U, R - 1]
    for t in range(1, R // SCAN_TILE + 1):
        edge += [t * SCAN_TILE - 1, t * SCAN_TILE]
    edge = sorted(set(r for r in edge if 0 <= r < R))
    urows = [r for r in edge if r < U]
    irows = [r - U for r in edge if r >= U]
    g = torch.Generator(device=dev).manual_seed(2)
    B = 4096
    users, items, negs = _ids(g, U, B, dev), _ids(g, I, B, dev), _ids(g, I, B, dev)
    users[:len(urows)] = torch.tensor(urows, device=dev)
    items[:len(irows)] = torch.tensor(irows, device=dev)
    negs[-len(irows):] = torch.tensor(irows, device=dev)
    run(pl, users, items, negs)
    # only edge rows, each once or twice: row U - 1 ends the user side, row U starts the items
    n = min(len(urows), len(irows))
    run(pl, torch.tensor(urows[:n], device=dev), torch.tensor(irows[:n], device=dev),
        torch.tensor(irows[::-1][:n], device=dev))


def test_plan_batch_shrinks_then_grows(dev):
    # A sharded step's local batch changes every step inside one workspace, and the plan of step
    # k + 1 is built in one slot while step k still reads the other.  Here each plan is built on a
    # side stream while the main stream copies out the previous one (other slot, other batch); both
    # must come out exact, so neither slot may land on the other whatever the two batches.
    U, I, cap_batch = 200_000, 30_000, 100_000
    pl = Planner(U, I, 64, cap_batch, dev)
    g = torch.Generator(device=dev).manual_seed(9)
    cap = _cap(64)
    side = torch.cuda.Stream(device=dev)
    prev = None
    for k, B in enumerate((90_000, 20_000, 3, 100_000, 50_000, 99_999, 1)):
        ids = (_ids(g, U, B, dev), _ids(g, I, B, dev), _ids(g, I, B, dev))
        side.wait_stream(torch.cuda.current_stream(dev))
        with torch.cuda.stream(side):
            pl.build(*ids, slot=k & 1)
        if prev is not None:
            old = pl.copy_async(prev[0].numel(), (k - 1) & 1)       # concurrent with the build above
        torch.cuda.synchronize()
        if prev is not None:
            check({n: v.cpu().numpy() for n, v in old.items()}, expected(*prev, U, I, cap))
        check(pl.copy(B, k & 1), expected(*ids, U, I, cap))
        prev = ids
