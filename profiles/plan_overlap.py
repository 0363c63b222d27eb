"""How much of the planned step's integer plan the float kernels fail to hide.

One process at the bench shape (bench.py defaults: 1 M users x 100 K items x 64, B = 524 288, BPR,
Adagrad, K = 100 steps after W = 10 warm-up steps, same allocator priming).  Per step, in us:

  a        the epoch exactly as bench.py times it (plan on its own stream, one step ahead)
  a_prio   the same with the plan stream at the other priority (normal if the library's default is
           high, high if it is normal)
  b        the same epoch with SLB_PLAN_SAME_STREAM=1: plan and float kernels serialised
  c        floor: K back-to-back float phases (slb_mf_train_step_phases, phases = 6) over one plan
           built beforehand, no sync in between, on clones of the tables and Adagrad sums (what it
           trains is thrown away)
  sampler  the epoch's negative draws alone on the side stream (device time / K)

exposed = a - c - sampler is what the plan adds to a step.  The three epochs and the floor are
interleaved, R rounds; medians are printed as one JSON line, with the card and its power limit.

    python profiles/plan_overlap.py [--rounds 3] [--steps 100] [--warmup 10]
"""

import argparse
import ctypes
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def card():
    try:
        out = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit', '--format=csv,noheader'],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return out[0] if out else None
    except (OSError, subprocess.SubprocessError):
        return None


def floor_args(model, users, items, negs, a):
    """slb_mf_step_args of one planned step (as bench.kernel_breakdown) over clones of the model's
    tables and Adagrad sums: what the floor trains is thrown away, the model stays as it was."""
    import torch
    from spotlight_b200 import _lib, ops
    lib = _lib.load()
    net, opt = model._net, model._optimizer
    dev = users.device
    B = a.batch
    params = [p.detach().clone() for p in (net.user_embeddings.weight, net.item_embeddings.weight,
                                            net.user_biases.weight, net.item_biases.weight)]
    states = [opt.fused_state(p).clone() for p in (net.user_embeddings.weight, net.item_embeddings.weight,
                                                   net.user_biases.weight, net.item_biases.weight)]
    Wu, Wi, bu, bi = params
    st = ops.mf_step_args(Wu, Wi, bu, bi, users[:B], items[:B], negs[:B], a.loss, 1, batch=B)
    st.grad_mode = _lib.GRAD_COMPACT
    keep = [torch.empty(64, device=dev)] + params + states
    need = lib.slb_mf_fused_workspace_bytes(B, a.users, a.items, a.dim)
    assert need, 'the planned step is not available at this shape'
    keep.append(ops.workspace('mfv2_%d_%d_%d' % (a.users, a.items, a.dim), need, dev))
    st.fused_workspace, st.fused_workspace_bytes = keep[-1].data_ptr(), keep[-1].numel()
    st.loss_out = keep[0].data_ptr()
    hp = opt.fused_hparams()
    st.opt, st.lr, st.weight_decay, st.eps = opt.fused_kind, hp['lr'], hp['weight_decay'], hp['eps']
    st.state_Wu, st.state_Wi, st.state_bu, st.state_bi = [s.data_ptr() for s in states]
    wneed = lib.slb_mf_step_workspace_bytes(B, 1, st.loss, a.users, a.items)
    keep.append(ops.workspace('mf%d_%d' % (a.users, a.items), wneed, dev))
    st.workspace, st.workspace_bytes = keep[-1].data_ptr(), keep[-1].numel()
    return st, keep


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--rounds', type=int, default=3)
    ap.add_argument('--steps', type=int, default=100)
    ap.add_argument('--warmup', type=int, default=10)
    ap.add_argument('--label', default='')
    cli = ap.parse_args()

    import torch
    import bench
    from spotlight_b200 import _lib, ops
    from spotlight_b200 import rng as _rng
    from spotlight_b200.factorization import implicit
    from spotlight_b200.sampling import sample_items

    a = argparse.Namespace(users=1_000_000, items=100_000, dim=64, batch=524288, loss='bpr', lr=0.05)
    model = bench.build_model(a, 0)
    dev = torch.device('cuda', 0)
    B, K, W = a.batch, cli.steps, cli.warmup
    g = torch.Generator(device=dev).manual_seed(1234)
    n = (K + W) * B
    users = torch.randint(0, a.users, (n,), device=dev, generator=g)
    items = torch.randint(0, a.items, (n,), device=dev, generator=g)
    model._run_epoch_device(users[:W * B], items[:W * B])
    _prime = torch.empty(K * B, dtype=torch.int64, device=dev)
    with torch.cuda.stream(implicit._side_stream(dev)):
        _rng.reserve(a.items, min(64, K) * B, dev)
    del _prime
    tu, ti = users[W * B:], items[W * B:]

    def timed(fn):
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) * 1e3 / K          # us per step

    plan_stream = implicit._plan_stream(dev)
    other = torch.cuda.Stream(device=dev, priority=0 if plan_stream.priority < 0 else -1)

    def epoch():
        model._run_epoch_device(tu, ti)

    def epoch_other_priority():
        implicit._PLAN_STREAMS[dev.index] = other
        try:
            model._run_epoch_device(tu, ti)
        finally:
            implicit._PLAN_STREAMS[dev.index] = plan_stream

    def epoch_same_stream():
        os.environ['SLB_PLAN_SAME_STREAM'] = '1'
        try:
            model._run_epoch_device(tu, ti)
        finally:
            del os.environ['SLB_PLAN_SAME_STREAM']

    lib = _lib.load()
    negs = sample_items(a.items, K * B, random_state=np.random.RandomState(1), device=dev)
    st, keep = floor_args(model, tu, ti, negs, a)
    stream = ops._stream()

    def floor():
        # the epochs share this workspace: rebuild the floor's plan first (not timed)
        _lib.check(lib.slb_mf_train_step_phases(ctypes.byref(st), 1, stream), 'plan')
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(K):
            _lib.check(lib.slb_mf_train_step_phases(ctypes.byref(st), 6, stream), 'float phases')
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) * 1e3 / K

    side = implicit._side_stream(dev)

    def sampler():
        rs = np.random.RandomState(3)
        out = torch.empty(K * B, dtype=torch.int64, device=dev)
        side.wait_stream(torch.cuda.current_stream(dev))
        with torch.cuda.stream(side):
            ds = _rng.DeviceStream(rs, dev)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(side)
            lo, chunk = 0, 48 * B
            while lo < K * B:
                cur = min(chunk, K * B - lo)
                ds.draw(a.items, cur, out=out[lo:lo + cur])
                lo += cur
            e1.record(side)
            ds.finish()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) * 1e3 / K

    rows = {k: [] for k in ('a', 'a_prio', 'b', 'c', 'sampler')}
    for _ in range(cli.rounds):
        rows['a'].append(timed(epoch))
        rows['b'].append(timed(epoch_same_stream))
        rows['a_prio'].append(timed(epoch_other_priority))
        rows['c'].append(floor())
        rows['sampler'].append(sampler())
    med = {k: float(np.median(v)) for k, v in rows.items()}
    line = {'label': cli.label, 'card': card(), 'steps': K, 'batch': B, 'rounds': cli.rounds,
            'plan_stream_priority': plan_stream.priority, 'a_prio_priority': other.priority,
            'us_per_step': med, 'runs': rows,
            'exposed_plan_us': med['a'] - med['c'] - med['sampler'],
            'exposed_plan_us_other_priority': med['a_prio'] - med['c'] - med['sampler'],
            'serial_plan_us': med['b'] - med['c'] - med['sampler']}
    del keep
    print(json.dumps(line))


if __name__ == '__main__':
    main()
