"""Device time of each kernel of the planned step's integer plan, run alone.

Builds the plan of one bench-shape minibatch (1 M users x 100 K items, B = 524 288, uniform ids)
through slb_mf_train_step_phases bit 1, N times back to back under torch.profiler, and prints one
JSON line: mean device microseconds per plan, per kernel, with the card and its power limit.

    python profiles/plan_kernels.py [--iters 50] [--label name]
"""

import argparse
import ctypes
import json
import os
import re
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--iters', type=int, default=50)
    ap.add_argument('--label', default='')
    cli = ap.parse_args()

    import torch
    from torch.profiler import ProfilerActivity, profile
    from spotlight_b200 import _lib, ops
    sys.path.insert(0, os.path.join(ROOT, 'profiles'))
    import plan_overlap

    U, I, D, B = 1_000_000, 100_000, 64, 524288
    dev = torch.device('cuda', 0)
    torch.cuda.set_device(dev)
    g = torch.Generator(device=dev).manual_seed(1234)
    users, items, negs = (torch.randint(0, n, (B,), device=dev, generator=g) for n in (U, I, I))
    Wu, Wi = torch.zeros((U, D), device=dev), torch.zeros((I, D), device=dev)
    bu, bi = torch.zeros((U, 1), device=dev), torch.zeros((I, 1), device=dev)
    lib = _lib.load()
    a = ops.mf_step_args(Wu, Wi, bu, bi, users, items, negs, 'bpr', 1, batch=B)
    a.grad_mode, a.opt, a.lr, a.eps = _lib.GRAD_COMPACT, _lib.OPT_ADAGRAD, 0.05, 1e-10
    a.state_Wu, a.state_Wi, a.state_bu, a.state_bi = Wu.data_ptr(), Wi.data_ptr(), bu.data_ptr(), bi.data_ptr()
    loss = torch.zeros(1, device=dev)
    a.loss_out = loss.data_ptr()
    fws = torch.zeros(lib.slb_mf_fused_workspace_bytes(B, U, I, D), dtype=torch.uint8, device=dev)
    a.fused_workspace, a.fused_workspace_bytes = fws.data_ptr(), fws.numel()
    ws = torch.zeros(lib.slb_mf_step_workspace_bytes(B, 1, a.loss, U, I), dtype=torch.uint8, device=dev)
    a.workspace, a.workspace_bytes = ws.data_ptr(), ws.numel()
    stream = ops._stream()
    for _ in range(5):
        _lib.check(lib.slb_mf_train_step_phases(ctypes.byref(a), 1, stream), 'plan')
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(cli.iters):
        _lib.check(lib.slb_mf_train_step_phases(ctypes.byref(a), 1, stream), 'plan')
    e1.record()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(cli.iters):
            _lib.check(lib.slb_mf_train_step_phases(ctypes.byref(a), 1, stream), 'plan')
        torch.cuda.synchronize()
    per = {}
    for e in prof.events():
        if e.device_type.name != 'CUDA':
            continue
        m = re.search(r'(\w+_kernel)', e.name)
        name = m.group(1) if m else e.name
        per[name] = per.get(name, 0.0) + e.device_time_total / cli.iters
    print(json.dumps({'label': cli.label, 'card': plan_overlap.card(), 'batch': B, 'iters': cli.iters,
                      'events_us_per_plan': e0.elapsed_time(e1) * 1e3 / cli.iters,
                      'kernel_us_per_plan': {k: round(v, 2) for k, v in sorted(per.items(), key=lambda t: -t[1])},
                      'kernel_sum_us': round(sum(per.values()), 2)}))


if __name__ == '__main__':
    main()
