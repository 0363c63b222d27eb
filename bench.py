#!/usr/bin/env python
"""Headline benchmark: interactions/sec, BPR matrix factorisation, 1M users x
100K items x dim 64 (BASELINE.json configs[1]), synthetic uniform ids.

    python bench.py --gpus N --steps K --warmup W [--impl reference]

A *step* is one minibatch through the fit() hot path: negative draw (device
MT19937, bit-exact with NumPy), the integer plan of the minibatch (row index of
both tables, on its own stream), mf_user_kernel (forward + user-row gradient +
in-place row-wise Adagrad) and mf_item_kernel (item-row gradient + update):
csrc/mf_v2.cuh, deterministic (no float atomics).

One JSON line on stdout (rank 0):
  value      whole-job interactions/s with ids resident in HBM (device timed,
             CUDA events, max over ranks)
  e2e        the same metric through the public API with HOST numpy ids in
             page-locked memory, wall clock around the whole call:
             ImplicitFactorizationModel.fit(Interactions) at N = 1,
             ShardedImplicitFactorizationModel.fit(Interactions) at N > 1 --
             H2D of the ids, range check, the bit-exact RandomState.shuffle
             permutation (on the device), id gather, device negatives, K training
             steps, D2H of the per-batch losses.  Two consecutive calls; `value`
             is the second, `first_call_value` the first (allocator cold).
  roofline   dominant kernel: algorithmic bytes / CUDA-event duration vs the
             measured HBM copy bandwidth (MEASURED_PEAKS.json)
  cpu_baseline  the unmodified reference (oracle/_ref, kind "reference"; the
             torch-CPU restatement oracle/torch_port.py, kind "port", only if the
             install is absent) timed on this box's host cores on a bounded sample
             of the same workload

``--impl reference`` times only that CPU arm (all host threads) on the same
config and prints the same line shape with "impl": "reference".

``--dump-outputs DIR`` (single GPU) writes, right after the timed steps, what they
hand their caller as DIR/<name>.npy: ``epoch_loss`` (float64) and a fixed seeded
sample of rows of the four trained tables with their Adagrad sums (float32, about
34 MB at the default shape).  Ids, initial weights and the sample are seeded, so two
builds run with the same arguments can be compared output for output.
"""

import argparse
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = 'interactions/sec (BPR MF, 1Mx100Kx64)'
UNIT = 'interactions/s'


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=100)
    ap.add_argument('--warmup', type=int, default=10)
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--batch', type=int, default=524288)
    ap.add_argument('--users', type=int, default=1_000_000)
    ap.add_argument('--items', type=int, default=100_000)
    ap.add_argument('--dim', type=int, default=64)
    ap.add_argument('--loss', default='bpr')
    ap.add_argument('--lr', type=float, default=0.05)
    ap.add_argument('--cpu-steps', type=int, default=4)
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--no-e2e', action='store_true')
    ap.add_argument('--exchange', default='auto', choices=['auto', 'a2a', 'dense'])
    ap.add_argument('--dump-outputs', metavar='DIR', default=None,
                    help='write what the timed steps computed as DIR/<name>.npy (single GPU, --impl ours)')
    a = ap.parse_args()
    if a.dump_outputs and (a.impl != 'ours' or int(os.environ.get('WORLD_SIZE', '1')) > 1):
        ap.error('--dump-outputs is supported for --impl ours on a single GPU')
    return a


def workload_config(a, n_gpus):
    return {'workload': 'synthetic uniform 1M users x 100K items, BilinearNet dim=64, bpr_loss '
                        '(BASELINE.json configs[1])',
            'num_users': a.users, 'num_items': a.items, 'dim': a.dim, 'loss': a.loss,
            'batch': a.batch, 'optimizer': 'adagrad(lr=%g), row-wise fused' % a.lr,
            'negatives': 'device MT19937 masked rejection (numpy-bit-exact)',
            'parallelism': 'single GPU' if n_gpus == 1 else 'replicas x%d' % n_gpus,
            'l2': 'inputs (embedding tables 282 MB + ids) exceed the 126 MB L2; no flush'}


# --------------------------------------------------------------------------
# clocks
# --------------------------------------------------------------------------

class ClockSampler(object):
    """SM clock and throttle reasons sampled in-process through NVML (nvidia_ml_py).

    NVML is initialised and the sampling thread started well BEFORE the warm-up; only
    samples whose timestamp falls inside [mark_begin, mark_end] are reported.  (Round 1
    spawned `nvidia-smi -lms` right before the timed region, so its start-up -- NVML
    attaching to every GPU of the node -- ran inside a 12 ms timed region; that is the
    prime suspect for the one-off ~65 ms stall the 8-GPU node showed.  Nothing is spawned
    or initialised near the timed region any more.)
    """
    NAMES = (('hw_slowdown', 0x8), ('hw_thermal_slowdown', 0x40), ('sw_thermal_slowdown', 0x20),
             ('sw_power_cap', 0x4))

    def __init__(self, index=0, period_s=0.001):
        self.index, self.period = index, period_s
        self.samples, self.t0, self.t1 = [], None, None
        self._stop = threading.Event()
        self._thread, self._h, self._nv = None, None, None
        self.max_mhz = None

    def start(self):
        try:
            import pynvml as nv
            nv.nvmlInit()
            h = None
            try:
                import torch
                uuid = str(torch.cuda.get_device_properties(self.index).uuid)
                h = nv.nvmlDeviceGetHandleByUUID(('GPU-' + uuid) if not uuid.startswith('GPU-') else uuid)
            except Exception:
                vis = os.environ.get('CUDA_VISIBLE_DEVICES')
                phys = int(vis.split(',')[self.index]) if vis and vis.split(',')[self.index].isdigit() \
                    else self.index
                h = nv.nvmlDeviceGetHandleByIndex(phys)
            self._nv, self._h = nv, h
            self.max_mhz = float(nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM))
            self._thread = threading.Thread(target=self._run, daemon=True)
            self._thread.start()
        except Exception as exc:            # no NVML: the line says so instead of inventing clocks
            self._err = repr(exc)[:200]
        return self

    def _run(self):
        nv, h = self._nv, self._h
        while not self._stop.is_set():
            try:
                mhz = nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)
                try:
                    rs = nv.nvmlDeviceGetCurrentClocksEventReasons(h)
                except Exception:
                    rs = nv.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                self.samples.append((time.perf_counter(), float(mhz), int(rs)))
            except Exception:
                pass
            time.sleep(self.period)

    def nvlink_kib(self):
        """Cumulative NVLink payload counters of this GPU (KiB transmitted, KiB received), summed
        over its links, from the driver's hardware counters (NVML field values); None if absent."""
        if self._h is None:
            return None
        nv = self._nv
        try:
            vals = nv.nvmlDeviceGetFieldValues(self._h, [(nv.NVML_FI_DEV_NVLINK_THROUGHPUT_DATA_TX, 0xFFFFFFFF),
                                                         (nv.NVML_FI_DEV_NVLINK_THROUGHPUT_DATA_RX, 0xFFFFFFFF)])
            out = []
            for v in vals:
                if v.nvmlReturn != 0:
                    return None
                out.append(int(v.value.ullVal))
            return tuple(out)
        except Exception:
            return None

    def mark_begin(self):
        self.nv0 = self.nvlink_kib()
        self.t0 = time.perf_counter()

    def mark_end(self):
        self.t1 = time.perf_counter()
        self.nv1 = self.nvlink_kib()

    def nvlink_delta_bytes(self):
        a, b = getattr(self, 'nv0', None), getattr(self, 'nv1', None)
        if not a or not b:
            return None
        return {'tx_bytes': (b[0] - a[0]) * 1024, 'rx_bytes': (b[1] - a[1]) * 1024}

    def stop(self):
        self._stop.set()
        if self._thread is not None:
            self._thread.join(timeout=1.0)
        if self._thread is None:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': [], 'samples': 0,
                    'error': getattr(self, '_err', 'NVML unavailable')}
        inside = [x for x in self.samples if self.t0 is not None and self.t0 <= x[0] <= self.t1]
        note = None
        if not inside and self.samples and self.t0 is not None:
            # region shorter than the sampling period: the two samples that bracket it
            before = [x for x in self.samples if x[0] < self.t0][-1:]
            after = [x for x in self.samples if x[0] > self.t1][:1]
            inside, note = before + after, 'region shorter than the sampling period: bracketing samples'
        sm = [x[1] for x in inside]
        bits = 0
        for x in inside:
            bits |= x[2]
        out = {'sm_mhz': float(np.median(sm)) if sm else None, 'sm_max_mhz': self.max_mhz,
               'reasons': sorted(n for n, b in self.NAMES if bits & b), 'samples': len(sm),
               'source': 'NVML in-process, %.0f ms period, started before warm-up' % (self.period * 1e3)}
        if note:
            out['note'] = note
        return out


# --------------------------------------------------------------------------
# CPU port (cpu_baseline and the reference arm)
# --------------------------------------------------------------------------

REF_DIR = os.path.join(ROOT, 'oracle', '_ref')


def _reference_runner(a):
    """fit_steps(lo, nsteps) on the UNMODIFIED reference (oracle/_ref, installed by build() from a
    reference checkout, oracle/reference.py: `spotlight.factorization.implicit.ImplicitFactorizationModel.fit`
    on CPU through its own public API), or None when the install is not on this box."""
    if not os.path.isdir(os.path.join(REF_DIR, 'spotlight')):
        return None
    import torch
    if REF_DIR not in sys.path:
        sys.path.insert(0, REF_DIR)
    try:
        from spotlight.factorization.implicit import ImplicitFactorizationModel as RefModel
        from spotlight.interactions import Interactions as RefInteractions
    except Exception:
        return None
    model = RefModel(loss=a.loss, embedding_dim=a.dim, n_iter=1, batch_size=a.batch, learning_rate=a.lr,
                     optimizer_func=lambda p: torch.optim.Adagrad(p, lr=a.lr), use_cuda=False,
                     random_state=np.random.RandomState(42))

    def fit_steps(users, items, nsteps):
        n = nsteps * a.batch
        model.fit(RefInteractions(users[:n].astype(np.int32), items[:n].astype(np.int32),
                                  num_users=a.users, num_items=a.items))
    return fit_steps


def _port_runner(a):
    import torch
    from oracle import torch_port
    torch.manual_seed(0)
    net = torch_port.PortBilinearNet(a.users, a.items, a.dim)
    opt = torch.optim.Adagrad(net.parameters(), lr=a.lr)
    rs = np.random.RandomState(0)

    def fit_steps(users, items, nsteps):
        torch_port.fit_steps(net, opt, users, items, a.items, a.batch, a.loss, rs, max_steps=nsteps)
    return fit_steps


def run_cpu_port(a, steps, warmup):
    """interactions/s of the reference's CPU fit() loop on this box's host cores.

    kind "reference": the unmodified reference from oracle/_ref (stock code path, its own
    shuffle, sampler, autograd and the same Adagrad optimizer handed in through its
    `optimizer_func`); kind "port": oracle/torch_port.py, the same loop restated on stock
    torch CPU ops, when the install is absent.
    "All the host threads it can use": ATen's embedding backward / optimizer kernels stop
    scaling (and regress) well before 100+ threads, so one step is timed at a few thread
    counts and the fastest setting is used for the run.
    """
    import torch
    ncpu = os.cpu_count() or 1
    fit_steps, kind = _reference_runner(a), 'reference'
    if fit_steps is None:
        fit_steps, kind = _port_runner(a), 'port'
    rs = np.random.RandomState(0)
    B = a.batch
    cands = sorted({min(ncpu, c) for c in (8, 16, 32, 64, ncpu)})
    n = (steps + warmup + len(cands)) * B
    users = rs.randint(0, a.users, n).astype(np.int64)
    items = rs.randint(0, a.items, n).astype(np.int64)
    torch.set_num_threads(cands[-1])
    lo = warmup * B
    fit_steps(users[:lo], items[:lo], warmup)
    best, best_t = cands[-1], None
    for c in cands:
        torch.set_num_threads(c)
        t0 = time.perf_counter()
        fit_steps(users[lo:lo + B], items[lo:lo + B], 1)
        dt = time.perf_counter() - t0
        lo += B
        if best_t is None or dt < best_t:
            best, best_t = c, dt
    torch.set_num_threads(best)
    t0 = time.perf_counter()
    fit_steps(users[lo:], items[lo:], steps)
    dt = time.perf_counter() - t0
    what = ('unmodified reference (oracle/_ref: spotlight.factorization.implicit.'
            'ImplicitFactorizationModel.fit, use_cuda=False)' if kind == 'reference'
            else 'reference loop restated on torch CPU ops (oracle/torch_port.py)')
    return {'value': steps * B / dt, 'unit': UNIT, 'cores': best, 'kind': kind,
            'sample': '%d steps of batch %d after %d warm-up, torch %s CPU with %d of %d host '
                      'threads (fastest of %s), Adagrad dense, %s'
                      % (steps, B, warmup, torch.__version__, best, ncpu, cands, what),
            'ms_per_step': dt / steps * 1e3}


def main_reference(a):
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    # each reference step is O(table + batch): about a second at the default batch on host cores
    steps, warm = max(1, a.steps), max(1, a.warmup)
    r = run_cpu_port(a, steps, warm)
    line = {'impl': 'reference', 'metric': METRIC, 'value': r['value'], 'unit': UNIT,
            'n_gpus': a.gpus, 'steps': steps, 'warmup': warm, 'ms_per_step': r['ms_per_step'],
            'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f32',
            'data': 'synthetic', 'config': workload_config(a, a.gpus),
            'cpu_baseline': {k: r[k] for k in ('value', 'unit', 'cores', 'kind', 'sample')},
            'e2e': {'value': r['value'], 'unit': UNIT, 'h2d_bytes_per_step': 0,
                    'd2h_bytes_per_step': 0},
            'gpu_launches': 0}
    print(json.dumps(line))


# --------------------------------------------------------------------------
# our arm
# --------------------------------------------------------------------------

class _Shape(object):
    def __init__(self, num_users, num_items):
        self.num_users, self.num_items = num_users, num_items


def build_model(a, device_index):
    import torch
    from spotlight_b200 import optim
    from spotlight_b200.factorization.implicit import ImplicitFactorizationModel
    torch.cuda.set_device(device_index)
    model = ImplicitFactorizationModel(loss=a.loss, embedding_dim=a.dim, batch_size=a.batch,
                                       n_iter=1, optimizer_func=optim.fused_adagrad(lr=a.lr),
                                       use_cuda=True, random_state=np.random.RandomState(42))
    model._initialize(_Shape(a.users, a.items))
    assert model._route() == 'epoch'
    return model


DUMP_ROWS = 32768
DUMP_BYTES = 60 << 20       # sampled arrays; the .npy headers and epoch_loss stay well inside 64 MB


def dump_rows(dim):
    """Rows sampled per table: DUMP_ROWS, fewer when the two embedding tables and two bias tables,
    each with its Adagrad sum (16 * (dim + 1) bytes a sampled row), would exceed DUMP_BYTES."""
    return max(1, min(DUMP_ROWS, DUMP_BYTES // (16 * (dim + 1))))


def dump_outputs(model, epoch_loss, out_dir):
    """Write what the timed epoch hands its caller, taken right after its last step (the e2e and
    per-kernel legs that follow keep training the same model): the epoch loss it returns and the
    trained tables with their Adagrad sums.  A table of more than R = dump_rows(dim) rows is sampled
    at the rows np.random.RandomState(0).choice(rows, R, replace=False), sorted."""
    import torch
    net, opt = model._net, model._optimizer
    os.makedirs(out_dir, exist_ok=True)
    out = {'epoch_loss': np.array([epoch_loss], dtype=np.float64)}
    R = dump_rows(net.user_embeddings.weight.shape[1])
    for name in ('user_embeddings', 'item_embeddings', 'user_biases', 'item_biases'):
        w = getattr(net, name).weight
        n = w.shape[0]
        rows = np.sort(np.random.RandomState(0).choice(n, min(n, R), replace=False))
        idx = torch.from_numpy(rows).to(w.device)
        out[name] = w.detach().index_select(0, idx).float().cpu().numpy()
        out[name + '_adagrad_sum'] = opt.fused_state(w).index_select(0, idx).float().cpu().numpy()
    for name, arr in out.items():
        np.save(os.path.join(out_dir, name + '.npy'), arr)


def kernel_breakdown(model, users, items, a, steps):
    """Per-kernel average duration (ms) with CUDA events around single-kernel launches."""
    import ctypes
    import torch
    from spotlight_b200 import _lib, ops
    from spotlight_b200.sampling import sample_items
    lib = _lib.load()
    net, opt = model._net, model._optimizer
    dev = users.device
    B = a.batch
    Wu, Wi = net.user_embeddings.weight, net.item_embeddings.weight
    bu, bi = net.user_biases.weight, net.item_biases.weight
    negs = sample_items(a.items, steps * B, random_state=np.random.RandomState(1), device=dev)
    from spotlight_b200.factorization import implicit as _impl
    fused_need = lib.slb_mf_fused_workspace_bytes(B, a.users, a.items, a.dim) if _impl.PLANNED_STEP else 0
    if fused_need:      # planned step: integer plan, user kernel (forward + dU + update), item kernel
        names, bits = ['plan', 'mf_user', 'mf_item'], [1, 2, 4]
    else:
        names, bits = ['mf_fwd', 'seg_scan', 'mf_fill', 'mf_bwd', 'mf_apply'], [1, 2, 4, 8, 16]
    tot = dict.fromkeys(names, 0.0)
    with torch.no_grad():
        st = ops.mf_step_args(Wu, Wi, bu, bi, users[:B], items[:B], negs[:B], a.loss, 1, batch=B)
        st.grad_mode = _lib.GRAD_COMPACT
        bufs = dict(loss=torch.empty(1, device=dev))
        if fused_need:
            bufs['fws'] = ops.workspace('mfv2_%d_%d_%d' % (a.users, a.items, a.dim), fused_need, dev)
            st.fused_workspace, st.fused_workspace_bytes = bufs['fws'].data_ptr(), bufs['fws'].numel()
        else:
            rows = lib.slb_mf_compact_rows(B, 1, st.loss, 0)
            bufs.update(urows=torch.empty(rows, dtype=torch.int64, device=dev),
                        irows=torch.empty(rows, dtype=torch.int64, device=dev),
                        gWu=torch.empty((rows, a.dim), device=dev), gWi=torch.empty((rows, a.dim), device=dev),
                        gbu=torch.empty(rows, device=dev), gbi=torch.empty(rows, device=dev),
                        counts=torch.zeros(2, dtype=torch.int32, device=dev))
            st.urows, st.gWu, st.gbu = bufs['urows'].data_ptr(), bufs['gWu'].data_ptr(), bufs['gbu'].data_ptr()
            st.irows, st.gWi, st.gbi = bufs['irows'].data_ptr(), bufs['gWi'].data_ptr(), bufs['gbi'].data_ptr()
            st.compact_counts = bufs['counts'].data_ptr()
        st.loss_out = bufs['loss'].data_ptr()
        hp = opt.fused_hparams()
        st.opt, st.lr, st.weight_decay, st.eps = opt.fused_kind, hp['lr'], hp['weight_decay'], hp['eps']
        states = [opt.fused_state(p) for p in (Wu, Wi, bu, bi)]
        st.state_Wu, st.state_Wi, st.state_bu, st.state_bi = [s.data_ptr() for s in states]
        need = lib.slb_mf_step_workspace_bytes(B, 1, st.loss, a.users, a.items)
        ws = ops.workspace('mf%d_%d' % (a.users, a.items), need, dev)
        st.workspace, st.workspace_bytes = ws.data_ptr(), ws.numel()
        evs = [torch.cuda.Event(enable_timing=True) for _ in range(len(names) + 1)]
        stream = ops._stream()
        for k in range(steps):
            st.users = users[k * B:].data_ptr()
            st.items = items[k * B:].data_ptr()
            st.negs = negs[k * B:].data_ptr()
            evs[0].record()
            for i, bit in enumerate(bits):
                _lib.check(lib.slb_mf_train_step_phases(ctypes.byref(st), bit, stream), 'phase')
                evs[i + 1].record()
            torch.cuda.synchronize()
            for i, nm in enumerate(names):
                tot[nm] += evs[i].elapsed_time(evs[i + 1])
    return {nm: tot[nm] / steps for nm in names}


def sharded_e2e(a, rank, world, dev):
    """fit() through the public multi-GPU API on host ids; returns the e2e object."""
    import torch
    import torch.distributed as dist
    from spotlight_b200.interactions import Interactions
    from spotlight_b200.sharded import ShardedImplicitFactorizationModel
    B, K = a.batch, a.steps
    n_all = world * K * B                    # weak scaling: K global minibatches of world * B
    rs = np.random.RandomState(7)            # every rank holds the same global data set
    pin_u = torch.empty(n_all, dtype=torch.int32).pin_memory()
    pin_i = torch.empty(n_all, dtype=torch.int32).pin_memory()
    hu, hi = pin_u.numpy(), pin_i.numpy()
    hu[:] = rs.randint(0, a.users, n_all)
    hi[:] = rs.randint(0, a.items, n_all)
    inter = Interactions(hu, hi, num_users=a.users, num_items=a.items)
    fm = ShardedImplicitFactorizationModel(a.users, a.items, rank, world, dev, loss=a.loss,
                                           embedding_dim=a.dim, n_iter=1, batch_size=world * B,
                                           learning_rate=a.lr, random_state=np.random.RandomState(5),
                                           exchange=a.exchange)
    calls = []
    for _ in range(2):                       # first call warms the allocator (reported too)
        dist.barrier()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        fm.fit(inter)
        torch.cuda.synchronize()
        t = torch.tensor([time.perf_counter() - t0], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        calls.append(n_all / float(t.item()))
    e2e = {'value': calls[1], 'unit': UNIT, 'first_call_value': calls[0],
           'h2d_bytes_per_step': 8 * B, 'd2h_bytes_per_step': 4,      # per rank: 1/world of the global minibatch's two int32 ids
           'note': 'ShardedImplicitFactorizationModel.fit(Interactions) on every rank with the same '
                   'page-locked host int32 ids: H2D of 1/world of the ids per rank + NVLink all-gather, '
                   'range check, the global bit-exact RandomState.shuffle permutation and the global '
                   'negative stream computed on every rank (single-process minibatch membership), owner '
                   'routing, K sharded steps of global batch world*B, loss read-back; wall clock, max '
                   'over ranks, second of two calls'}
    return e2e


def main_sharded(a, rank, world, local):
    """N > 1: item rows range-sharded over the ranks, users owner-routed, NCCL exchange
    (spotlight_b200/sharded.py).  Weak scaling: the global minibatch is world * batch.

    `value` times ShardedImplicitFactorizationModel's own epoch loop on device-resident
    (already shuffled) GLOBAL ids -- the global negative stream (device MT19937, chunked on a
    side stream), the owner partition of every minibatch, the item-row exchange, the fused
    local step and the owners' updates are all inside the timed region.
    """
    import torch
    import torch.distributed as dist
    from spotlight_b200.sharded import ShardedImplicitFactorizationModel
    torch.cuda.set_device(local)
    dev = torch.device('cuda', local)
    dist.init_process_group('nccl', device_id=dev)
    sampler = ClockSampler(local).start() if rank == 0 else None
    B, K, W = a.batch, a.steps, a.warmup
    gB = world * B
    fm = ShardedImplicitFactorizationModel(a.users, a.items, rank, world, dev, loss=a.loss,
                                           embedding_dim=a.dim, n_iter=1, batch_size=gB,
                                           learning_rate=a.lr, random_state=np.random.RandomState(5),
                                           exchange=a.exchange)
    g = torch.Generator(device=dev).manual_seed(1234)           # same global ids on every rank
    n = (K + W) * gB
    users = torch.randint(0, a.users, (n,), device=dev, generator=g)
    items = torch.randint(0, a.items, (n,), device=dev, generator=g)
    chk = torch.stack([users.sum(), items.sum()]).double()
    lo_, hi_ = chk.clone(), chk.clone()
    dist.all_reduce(lo_, op=dist.ReduceOp.MIN)
    dist.all_reduce(hi_, op=dist.ReduceOp.MAX)
    assert torch.equal(lo_, hi_), 'ranks generated different global ids'

    fm._run_epoch_device(users[:W * gB], items[:W * gB])        # W warm-up steps, same code path
    # allocator priming (no training work): the timed epoch is K / W times longer than the warm-up,
    # so its epoch-sized temporaries (owner partition, negatives, sampler scratch) would each be a
    # fresh cudaMalloc inside the timed region; carve them from cached blocks instead -- one per
    # stream pool (main, sampler side stream)
    from spotlight_b200 import rng as _rng
    from spotlight_b200.factorization.implicit import _side_stream
    _prime = torch.empty(64 * K * gB, dtype=torch.uint8, device=dev)
    with torch.cuda.stream(_side_stream(dev)):
        _rng.reserve(a.items, K * gB, dev)
        _prime2 = torch.empty(16 * K * gB, dtype=torch.uint8, device=dev)
    del _prime, _prime2
    import gc
    gc.collect()
    gc.disable()            # no collector pause inside a 10-30 ms timed region (re-enabled right after)
    dist.barrier()
    torch.cuda.synchronize()
    if sampler:
        sampler.mark_begin()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    fm.mf.stats = {'rows_requested': 0, 'bytes_a2a': 0}
    e0.record()
    last = fm._run_epoch_device(users[W * gB:], items[W * gB:])  # exactly K global steps
    e1.record()
    dist.barrier()
    torch.cuda.synchronize()
    gc.enable()
    if sampler:
        sampler.mark_end()
    t = torch.tensor([e0.elapsed_time(e1)], device=dev, dtype=torch.float64)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t.item())
    clocks = sampler.stop() if sampler else None
    hw_nv = None
    if sampler:
        d = sampler.nvlink_delta_bytes()
        if d:
            hw_nv = dict(d, tx_gbs=d['tx_bytes'] / (ms * 1e-3) / 1e9, rx_gbs=d['rx_bytes'] / (ms * 1e-3) / 1e9,
                         note='counter window = the timed region (host marks around it)')

    # ---- end to end through the public multi-GPU API (host ids) ---------
    e2e = None
    stats = dict(fm.mf.stats)
    if not a.no_e2e:
        del users, items, fm
        torch.cuda.empty_cache()
        try:
            e2e = sharded_e2e(a, rank, world, dev)
        except Exception as exc:                 # keep the device-timed line even if the e2e leg fails
            e2e = {'value': None, 'unit': UNIT, 'error': repr(exc)[:300]}

    if rank == 0:
        cfg = workload_config(a, world)
        dense = a.exchange == 'dense' or (a.exchange == 'auto' and 2 * B >= a.items)
        cfg['parallelism'] = ('item rows range-sharded x%d, interactions routed to the user-owning rank, '
                              % world + ('whole-shard NCCL all-gather / reduce-scatter per step (2B >= '
                                         'num_items: every row is needed by every rank)' if dense else
                                         'NCCL all-to-all of requests / rows / gradient rows'))
        cfg['batch'] = gB
        cfg['batch_per_gpu'] = B
        cfg['negatives'] = ('one global device MT19937 stream (numpy-bit-exact), drawn inside the timed '
                            'region on every rank, chunked on a side stream')
        cfg['timed_region'] = ('ShardedImplicitFactorizationModel._run_epoch_device on device-resident '
                               'shuffled global ids: sampler + owner partition + exchange + steps')
        a2a_gb = stats['bytes_a2a'] / 1e9
        line = {'metric': METRIC, 'value': world * K * B / (ms * 1e-3), 'unit': UNIT,
                'n_gpus': world, 'steps': K, 'warmup': W, 'ms_per_step': ms / K,
                'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f32',
                'data': 'synthetic', 'config': cfg, 'epoch_loss': float(last), 'clocks': clocks,
                'e2e': e2e, 'gpu_launches': K * 20,
                'nvlink': {'exchange_gbytes_per_rank': a2a_gb,
                           'achieved_gbs_per_rank': a2a_gb / (ms * 1e-3),
                           'rows_requested_per_step': stats['rows_requested'] / K,
                           'source': 'bytes counted from the tensors handed to NCCL / timed region',
                           # the same window through the GPU's NVLink hardware counters (NVML field
                           # values NVLINK_THROUGHPUT_DATA_TX / RX of rank 0's GPU, all links)
                           'hw_counters': hw_nv,
                           'peak_gbs_per_direction': 900.0},
                'roofline': None, 'cpu_baseline': None}
        print(json.dumps(line))
    dist.destroy_process_group()


def main_ours(a):
    import torch
    import torch.distributed as dist
    rank = int(os.environ.get('RANK', '0'))
    world = int(os.environ.get('WORLD_SIZE', '1'))
    local = int(os.environ.get('LOCAL_RANK', '0'))
    if world > 1:
        return main_sharded(a, rank, world, local)
    sampler = ClockSampler(local).start() if rank == 0 else None      # long before the timed region
    model = build_model(a, local)
    dev = torch.device('cuda', local)
    B, K, W = a.batch, a.steps, a.warmup
    g = torch.Generator(device=dev).manual_seed(1234 + rank)
    n = (K + W) * B
    users = torch.randint(0, a.users, (n,), device=dev, generator=g)
    items = torch.randint(0, a.items, (n,), device=dev, generator=g)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- device-resident throughput ------------------------------------
    model._run_epoch_device(users[:W * B], items[:W * B])              # warm-up steps
    # allocator priming (no training work): the timed epoch's buffers come from the cache
    _prime = torch.empty(K * B, dtype=torch.int64, device=dev)
    from spotlight_b200 import rng as _rng
    from spotlight_b200.factorization.implicit import _side_stream
    with torch.cuda.stream(_side_stream(dev)):
        _rng.reserve(a.items, min(64, K) * B, dev)
    del _prime
    import gc
    gc.collect()
    gc.disable()            # no collector pause inside the timed region (re-enabled right after)
    barrier()
    if sampler:
        sampler.mark_begin()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    epoch_loss = model._run_epoch_device(users[W * B:], items[W * B:])  # exactly K steps
    e1.record()
    barrier()
    gc.enable()
    if sampler:
        sampler.mark_end()
    ms = e0.elapsed_time(e1)
    clocks = sampler.stop() if sampler else None
    t = torch.tensor([ms], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t.item())
    value = world * K * B / (ms * 1e-3)
    if a.dump_outputs:
        dump_outputs(model, epoch_loss, a.dump_outputs)

    # ---- end to end through the public API (host ids) -------------------
    e2e = None
    if not a.no_e2e:
        from spotlight_b200.interactions import Interactions
        rs = np.random.RandomState(7 + rank)
        # host ids live in page-locked memory (the contract's "pinned host memory"); the arrays
        # handed to Interactions are plain numpy views of it
        pin_u = torch.empty(K * B, dtype=torch.int32).pin_memory()
        pin_i = torch.empty(K * B, dtype=torch.int32).pin_memory()
        hu, hi = pin_u.numpy(), pin_i.numpy()
        hu[:] = rs.randint(0, a.users, K * B)
        hi[:] = rs.randint(0, a.items, K * B)
        inter = Interactions(hu, hi, num_users=a.users, num_items=a.items)
        calls = []
        for _ in range(2):                 # first call warms the allocator (its value is reported too)
            barrier()
            t0 = time.perf_counter()
            model.fit(inter)                                           # n_iter = 1 -> K steps
            torch.cuda.synchronize()
            dt = time.perf_counter() - t0
            t = torch.tensor([dt], device=dev, dtype=torch.float64)
            if world > 1:
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
            calls.append(world * K * B / float(t.item()))
        e2e = {'value': calls[1], 'unit': UNIT, 'first_call_value': calls[0],
               'h2d_bytes_per_step': 8 * B, 'd2h_bytes_per_step': 4,
               'note': 'ImplicitFactorizationModel.fit(Interactions) on host numpy int32 ids (page-locked), whole call '
                       'timed on the wall clock: H2D of both id arrays, id range check, bit-exact '
                       'RandomState.shuffle permutation on the device (csrc/shuffle.cu), id gather, device '
                       'negatives, K fused steps, D2H of the per-batch losses; second of two '
                       'consecutive fit() calls'}

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    # ---- per-kernel durations and roofline ------------------------------
    kb = kernel_breakdown(model, users, items, a, min(K, 50))
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, 'MEASURED_PEAKS.json')))
    except (OSError, ValueError):
        pass
    peak = float(peaks.get('hbm_gbs', 6650.0))
    R = 4 * a.dim
    if 'mf_user' in kb:     # planned step (DESIGN.md section 3): bytes / interaction, rows counted per use
        # mf_user: reads U, Q+, Q- rows + 3 biases + one 16-byte plan record; writes the updated U row + 2 g
        # mf_item: reads the 2 stashed user rows + 2 x (8-byte record + g); writes the 2 updated item rows
        alg = {'mf_user': 4 * R + 36, 'mf_item': 4 * R + 32}
        traffic_file = 'traffic_r02.json'
    else:
        alg = {'mf_fwd': 3 * R + 60, 'mf_bwd': 7 * R + 84}
        traffic_file = 'traffic_r01j.json'
    dom = max(alg, key=lambda k: kb[k])
    achieved = alg[dom] * B / (kb[dom] * 1e-3) / 1e9
    step_ms = sum(kb.values())
    traffic = None
    try:        # DRAM bytes of the dominant kernel from the committed ncu --set full capture
        tr = json.load(open(os.path.join(ROOT, 'profiles', traffic_file)))
        if tr['batch'] == B and tr['dim'] == a.dim:
            traffic = tr['dram_bytes_per_launch'].get(dom)
    except (OSError, ValueError, KeyError):
        pass
    step_bytes = (6 * R + 40) * B
    roofline = {'bound': 'hbm', 'kernel': dom, 'achieved': achieved, 'peak': peak, 'unit': 'GB/s',
                'frac': achieved / peak, 'traffic': traffic,
                'algorithmic_bytes_per_launch': alg[dom] * B,
                'peak_source': 'MEASURED_PEAKS.json hbm_gbs (measured copy)' if peaks else 'fallback 6650',
                'algorithmic_bytes_per_interaction': alg[dom],
                'kernel_ms': kb,
                'per_kernel_frac': {k: alg[k] * B / (kb[k] * 1e-3) / 1e9 / peak for k in alg},
                # SURVEY section 8(d)'s figure for the whole step (6R + 40 per interaction) against the
                # sum of the kernels timed one by one, and against the timed K-step region itself
                'step_algorithmic': {'bytes_per_interaction': 6 * R + 40,
                                     'achieved_gbs': step_bytes / (step_ms * 1e-3) / 1e9,
                                     'frac': step_bytes / (step_ms * 1e-3) / 1e9 / peak,
                                     'frac_of_timed_region': step_bytes / (ms / K * 1e-3) / 1e9 / peak}}

    cpu = None
    if not a.no_cpu_baseline and world == 1:
        r = run_cpu_port(a, a.cpu_steps, 2)
        cpu = {k: r[k] for k in ('value', 'unit', 'cores', 'kind', 'sample')}

    n_chunks = (K + 47) // 48                        # sampler chunks of up to 48 batches
    per_step = 10 if 'mf_user' in kb else 10         # planned: 6 plan + 2 user + 2 item; first generation: 10
    line = {'metric': METRIC, 'value': value, 'unit': UNIT, 'n_gpus': world, 'steps': K,
            'warmup': W, 'ms_per_step': ms / K, 'higher_is_better': True, 'scaling': 'weak',
            'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
            'config': workload_config(a, world), 'epoch_loss': epoch_loss,
            'clocks': clocks, 'e2e': e2e, 'gpu_launches': K * per_step + n_chunks * 6,     # kernels per step + sampler (jump round, fill, 4 compaction)
            'roofline': roofline, 'cpu_baseline': cpu}
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == '__main__':
    args = parse()
    if args.impl == 'reference':
        main_reference(args)
    else:
        main_ours(args)
