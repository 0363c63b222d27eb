"""Implicit-feedback factorization model with the reference's estimator API
(spotlight/factorization/implicit.py:22-311): same constructor arguments,
``fit(interactions, verbose)``, ``predict(user_ids, item_ids=None)``, private
attributes (``_net``, ``_optimizer``, ``_random_state``, ``_num_users``,
``_num_items``) and error behaviour.

What changed is where the ``fit`` loop body runs.  Three routes, chosen per
model, all producing the reference's losses and gradients:

``epoch pipeline``   BilinearNet with plain tables + a fused optimizer
                     (:mod:`spotlight_b200.optim`): the whole epoch -- negative
                     draw, fused forward kernel, deterministic gradient kernel,
                     row-wise optimizer -- is enqueued by one C call and the
                     host reads the per-batch losses once at the end.
``fused autograd``   BilinearNet with plain tables + any ``torch.optim``
                     optimizer (incl. the reference's default dense Adam): one
                     fused op per minibatch fills dense ``.grad``.
``generic``          custom ``representation`` / Bloom layers: the reference's
                     loop shape over this package's gather and loss ops.

There is no CPU route: ``use_cuda=False`` raises at ``fit``.
"""

import ctypes
import os

import numpy as np
import torch
import torch.optim as optim

from spotlight_b200 import _lib, ops
from spotlight_b200.factorization._components import _predict_process_ids
from spotlight_b200.factorization.representations import BilinearNet
from spotlight_b200.helpers import _repr_model
from spotlight_b200.losses import adaptive_hinge_loss, bpr_loss, hinge_loss, pointwise_loss
from spotlight_b200.rng import (SHUFFLE_DEVICE_MAX, permute_ids, shuffle_begin, shuffle_end,
                                shuffled_order_device)
from spotlight_b200.sampling import sample_items
from spotlight_b200.torch_utils import cpu, gpu, minibatch, set_seed, shuffled_order

_SIDE_STREAMS = {}


def _side_stream(device):
    """Per-device side stream for the sampler (module-level: models stay picklable)."""
    key = torch.device(device).index
    if key not in _SIDE_STREAMS:
        _SIDE_STREAMS[key] = torch.cuda.Stream(device=device, priority=-1)
    return _SIDE_STREAMS[key]


_PLAN_STREAMS = {}


def _plan_stream(device):
    """Per-device stream for the planned step's integer plan kernels (csrc/mf_v2.cuh).

    Normal priority, like the main stream: the plan has a whole step of float kernels to finish
    under, and at high priority its blocks are dispatched ahead of theirs and displace them
    (profiles/plan_overlap.py)."""
    key = torch.device(device).index
    if key not in _PLAN_STREAMS:
        _PLAN_STREAMS[key] = torch.cuda.Stream(device=device, priority=0)
    return _PLAN_STREAMS[key]


def _to_device_ids(ids, device):
    """Host id array -> int64 CUDA tensor (narrow on the wire, widened on the device)."""
    return _to_device_narrow(ids, device).long()


def _to_device_narrow(ids, device):
    """Host id array -> CUDA tensor in its own width (int32 stays int32 on the wire and in
    HBM; the permutation gather widens)."""
    arr = np.ascontiguousarray(ids)
    if arr.dtype not in (np.int32, np.int64):
        arr = arr.astype(np.int64)
    host = torch.from_numpy(arr)
    return host.to(device, non_blocking=host.is_pinned())     # page-locked callers get an async DMA


# route pointwise / bpr / hinge epochs through the planned two-kernel step (csrc/mf_v2.cuh);
# False selects the first-generation step (kept for A/B measurements and as the reference
# implementation of the compact-gradient mode)
PLANNED_STEP = True

# epochs at least this long take their permutation from the device shuffle (csrc/shuffle.cu);
# both paths are bit-exact with numpy, so the threshold is a speed knob only
DEVICE_SHUFFLE_MIN = 1 << 17

_NO_CPU = ('spotlight_b200 runs the fit() hot path in sm_100a CUDA kernels and has no CPU '
           'route; construct the model with use_cuda=True.')


class ImplicitFactorizationModel(object):
    """Implicit feedback matrix factorization trained by negative sampling.

    Parameters (identical to the reference, implicit.py:76-88)
    ----------
    loss: 'pointwise' | 'bpr' | 'hinge' | 'adaptive_hinge'
    embedding_dim, n_iter, batch_size, l2, learning_rate
    optimizer_func: callable(params) -> torch optimizer; default is the
        reference's dense ``Adam(weight_decay=l2, lr=learning_rate)``.  Pass
        :func:`spotlight_b200.optim.fused_adagrad` / ``fused_sgd`` for the
        on-device epoch pipeline.
    use_cuda: must be True to ``fit`` / ``predict``.
    representation: optional custom network module.
    sparse: use sparse gradients for embedding layers.
    random_state: ``numpy.random.RandomState`` driving shuffling and negative
        sampling (one MT19937 stream, consumed exactly as the reference does).
    num_negative_samples: negatives per positive for adaptive hinge.
    """

    def __init__(self, loss='pointwise', embedding_dim=32, n_iter=10, batch_size=256, l2=0.0,
                 learning_rate=1e-2, optimizer_func=None, use_cuda=False, representation=None,
                 sparse=False, random_state=None, num_negative_samples=5):

        assert loss in ('pointwise', 'bpr', 'hinge', 'adaptive_hinge')

        self._loss = loss
        self._embedding_dim = embedding_dim
        self._n_iter = n_iter
        self._learning_rate = learning_rate
        self._batch_size = batch_size
        self._l2 = l2
        self._use_cuda = use_cuda
        self._representation = representation
        self._sparse = sparse
        self._optimizer_func = optimizer_func
        self._random_state = random_state or np.random.RandomState()
        self._num_negative_samples = num_negative_samples

        self._num_users = None
        self._num_items = None
        self._net = None
        self._optimizer = None
        self._loss_func = None

        # same stream position as the reference (implicit.py:114)
        set_seed(self._random_state.randint(-10**8, 10**8), cuda=self._use_cuda)

    def __repr__(self):
        return _repr_model(self)

    @property
    def _initialized(self):
        return self._net is not None

    def _initialize(self, interactions):
        if not self._use_cuda:
            raise RuntimeError(_NO_CPU)
        (self._num_users, self._num_items) = (interactions.num_users, interactions.num_items)

        if self._representation is not None:
            self._net = gpu(self._representation, self._use_cuda)
        else:
            self._net = gpu(BilinearNet(self._num_users, self._num_items, self._embedding_dim,
                                        sparse=self._sparse), self._use_cuda)

        if self._optimizer_func is None:
            if isinstance(self._net, BilinearNet) and self._net.plain_tables() and not self._sparse:
                # the reference's default, optim.Adam(weight_decay=l2, lr) (implicit.py:143-148), as
                # the row-wise lazy-exact Adam: same trajectory, O(batch) instead of O(table) per step
                from spotlight_b200.optim import FusedAdam
                self._optimizer = FusedAdam(self._net.parameters(), weight_decay=self._l2,
                                            lr=self._learning_rate)
            else:
                self._optimizer = optim.Adam(self._net.parameters(), weight_decay=self._l2,
                                             lr=self._learning_rate)
        else:
            self._optimizer = self._optimizer_func(self._net.parameters())

        self._loss_func = {'pointwise': pointwise_loss, 'bpr': bpr_loss, 'hinge': hinge_loss,
                           'adaptive_hinge': adaptive_hinge_loss}[self._loss]

    def _check_input(self, user_ids, item_ids, allow_items_none=False):
        user_id_max = user_ids if isinstance(user_ids, int) else user_ids.max()
        if user_id_max >= self._num_users:
            raise ValueError('Maximum user id greater than number of users in model.')
        if allow_items_none and item_ids is None:
            return
        item_id_max = item_ids if isinstance(item_ids, int) else item_ids.max()
        if item_id_max >= self._num_items:
            raise ValueError('Maximum item id greater than number of items in model.')

    # ------------------------------------------------------------------ routes

    def _route(self):
        net = self._net
        fusable = isinstance(net, BilinearNet) and net.plain_tables()
        if fusable and getattr(self._optimizer, 'fused_kind', None) is not None:
            return 'epoch'
        if fusable and not self._sparse:
            return 'fused'
        if isinstance(net, BilinearNet) and not self._sparse and net.fused_spec() is not None:
            return 'bloom'
        return 'generic'

    def _n_neg(self):
        return self._num_negative_samples if self._loss == 'adaptive_hinge' else 1

    def _device(self):
        return next(self._net.parameters()).device

    def _epoch_negatives(self, n_interactions):
        """All of this epoch's negatives in one device draw.

        Consecutive ``randint`` calls consume the masked-rejection stream
        contiguously, so one draw of ``sum(B_k * n)`` values equals the
        reference's per-minibatch draws (implicit.py:256-259) concatenated.
        """
        return sample_items(self._num_items, n_interactions * self._n_neg(),
                            random_state=self._random_state, device=self._device())

    def fit(self, interactions, verbose=False):
        """Fit the model; repeated calls resume from the current weights and
        optimizer state (implicit.py:184-252)."""
        user_ids = interactions.user_ids
        item_ids = interactions.item_ids

        if not self._initialized:
            self._initialize(interactions)
        if not self._use_cuda:
            raise RuntimeError(_NO_CPU)

        route = self._route()
        device = self._device()
        n = len(user_ids)
        on_device = DEVICE_SHUFFLE_MIN <= n <= SHUFFLE_DEVICE_MAX and \
            self._random_state.get_state()[0] == 'MT19937'
        # the first epoch's permutation is resolved on the device while the ids travel
        main = torch.cuda.current_stream(device)
        pending = (shuffle_begin(n, self._random_state, device), main) if on_device and self._n_iter > 0 \
            else None
        # ids go to the device once per fit(); each epoch only the permutation is made
        # there (the reference re-uploads both shuffled id arrays, implicit.py:216-219)
        copy_stream = _side_stream(device)          # independent of the shuffle kernels just queued
        with torch.cuda.stream(copy_stream):
            users_dev = _to_device_narrow(user_ids, device)
            items_dev = _to_device_narrow(item_ids, device)
        torch.cuda.current_stream(device).wait_stream(copy_stream)
        users_dev.record_stream(torch.cuda.current_stream(device))
        items_dev.record_stream(torch.cuda.current_stream(device))
        if users_dev.dtype != items_dev.dtype:
            users_dev, items_dev = users_dev.long(), items_dev.long()
        # _check_input (implicit.py:166-181) on the resident copy: same errors, no host pass
        if n:
            umax, imax, umin, imin = torch.stack([users_dev.max(), items_dev.max(), users_dev.min(),
                                                  items_dev.min()]).tolist()        # one sync
            self._check_input(int(umax), int(imax))
            if umin < 0 or imin < 0:
                # the reference fails inside the embedding lookup (IndexError); same outcome,
                # raised before any kernel runs, on every route
                raise IndexError('index out of range in self: negative user or item id')

        for epoch_num in range(self._n_iter):
            # shuffle(): same stream consumption as random_state.shuffle(arange(n))
            # (torch_utils.py:46-47); the fancy-index gathers run on the device
            if pending is not None:
                handle, stream = pending
                with torch.cuda.stream(stream):           # any extra rounds go where it was begun
                    order_dev = shuffle_end(handle)
                if stream is not main:
                    main.wait_stream(stream)
                    order_dev.record_stream(main)
                pending = None
            elif on_device:
                order_dev = shuffled_order_device(n, self._random_state, device)
            else:                               # short epochs: the host loop beats the launches
                order = shuffled_order(n, self._random_state)
                order_dev = torch.from_numpy(order).to(device).long()
            user_ids_tensor, item_ids_tensor = permute_ids(order_dev, users_dev, items_dev)
            del order_dev

            if route == 'epoch':
                def next_permutation(last=epoch_num + 1 >= self._n_iter):
                    # the epoch's last negatives are drawn: the stream now stands where the next
                    # shuffle starts, and that shuffle can run under this epoch's remaining steps
                    nonlocal pending
                    if on_device and not last:
                        side = _side_stream(device)
                        with torch.cuda.stream(side):
                            pending = (shuffle_begin(n, self._random_state, device), side)
                epoch_loss = self._run_epoch_device(user_ids_tensor, item_ids_tensor,
                                                    after_sampling=next_permutation)
            elif route == 'bloom' and getattr(self._optimizer, 'fused_kind', None) in (_lib.OPT_SGD, _lib.OPT_ADAGRAD):
                negatives = self._epoch_negatives(len(user_ids))
                epoch_loss = self._fit_epoch_bloom_fused(user_ids_tensor, item_ids_tensor, negatives)
            else:
                negatives = self._epoch_negatives(len(user_ids))
                epoch_loss = self._fit_epoch_autograd(user_ids_tensor, item_ids_tensor, negatives,
                                                      fused=route)

            if verbose:
                print('Epoch {}: loss {}'.format(epoch_num, epoch_loss))

            if np.isnan(epoch_loss) or epoch_loss == 0.0:
                raise ValueError('Degenerate epoch loss: {}'.format(epoch_loss))
        if hasattr(self._optimizer, 'flush'):
            self._optimizer.flush()             # lazy-exact Adam: every row current before fit() returns

    def _run_epoch_device(self, users, items, chunk_batches=48, after_sampling=None):
        """The epoch pipeline over device-resident (already shuffled) ids.

        Negatives are drawn chunk by chunk on a side stream (the MT19937 block
        generator is a single-CTA kernel) while the main stream runs the
        previous chunk's training steps; the per-batch losses are read back
        once at the end.  Returns the epoch loss exactly as the reference
        defines it: the mean of the per-minibatch losses (implicit.py:240,245).
        """
        n, B, n_neg = users.numel(), int(self._batch_size), self._n_neg()
        dev = users.device
        main = torch.cuda.current_stream(dev)
        side = _side_stream(dev)
        chunk = max(1, int(chunk_batches)) * B

        # one buffer for the epoch's negatives (cached by the allocator across epochs);
        # sampler scratch sized once for the largest chunk (no cudaMalloc mid-epoch)
        negs_all = torch.empty(n * n_neg, dtype=torch.int64, device=dev)
        # the block just handed out may still be read by work queued on the main stream
        # (it was freed there); the sampler writes it on the side stream
        side.wait_stream(main)
        from spotlight_b200 import rng as _rng
        with torch.cuda.stream(side):
            _rng.reserve(self._num_items, min(chunk, n) * n_neg, dev)
            # the generator lives on the device for the whole epoch: the draws chain without
            # a host round trip and finish() hands the state back once (spotlight_b200/rng.py)
            stream = _rng.DeviceStream(self._random_state, dev)
        # All of the epoch's draws are enqueued first (side stream), in chunks of up to
        # `chunk_batches` minibatches, each followed by an event; then ONE C call enqueues every
        # training step, making its streams wait for the event of the chunk a step belongs to.
        # Nothing on the host waits in between.  A chunk costs one jump round + one block-fill
        # round whatever its size (up to the one-round reach of the jump table, ~31 M values), so
        # the first chunk is as large as the others: only ~0.1 ms more exposed than a one-batch
        # chunk, and the latency-bound generator never competes with the training kernels for a
        # short epoch.
        waits = []
        lo = 0
        with torch.cuda.stream(side):
            while lo < n:
                cur = min(chunk, n - lo)
                stream.draw(self._num_items, cur * n_neg, out=negs_all[lo * n_neg:(lo + cur) * n_neg])
                ev = torch.cuda.Event()
                ev.record(side)
                waits.append((lo // B, ev))
                lo += cur
        losses = self._fit_epoch_pipeline(users, items, negs_all, sync=False, waits=waits)
        with torch.cuda.stream(side):
            stream.finish()                     # waits for the sampler only: RandomState is final
        if after_sampling is not None:
            after_sampling()                    # next epoch's shuffle, under this epoch's training
        host = losses.cpu().numpy().astype(np.float64)                  # one sync per epoch
        ws = ops.workspace('mf%d_%d' % (self._num_users, self._num_items), 0, dev)
        if ops.workspace_error_flag(ws):
            raise ValueError('ids out of range reached the device kernels')
        return float(host.sum() / len(host))

    def _fit_epoch_pipeline(self, users, items, negatives, sync=True, waits=()):
        """One C call enqueues every minibatch step of ``users``/``items``; returns the
        device tensor of per-batch losses (``sync=False``) or their mean."""
        net, opt = self._net, self._optimizer
        lib = _lib.load()
        n, B, n_neg = users.numel(), int(self._batch_size), self._n_neg()
        Wu, Wi = net.user_embeddings.weight, net.item_embeddings.weight
        bu, bi = net.user_biases.weight, net.item_biases.weight
        dev = Wu.device
        with torch.no_grad():
            a = ops.mf_step_args(Wu, Wi, bu, bi, users, items, negatives, self._loss, n_neg,
                                 batch=min(B, n))
            a.grad_mode = _lib.GRAD_COMPACT
            # planned two-kernel step (plan + user kernel + item kernel, csrc/mf_v2.cuh) whenever the
            # library supports the shape; otherwise the first-generation step with compact gradients
            fused_need = 0
            if self._loss != 'adaptive_hinge' and PLANNED_STEP and opt.fused_kind != _lib.OPT_ADAM:
                fused_need = lib.slb_mf_fused_workspace_bytes(a.batch, a.num_users, a.num_items, a.dim)
            if fused_need:
                fws = ops.workspace('mfv2_%d_%d_%d' % (a.num_users, a.num_items, a.dim),
                                    fused_need, dev)
                a.fused_workspace, a.fused_workspace_bytes = fws.data_ptr(), fws.numel()
                if not os.environ.get('SLB_PLAN_SAME_STREAM'):      # A/B switch for measurements
                    a.plan_stream = _plan_stream(dev).cuda_stream
                keep = (fws,)
            else:
                rows = lib.slb_mf_compact_rows(a.batch, n_neg, a.loss, 0)
                D = a.dim
                urows = torch.empty(rows, dtype=torch.int64, device=dev)
                irows = torch.empty(rows, dtype=torch.int64, device=dev)
                gWu = torch.empty((rows, D), dtype=torch.float32, device=dev)
                gWi = torch.empty((rows, D), dtype=torch.float32, device=dev)
                gbu = torch.empty(rows, dtype=torch.float32, device=dev)
                gbi = torch.empty(rows, dtype=torch.float32, device=dev)
                counts = torch.zeros(2, dtype=torch.int32, device=dev)
                a.urows, a.gWu, a.gbu = urows.data_ptr(), gWu.data_ptr(), gbu.data_ptr()
                a.irows, a.gWi, a.gbi = irows.data_ptr(), gWi.data_ptr(), gbi.data_ptr()
                a.compact_counts = counts.data_ptr()
                keep = (urows, irows, gWu, gWi, gbu, gbi, counts)
            hp = opt.fused_hparams()
            a.opt, a.lr, a.weight_decay, a.eps = opt.fused_kind, hp['lr'], hp['weight_decay'], hp['eps']
            n_steps = (n + B - 1) // B
            if opt.fused_kind == _lib.OPT_ADAGRAD:
                states = [opt.fused_state(p) for p in (Wu, Wi, bu, bi)]
                a.state_Wu, a.state_Wi, a.state_bu, a.state_bi = [s.data_ptr() for s in states]
            elif opt.fused_kind == _lib.OPT_ADAM:
                states = [opt.fused_states(p) for p in (Wu, Wi, bu, bi)]
                a.state_Wu, a.state_Wi, a.state_bu, a.state_bi = [s[0].data_ptr() for s in states]
                a.state2_Wu, a.state2_Wi, a.state2_bu, a.state2_bi = [s[1].data_ptr() for s in states]
                a.last_u, a.last_i = states[0][2].data_ptr(), states[1][2].data_ptr()
                a.beta1, a.beta2 = hp['beta1'], hp['beta2']
                a.one_minus_beta1, a.one_minus_beta2 = 1.0 - hp['beta1'], 1.0 - hp['beta2']
                sched = opt.schedule(opt.steps_taken + n_steps, dev)
                a.adam_sched, a.adam_step = sched.data_ptr(), opt.steps_taken + 1
                opt.advance(n_steps)
            need = lib.slb_mf_step_workspace_bytes(a.batch, n_neg, a.loss, a.num_users, a.num_items)
            ws = ops.workspace('mf%d_%d' % (a.num_users, a.num_items), need, dev)
            a.workspace, a.workspace_bytes = ws.data_ptr(), ws.numel()
            n_steps = (n + B - 1) // B
            losses = torch.empty(n_steps, dtype=torch.float32, device=dev)
            # steps wait (on the device) for the event of the chunk of negatives they read
            w_steps = (ctypes.c_int64 * max(1, len(waits)))(*[int(k) for k, _ in waits])
            w_events = (ctypes.c_void_p * max(1, len(waits)))(*[ev.cuda_event for _, ev in waits])
            rc = lib.slb_mf_fit_epoch_events(ctypes.byref(a), ops._ptr(users), ops._ptr(items),
                                             ops._ptr(negatives), n, ops._ptr(losses), ops._stream(),
                                             w_steps, w_events, len(waits))
            _lib.check(rc, 'mf_fit_epoch')
            if not sync:
                return losses
            # the reference averages float(loss.item()) per batch (implicit.py:240,245)
            host = losses.cpu().numpy().astype(np.float64)
            if ops.workspace_error_flag(ws):
                raise ValueError('ids out of range reached the device kernels')
        return float(host.sum() / n_steps)

    def _fit_epoch_bloom_fused(self, users, items, negatives):
        """Hashed-table model with a fused row-wise optimizer: one in-place step per minibatch
        (csrc/mf.cu slb_mf_bloom_train_step, fused mode), no dense gradient of any table."""
        net, opt = self._net, self._optimizer
        spec = net.fused_spec()
        n_neg = self._n_neg()
        hp = opt.fused_hparams()
        params = (spec['Wu'], spec['Wi'], net.user_biases.weight, net.item_biases.weight)
        states = [opt.fused_state(p) for p in params] if opt.fused_kind == _lib.OPT_ADAGRAD else None
        losses = []
        lo = 0
        for batch_user, batch_item in minibatch(users, items, batch_size=self._batch_size):
            B = batch_user.numel()
            batch_neg = negatives[lo * n_neg:(lo + B) * n_neg]
            lo += B
            losses.append(ops.mf_bloom_train_step_inplace(
                *params, batch_user, batch_item, batch_neg, self._loss, n_neg, spec['user_seeds'],
                spec['item_seeds'], spec['user_pad'], spec['item_pad'], opt.fused_kind, hp['lr'], states,
                hp['weight_decay'], hp['eps']))
        host = torch.stack(losses).cpu().numpy().astype(np.float64)        # one sync per epoch
        return float(host.sum() / len(host))

    def _fit_epoch_autograd(self, users, items, negatives, fused):
        net = self._net
        n_neg = self._n_neg()
        epoch_loss = torch.zeros((), dtype=torch.float64, device=users.device)
        lo = 0
        minibatch_num = -1
        for minibatch_num, (batch_user, batch_item) in enumerate(
                minibatch(users, items, batch_size=self._batch_size)):
            B = batch_user.numel()
            batch_neg = negatives[lo * n_neg:(lo + B) * n_neg]
            lo += B
            self._optimizer.zero_grad()
            if fused == 'fused':
                loss = ops.fused_mf_loss(net.user_embeddings.weight, net.item_embeddings.weight,
                                         net.user_biases.weight, net.item_biases.weight,
                                         batch_user, batch_item, batch_neg, self._loss, n_neg)
            elif fused == 'bloom':
                spec = net.fused_spec()
                loss = ops.fused_bloom_loss(spec['Wu'], spec['Wi'], net.user_biases.weight,
                                            net.item_biases.weight, batch_user, batch_item, batch_neg,
                                            self._loss, n_neg, spec)
            else:
                positive_prediction = net(batch_user, batch_item)
                if self._loss == 'adaptive_hinge':
                    # reference quirk (implicit.py:266-275): users repeat [u0]*n,[u1]*n,..
                    # but the flat predictions are viewed as (n, B)
                    rep_users = batch_user.view(B, 1).expand(B, n_neg).reshape(B * n_neg)
                    negative_prediction = net(rep_users, batch_neg).view(n_neg, B)
                else:
                    negative_prediction = net(batch_user, batch_neg)
                loss = self._loss_func(positive_prediction, negative_prediction)
            epoch_loss += loss.detach().double()
            loss.backward()
            self._optimizer.step()
        return float(epoch_loss.item()) / (minibatch_num + 1)

    # reference-named helpers (implicit.py:254-275), kept for API parity
    def _get_negative_prediction(self, user_ids):
        negative_items = sample_items(self._num_items, len(user_ids),
                                      random_state=self._random_state, device=user_ids.device)
        return self._net(user_ids, negative_items)

    def _get_multiple_negative_predictions(self, user_ids, n=5):
        batch_size = user_ids.size(0)
        negative_prediction = self._get_negative_prediction(
            user_ids.view(batch_size, 1).expand(batch_size, n).reshape(batch_size * n))
        return negative_prediction.view(n, len(user_ids))

    def predict(self, user_ids, item_ids=None):
        """Scores for (user, item) pairs, or for one user against ``item_ids``
        (all items when None); returns a NumPy array (implicit.py:277-311)."""
        self._check_input(user_ids, item_ids, allow_items_none=True)
        self._net.train(False)
        user_ids, item_ids = _predict_process_ids(user_ids, item_ids, self._num_items,
                                                  self._use_cuda)
        with torch.no_grad():
            out = self._net(user_ids, item_ids)
        return cpu(out).detach().numpy().flatten()
