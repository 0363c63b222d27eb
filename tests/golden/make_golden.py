"""Generate golden vectors from the LIVE reference (build container only).

Run:  PYTHONDONTWRITEBYTECODE=1 python tests/golden/make_golden.py

Imports the unmodified reference from /root/reference (read-only), drives its
own modules / methods with fixed seeds, and stores inputs + outputs as small
``.npz`` fixtures next to this script.  The GPU box has no /root/reference; the
tests there read only the committed fixtures.

What is recorded (per case): the model ``state_dict``, the minibatch ids, the
RandomState key/pos before sampling, the negatives the reference drew, its
positive / negative predictions, the scalar loss, and every parameter's dense
``.grad`` after ``loss.backward()``.
"""

import contextlib
import io
import os
import sys

import numpy as np

sys.dont_write_bytecode = True
sys.path.insert(0, '/root/reference')

import torch  # noqa: E402

from spotlight.factorization.implicit import ImplicitFactorizationModel  # noqa: E402
from spotlight.factorization.representations import BilinearNet  # noqa: E402
from spotlight.interactions import Interactions, SequenceInteractions  # noqa: E402
from spotlight.layers import BloomEmbedding, ScaledEmbedding  # noqa: E402
from spotlight.sequence.implicit import ImplicitSequenceModel  # noqa: E402
from spotlight.sequence.representations import CNNNet, PoolNet  # noqa: E402

HERE = os.path.dirname(os.path.abspath(__file__))
torch.set_num_threads(1)


def _np(t):
    return t.detach().cpu().numpy().copy()


def _state(net):
    return {'sd.' + k: _np(v) for k, v in net.state_dict().items()}


def _grads(net):
    return {'grad.' + k: (_np(p.grad) if p.grad is not None else np.zeros(tuple(p.shape), np.float32))
            for k, p in net.named_parameters()}


def _rs_state(rs):
    st = rs.get_state()
    return {'rs_key': st[1].copy(), 'rs_pos': np.int64(st[2])}


def mf_case(name, loss, num_users, num_items, dim, batch, n_neg=5, seed=7,
            bloom=None, perturb_bias=True):
    rs = np.random.RandomState(seed)
    users = rs.randint(0, num_users, batch).astype(np.int64)
    items = rs.randint(0, num_items, batch).astype(np.int64)
    # force duplicates and boundary ids
    users[:4] = [0, num_users - 1, users[5], users[5]]
    items[:4] = [0, num_items - 1, items[6], items[6]]
    inter = Interactions(users.astype(np.int32), items.astype(np.int32),
                         num_users=num_users, num_items=num_items)
    model_rs = np.random.RandomState(seed + 1)
    rep = None
    if bloom is not None:
        ratio, H = bloom
        torch.manual_seed(seed)
        rep = BilinearNet(num_users, num_items, dim,
                          user_embedding_layer=ScaledEmbedding(num_users, dim),
                          item_embedding_layer=BloomEmbedding(num_items, dim,
                                                              compression_ratio=ratio,
                                                              num_hash_functions=H))
    model = ImplicitFactorizationModel(loss=loss, embedding_dim=dim, batch_size=batch,
                                       num_negative_samples=n_neg, representation=rep,
                                       random_state=model_rs)
    model._initialize(inter)
    net = model._net
    if perturb_bias:
        with torch.no_grad():   # zero-init biases would hide bias-gather bugs
            g = torch.Generator().manual_seed(seed)
            net.user_biases.weight.copy_(torch.randn(net.user_biases.weight.shape, generator=g) * 0.1)
            net.item_biases.weight.copy_(torch.randn(net.item_biases.weight.shape, generator=g) * 0.1)
    out = dict(_state(net))
    out.update(_rs_state(model._random_state))
    bu = torch.from_numpy(users)
    bi = torch.from_numpy(items)
    # replay of the reference loop body, spotlight/factorization/implicit.py:229-242
    rs_copy = np.random.RandomState()
    rs_copy.set_state(model._random_state.get_state())
    pos = model._net(bu, bi)
    if loss == 'adaptive_hinge':
        neg = model._get_multiple_negative_predictions(bu, n=n_neg)
        negs = rs_copy.randint(0, num_items, batch * n_neg, dtype=np.int64)
    else:
        neg = model._get_negative_prediction(bu)
        negs = rs_copy.randint(0, num_items, batch, dtype=np.int64)
    assert rs_copy.get_state()[2] == model._random_state.get_state()[2]
    model._optimizer.zero_grad()
    lv = model._loss_func(pos, neg)
    lv.backward()
    out.update(_grads(net))
    out.update(users=users, items=items, negs=negs, pos=_np(pos), neg=_np(neg),
               loss=np.float32(lv.item()), n_neg=np.int64(n_neg),
               num_users=np.int64(num_users), num_items=np.int64(num_items),
               dim=np.int64(dim))
    if bloom is not None:
        layer = net.item_embeddings
        out['bloom_rows_items'] = _np(layer._get_hashed_indices(bi.view(-1, 1)))
        out['bloom_ratio'] = np.float64(bloom[0])
        out['bloom_H'] = np.int64(bloom[1])
    np.savez_compressed(os.path.join(HERE, name + '.npz'), **out)
    print(name, 'loss', lv.item())


def seq_case(name, loss, representation, num_items, dim, batch, S, n_neg=3, seed=11,
             cnn_kwargs=None, bloom=None):
    rs = np.random.RandomState(seed)
    seqs = rs.randint(1, num_items, (batch, S)).astype(np.int64)
    for b in range(batch):                     # random left zero-pad
        pad = rs.randint(0, S)
        if b % 3 == 0:
            seqs[b, :pad] = 0
    seqs[1, :] = 0                             # one fully padded row
    seqs[2, -1] = num_items - 1
    inter = SequenceInteractions(seqs.astype(np.int32), num_items=num_items)
    torch.manual_seed(seed)
    emb = None
    if bloom is not None:
        emb = BloomEmbedding(num_items, dim, compression_ratio=bloom[0],
                             num_hash_functions=bloom[1], padding_idx=0)
    if representation == 'pooling':
        rep = PoolNet(num_items, dim, item_embedding_layer=emb)
    else:
        rep = CNNNet(num_items, dim, item_embedding_layer=emb, **(cnn_kwargs or {}))
    model = ImplicitSequenceModel(loss=loss, representation=rep, embedding_dim=dim,
                                  batch_size=batch, num_negative_samples=n_neg,
                                  random_state=np.random.RandomState(seed + 1))
    model._initialize(inter)
    net = model._net
    with torch.no_grad():
        g = torch.Generator().manual_seed(seed)
        net.item_biases.weight.copy_(torch.randn(net.item_biases.weight.shape, generator=g) * 0.1)
        net.item_biases.weight[0] = 0.0
    out = dict(_state(net))
    out.update(_rs_state(model._random_state))
    rs_copy = np.random.RandomState()
    rs_copy.set_state(model._random_state.get_state())
    sv = torch.from_numpy(seqs)
    # replay of spotlight/sequence/implicit.py:230-253
    user_rep, final = net.user_representation(sv)
    pos = net(user_rep, sv)
    if loss == 'adaptive_hinge':
        neg = model._get_multiple_negative_predictions(sv.size(), user_rep, n=n_neg)
        negs = rs_copy.randint(0, num_items, (n_neg * batch, S), dtype=np.int64)
    else:
        neg = model._get_negative_prediction(sv.size(), user_rep)
        negs = rs_copy.randint(0, num_items, (batch, S), dtype=np.int64)
    assert rs_copy.get_state()[2] == model._random_state.get_state()[2]
    model._optimizer.zero_grad()
    lv = model._loss_func(pos, neg, mask=(sv != 0))
    lv.backward()
    out.update(_grads(net))
    out.update(seqs=seqs, negs=negs, pos=_np(pos), neg=_np(neg), final=_np(final),
               user_rep=_np(user_rep),
               loss=np.float32(lv.item()), n_neg=np.int64(n_neg),
               num_items=np.int64(num_items), dim=np.int64(dim))
    if cnn_kwargs:
        for k, v in cnn_kwargs.items():
            out['cnn.' + k] = np.array(v)
    if bloom is not None:
        out['bloom_ratio'] = np.float64(bloom[0])
        out['bloom_H'] = np.int64(bloom[1])
    np.savez_compressed(os.path.join(HERE, name + '.npz'), **out)
    print(name, 'loss', lv.item())


def fit_case(name, loss, num_users, num_items, dim, n_inter, batch, n_iter, seed=3,
             optimizer='sgd', n_neg=3):
    """End-to-end: reference fit() with an order-independent optimizer."""
    rs = np.random.RandomState(seed)
    users = rs.randint(0, num_users, n_inter).astype(np.int32)
    items = rs.randint(0, num_items, n_inter).astype(np.int32)
    inter = Interactions(users, items, num_users=num_users, num_items=num_items)
    if optimizer == 'sgd':
        opt = lambda p: torch.optim.SGD(p, lr=0.5)            # noqa: E731
    elif optimizer == 'adagrad':
        opt = lambda p: torch.optim.Adagrad(p, lr=0.05)       # noqa: E731
    else:
        opt = None
    model = ImplicitFactorizationModel(loss=loss, embedding_dim=dim, batch_size=batch,
                                       n_iter=n_iter, optimizer_func=opt,
                                       num_negative_samples=n_neg,
                                       random_state=np.random.RandomState(seed))
    model._initialize(inter)
    out = {('init.' + k): _np(v) for k, v in model._net.state_dict().items()}
    buf = io.StringIO()
    with contextlib.redirect_stdout(buf):
        model.fit(inter, verbose=True)
    losses = [float(line.split('loss')[1]) for line in buf.getvalue().strip().split('\n')]
    out.update({('final.' + k): _np(v) for k, v in model._net.state_dict().items()})
    out.update(_rs_state(model._random_state))
    out.update(users=users, items=items, epoch_losses=np.array(losses),
               num_users=np.int64(num_users), num_items=np.int64(num_items),
               dim=np.int64(dim), batch=np.int64(batch), n_iter=np.int64(n_iter),
               seed=np.int64(seed), n_neg=np.int64(n_neg),
               predict_user3=model.predict(3))
    np.savez_compressed(os.path.join(HERE, name + '.npz'), **out)
    print(name, 'epoch losses', losses)


def seq_fit_case(name, loss, representation, num_items, dim, n_seq, S, batch, n_iter, seed=5):
    rs = np.random.RandomState(seed)
    seqs = rs.randint(1, num_items, (n_seq, S)).astype(np.int32)
    for b in range(0, n_seq, 2):
        seqs[b, :rs.randint(0, S)] = 0
    inter = SequenceInteractions(seqs, num_items=num_items)
    model = ImplicitSequenceModel(loss=loss, representation=representation,
                                  embedding_dim=dim, batch_size=batch, n_iter=n_iter,
                                  optimizer_func=lambda p: torch.optim.SGD(p, lr=0.5),
                                  random_state=np.random.RandomState(seed))
    model._initialize(inter)
    out = {('init.' + k): _np(v) for k, v in model._net.state_dict().items()}
    buf = io.StringIO()
    with contextlib.redirect_stdout(buf):
        model.fit(inter, verbose=True)
    losses = [float(line.split('loss')[1]) for line in buf.getvalue().strip().split('\n')]
    out.update({('final.' + k): _np(v) for k, v in model._net.state_dict().items()})
    out.update(_rs_state(model._random_state))
    out.update(seqs=seqs, epoch_losses=np.array(losses), num_items=np.int64(num_items),
               dim=np.int64(dim), batch=np.int64(batch), n_iter=np.int64(n_iter),
               seed=np.int64(seed), predict=model.predict(seqs[1]))
    np.savez_compressed(os.path.join(HERE, name + '.npz'), **out)
    print(name, 'epoch losses', losses)


def rng_case():
    """Stream-order fixture: ctor draw, shuffle, per-batch randint (A.1)."""
    rs = np.random.RandomState(42)
    ctor = rs.randint(-10**8, 10**8)
    idx = np.arange(1000)
    rs.shuffle(idx)
    negs = [rs.randint(0, n, sz, dtype=np.int64) for n, sz in
            [(100000, 257), (1683, 64), (1000000, 100), (50000000, 33), (1683, (5, 7))]]
    st = rs.get_state()
    np.savez_compressed(os.path.join(HERE, 'rng_stream.npz'), ctor=np.int64(ctor), shuffle=idx,
                        n0=negs[0], n1=negs[1], n2=negs[2], n3=negs[3], n4=negs[4],
                        end_key=st[1], end_pos=np.int64(st[2]))


def to_sequence_case():
    rs = np.random.RandomState(9)
    n = 400
    users = rs.randint(0, 23, n).astype(np.int32)
    items = rs.randint(1, 50, n).astype(np.int32)
    ts = rs.randint(0, 10000, n).astype(np.int32)
    inter = Interactions(users, items, timestamps=ts)
    out = dict(users=users, items=items, ts=ts)
    for tag, kw in [('a', dict(max_sequence_length=7)),
                    ('b', dict(max_sequence_length=5, step_size=1)),
                    ('c', dict(max_sequence_length=6, min_sequence_length=3, step_size=2))]:
        s = inter.to_sequence(**kw)
        out['seq_' + tag] = s.sequences
        out['uid_' + tag] = s.user_ids
    np.savez_compressed(os.path.join(HERE, 'to_sequence.npz'), **out)


def murmur_case():
    """sklearn.utils.murmurhash3_32, the hash the reference's BloomEmbedding calls
    (spotlight/layers.py:7,183), on the int32 edge values, a contiguous span and a seeded
    sample of the whole int32 range, for the seeds the tests use."""
    from sklearn.utils import murmurhash3_32
    rs = np.random.RandomState(11)
    keys = np.concatenate([np.arange(-5, 1000), [2**31 - 1, -2**31, 2**31 - 2, -2**31 + 1],
                           rs.randint(-2**31, 2**31 - 1, 4000, dtype=np.int64)]).astype(np.int32)
    seeds = np.array([0, 179424941, 179426549, 2**32 - 1], dtype=np.uint32)
    hashes = np.stack([murmurhash3_32(keys, seed=int(s)) for s in seeds]).astype(np.int32)
    np.savez_compressed(os.path.join(HERE, 'murmur_sklearn.npz'), keys=keys, seeds=seeds, hashes=hashes)


if __name__ == '__main__':
    rng_case()
    to_sequence_case()
    murmur_case()
    for loss in ('pointwise', 'bpr', 'hinge', 'adaptive_hinge'):
        mf_case('mf_' + loss, loss, num_users=97, num_items=53, dim=32, batch=192)
    mf_case('mf_bpr_d64', 'bpr', num_users=300, num_items=41, dim=64, batch=256)
    mf_case('mf_hinge_bloom', 'hinge', num_users=80, num_items=500, dim=16, batch=128,
            bloom=(0.2, 4))
    mf_case('mf_adaptive_bloom', 'adaptive_hinge', num_users=80, num_items=500, dim=16,
            batch=96, bloom=(0.5, 2), n_neg=4)
    for loss in ('pointwise', 'bpr', 'hinge', 'adaptive_hinge'):
        seq_case('pool_' + loss, loss, 'pooling', num_items=61, dim=16, batch=12, S=9)
    seq_case('pool_pointwise_bloom', 'pointwise', 'pooling', num_items=200, dim=16, batch=8,
             S=7, bloom=(0.3, 3))
    seq_case('cnn_pointwise', 'pointwise', 'cnn', num_items=61, dim=16, batch=10, S=9,
             cnn_kwargs=dict(kernel_width=3, dilation=1, num_layers=1))
    seq_case('cnn_bpr_l2_relu', 'bpr', 'cnn', num_items=61, dim=16, batch=10, S=11,
             cnn_kwargs=dict(kernel_width=3, dilation=(1, 2), num_layers=2, nonlinearity='relu'))
    # D = 128: the tcgen05 conv path of the product (csrc/seq_tc.cuh) against the live reference
    seq_case('cnn_pointwise_d128', 'pointwise', 'cnn', num_items=61, dim=128, batch=10, S=25,
             cnn_kwargs=dict(kernel_width=3, dilation=1, num_layers=1))
    seq_case('cnn_adaptive_k5_nores', 'adaptive_hinge', 'cnn', num_items=61, dim=16, batch=6,
             S=12, cnn_kwargs=dict(kernel_width=5, dilation=(2, 3), num_layers=2,
                                   residual_connections=False))
    fit_case('fit_bpr_sgd', 'bpr', 50, 40, 8, 300, 64, 2)
    fit_case('fit_adaptive_adagrad', 'adaptive_hinge', 50, 40, 8, 300, 64, 2, optimizer='adagrad')
    fit_case('fit_pointwise_adam', 'pointwise', 50, 40, 8, 300, 64, 2, optimizer='adam')
    seq_fit_case('fit_pool_hinge', 'hinge', 'pooling', 40, 8, 50, 6, 16, 2)
    seq_fit_case('fit_cnn_pointwise', 'pointwise', 'cnn', 40, 8, 50, 6, 16, 2)
