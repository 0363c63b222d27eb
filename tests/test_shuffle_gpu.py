"""Device epoch shuffle (csrc/shuffle.cu) against NumPy itself: same permutation as
``RandomState.shuffle(arange(n))`` (torch_utils.py:46-47) and the same generator state
afterwards, bit for bit."""

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu


def _same_state(a, b):
    sa, sb = a.get_state(), b.get_state()
    return sa[0] == sb[0] and np.array_equal(sa[1], sb[1]) and sa[2:] == sb[2:]


@pytest.mark.parametrize('n', [1, 2, 3, 5, 17, 624, 1000, 4097, 65539, 1 << 20, 3000001, (1 << 24) + 12345])
@pytest.mark.parametrize('seed', [0, 42])
def test_device_shuffle_matches_numpy(n, seed):
    from spotlight_b200.rng import shuffled_order_device
    ours, ref = np.random.RandomState(seed), np.random.RandomState(seed)
    ours.randint(0, 1000, 777)                      # start mid-block, like a second epoch does
    ref.randint(0, 1000, 777)
    got = shuffled_order_device(n, ours, 'cuda:0')
    want = np.arange(n)
    ref.shuffle(want)
    assert got.dtype == torch.int64 and got.shape == (n,)
    assert np.array_equal(got.cpu().numpy(), want)
    assert _same_state(ours, ref)
    # the stream continues seamlessly (the next epoch's negatives come from it)
    assert np.array_equal(ours.randint(0, 10 ** 6, 50), ref.randint(0, 10 ** 6, 50))


def test_device_shuffle_few_rounds_resumes():
    """rounds=1 forces the resume path: the result must not depend on how the global
    fixed-point rounds are batched."""
    from spotlight_b200.rng import shuffled_order_device
    n = 300000
    ours, ref = np.random.RandomState(5), np.random.RandomState(5)
    got = shuffled_order_device(n, ours, 'cuda:0', rounds=1)
    want = np.arange(n)
    ref.shuffle(want)
    assert np.array_equal(got.cpu().numpy(), want)
    assert _same_state(ours, ref)


def test_fit_uses_device_shuffle_and_matches_host_path(monkeypatch):
    """model.fit with the device permutation = model.fit with the host one."""
    from spotlight_b200.factorization import implicit
    from spotlight_b200.interactions import Interactions
    from spotlight_b200.optim import fused_adagrad
    rs = np.random.RandomState(3)
    inter = Interactions(rs.randint(0, 500, 40000).astype(np.int32), rs.randint(0, 300, 40000).astype(np.int32),
                         num_users=500, num_items=300)

    def run(min_n):
        monkeypatch.setattr(implicit, 'DEVICE_SHUFFLE_MIN', min_n)
        m = implicit.ImplicitFactorizationModel(loss='bpr', embedding_dim=16, n_iter=2, batch_size=4096,
                                                use_cuda=True, random_state=np.random.RandomState(11),
                                                optimizer_func=fused_adagrad(lr=0.05))
        m.fit(inter)
        return m._net.item_embeddings.weight.detach().cpu().numpy().copy()

    assert np.array_equal(run(1), run(1 << 62))


@pytest.mark.parametrize('dtype', [np.int32, np.int64])
def test_permute_ids(dtype):
    from spotlight_b200.rng import permute_ids
    rs = np.random.RandomState(0)
    n = 100003
    u, it = rs.randint(0, 10 ** 6, n).astype(dtype), rs.randint(0, 10 ** 5, n).astype(dtype)
    order = rs.permutation(n)
    gu, gi = permute_ids(torch.from_numpy(order).cuda(), torch.from_numpy(u).cuda(), torch.from_numpy(it).cuda())
    assert gu.dtype == torch.int64
    assert np.array_equal(gu.cpu().numpy(), u[order]) and np.array_equal(gi.cpu().numpy(), it[order])
    only = permute_ids(torch.from_numpy(order).cuda(), torch.from_numpy(u).cuda())
    assert np.array_equal(only.cpu().numpy(), u[order])


def test_fit_rejects_out_of_range_ids():
    from spotlight_b200.factorization.implicit import ImplicitFactorizationModel
    from spotlight_b200.interactions import Interactions
    inter = Interactions(np.array([0, 1, 2], dtype=np.int32), np.array([0, 1, 2], dtype=np.int32),
                         num_users=3, num_items=3)
    m = ImplicitFactorizationModel(n_iter=1, use_cuda=True, embedding_dim=8)
    m.fit(inter)
    bad = Interactions(np.array([0, 1, 5], dtype=np.int32), np.array([0, 1, 2], dtype=np.int32),
                       num_users=6, num_items=3)
    with pytest.raises(ValueError, match='Maximum user id'):
        m.fit(bad)
