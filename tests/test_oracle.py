"""Pin the oracle (oracle/*.py) against the live reference's golden vectors,
NumPy's RandomState and sklearn's murmurhash3_32 (recorded).  CPU only."""

import numpy as np
import pytest

from conftest import assert_close, load_golden
from oracle import mf as omf
from oracle import seq as oseq
from oracle.mt19937 import MT19937, jump, temper, twist, untemper
from oracle.murmur import bloom_rows, murmurhash3_32

MF_CASES = ['mf_pointwise', 'mf_bpr', 'mf_hinge', 'mf_adaptive_hinge', 'mf_bpr_d64']
LOSS_OF = lambda name: name.split('_', 1)[1].replace('_d64', '')  # noqa: E731


def test_rng_matches_numpy_randomstate():
    rs = np.random.RandomState(42)
    m = MT19937(42)
    st = rs.get_state()
    assert (st[1] == m.key).all() and st[2] == m.pos
    assert rs.randint(-10**8, 10**8) == int(m.randint(-10**8, 10**8, ()))
    idx = np.arange(2000)
    rs.shuffle(idx)
    assert (idx == m.shuffle_indices(2000)).all()
    for n, sz in [(100000, 70000), (1683, (5, 77)), (1000000, 1234), (50000000, 999),
                  (1, 5), (2, 7), (4096, 3000), (4097, 3000)]:
        assert (rs.randint(0, n, sz, dtype=np.int64) == m.randint(0, n, sz)).all(), n
    st = rs.get_state()
    assert (st[1] == m.key).all() and st[2] == m.pos


def test_rng_golden_stream():
    g = load_golden('rng_stream')
    m = MT19937(42)
    assert int(m.randint(-10**8, 10**8, ())) == int(g['ctor'])
    assert (m.shuffle_indices(1000) == g['shuffle']).all()
    for key, (n, sz) in zip(['n0', 'n1', 'n2', 'n3', 'n4'],
                            [(100000, 257), (1683, 64), (1000000, 100), (50000000, 33),
                             (1683, (5, 7))]):
        assert (m.randint(0, n, sz) == g[key]).all()
    assert (m.key == g['end_key']).all() and m.pos == int(g['end_pos'])


def test_untemper_roundtrip():
    w = np.random.RandomState(1).randint(0, 2**32, 5000, dtype=np.uint64).astype(np.uint32)
    assert (untemper(temper(w)) == w).all()


def test_jump_table_matches_sequential_twists():
    """spotlight_b200/data/mt19937_jump.npy: row k jumps 2^k blocks (checked against
    repeated twists for the reduced polynomials k = 5, 6, 9)."""
    import os
    from conftest import ROOT
    tab = np.load(os.path.join(ROOT, 'spotlight_b200', 'data', 'mt19937_jump.npy'))
    assert tab.shape == (27, 624)
    key = np.random.RandomState(7).get_state()[1]
    for k in (0, 5, 6, 9):
        j = jump(key, tab[k])
        ref = key.copy()
        for _ in range(2 ** k):
            ref = twist(ref)
        # the 31 low bits of word 0 are not part of the MT19937 state
        assert (j[1:] == ref[1:]).all() and ((int(j[0]) ^ int(ref[0])) & 0x80000000) == 0


def test_murmur_matches_sklearn():
    """Against sklearn.utils.murmurhash3_32 (the reference's BloomEmbedding hash) as recorded in
    tests/golden/murmur_sklearn.npz, and against the live function too where sklearn is installed."""
    g = load_golden('murmur_sklearn')
    for s, want in zip(g['seeds'], g['hashes']):
        assert (murmurhash3_32(g['keys'], int(s)) == want).all(), int(s)
    try:
        from sklearn.utils import murmurhash3_32 as sk
    except ImportError:
        return
    k = np.concatenate([np.arange(-5, 20000), [2**31 - 1, -2**31]]).astype(np.int32)
    for s in (0, 179424941, 179426549, 2**32 - 1):
        assert (sk(k, seed=s) == murmurhash3_32(k, s)).all()


@pytest.mark.parametrize('name', ['mf_hinge_bloom', 'mf_adaptive_bloom'])
def test_bloom_rows_golden(name):
    g = load_golden(name)
    M = g['sd.item_embeddings.embeddings.weight'].shape[0]
    rows = bloom_rows(g['items'], int(g['bloom_H']), M)
    assert (rows == g['bloom_rows_items']).all()


@pytest.mark.parametrize('name', MF_CASES)
def test_mf_step_golden(name):
    g = load_golden(name)
    loss = LOSS_OF(name)
    for dtype, tol in ((np.float32, 2e-6), (np.float64, 1e-6)):
        r = omf.mf_step(g['sd.user_embeddings.weight'], g['sd.item_embeddings.weight'],
                        g['sd.user_biases.weight'], g['sd.item_biases.weight'],
                        g['users'], g['items'], g['negs'], loss, int(g['n_neg']), dtype)
        assert_close(r['pos'], g['pos'], tol, what='pos')
        assert_close(r['neg'], g['neg'], tol, what='neg')
        assert_close(r['loss'], g['loss'], tol, what='loss')
        assert_close(r['dWu'], g['grad.user_embeddings.weight'], 1e-5, what='dWu')
        assert_close(r['dWi'], g['grad.item_embeddings.weight'], 1e-5, what='dWi')
        assert_close(r['dbu'], g['grad.user_biases.weight'], 1e-5, atol=1e-7, what='dbu')
        assert_close(r['dbi'], g['grad.item_biases.weight'], 1e-5, what='dbi')


def test_negatives_reproduce_from_saved_state():
    g = load_golden('mf_adaptive_hinge')
    m = MT19937(state=(g['rs_key'], int(g['rs_pos'])))
    negs = m.randint(0, int(g['num_items']), len(g['users']) * int(g['n_neg']))
    assert (negs == g['negs']).all()


@pytest.mark.parametrize('name', ['pool_pointwise', 'pool_bpr', 'pool_hinge',
                                  'pool_adaptive_hinge'])
def test_pool_step_golden(name):
    g = load_golden(name)
    loss = name.split('_', 1)[1]
    r = oseq.pool_step(g['sd.item_embeddings.weight'], g['sd.item_biases.weight'],
                       g['seqs'], g['negs'], loss, int(g['n_neg']), np.float64)
    assert_close(r['pos'], g['pos'], 2e-6, what='pos')
    assert_close(r['neg'], g['neg'], 2e-6, what='neg')
    assert_close(r['loss'], g['loss'], 2e-6, what='loss')
    assert_close(r['final'], g['final'], 2e-6, what='final')
    assert_close(r['dE'], g['grad.item_embeddings.weight'], 1e-5, what='dE')
    assert_close(r['dbias'], g['grad.item_biases.weight'], 1e-5, what='dbias')
    assert np.all(r['dE'][0] == 0) and np.all(r['dbias'][0] == 0)


@pytest.mark.parametrize('name', ['cnn_pointwise', 'cnn_bpr_l2_relu', 'cnn_adaptive_k5_nores'])
def test_cnn_step_golden(name):
    g = load_golden(name)
    loss = {'cnn_pointwise': 'pointwise', 'cnn_bpr_l2_relu': 'bpr',
            'cnn_adaptive_k5_nores': 'adaptive_hinge'}[name]
    L = int(g['cnn.num_layers'])
    kw = np.atleast_1d(g['cnn.kernel_width'])
    dl = np.atleast_1d(g['cnn.dilation'])
    kw = [int(kw[i % len(kw)]) for i in range(L)]
    dl = [int(dl[i % len(dl)]) for i in range(L)]
    nonlin = str(g['cnn.nonlinearity']) if 'cnn.nonlinearity' in g else 'tanh'
    res = bool(g['cnn.residual_connections']) if 'cnn.residual_connections' in g else True
    convs = [(g['sd.cnn_%d.weight' % i], g['sd.cnn_%d.bias' % i]) for i in range(L)]
    r = oseq.cnn_step(g['sd.item_embeddings.weight'], g['sd.item_biases.weight'], convs,
                      g['seqs'], g['negs'], kw, dl, loss, int(g['n_neg']), nonlin, res,
                      np.float64)
    assert_close(r['pos'], g['pos'], 3e-6, what='pos')
    assert_close(r['neg'], g['neg'], 3e-6, what='neg')
    assert_close(r['loss'], g['loss'], 3e-6, what='loss')
    assert_close(r['final'], g['final'], 3e-6, what='final')
    assert_close(r['dE'], g['grad.item_embeddings.weight'], 1e-5, what='dE')
    assert_close(r['dbias'], g['grad.item_biases.weight'], 1e-5, what='dbias')
    for i in range(L):
        assert_close(r['dconvs'][i][0], g['grad.cnn_%d.weight' % i], 1e-5, what='dW%d' % i)
        assert_close(r['dconvs'][i][1], g['grad.cnn_%d.bias' % i], 1e-5, what='db%d' % i)


@pytest.mark.parametrize('n', [1, 2, 3, 5, 17, 100, 1000, 4097, 100000])
def test_parallel_shuffle_formulation_matches_numpy(n):
    """The fixed-point / link-and-chase formulation csrc/shuffle.cu implements, restated in
    oracle/shuffle.py, is RandomState.shuffle (torch_utils.py:46-47): same permutation, same
    number of stream words consumed."""
    from oracle import shuffle as osh
    for seed in (0, 7):
        rs = np.random.RandomState(seed)
        rs.randint(0, 100, 33)                                   # mid-block start
        probe = np.random.RandomState()
        probe.set_state(rs.get_state())
        words = probe.randint(0, 2 ** 32, 2 * n + 64, dtype=np.uint64).astype(np.uint32)
        j, used = osh.resolve_draws(words, n)
        got = osh.apply_swaps(j)
        want = np.arange(n)
        rs.shuffle(want)
        assert np.array_equal(got, want)
        probe2 = np.random.RandomState(seed)                     # consume exactly `used` words
        probe2.randint(0, 100, 33)
        if used:
            probe2.randint(0, 2 ** 32, used, dtype=np.uint64)
        assert np.array_equal(probe2.get_state()[1], rs.get_state()[1])
        assert probe2.get_state()[2] == rs.get_state()[2]


def test_oracle_bloom_step_vs_reference_golden():
    """oracle.mf.mf_bloom_step (hashed item rows summed, raw-id biases) against the gradients the
    live reference produced for BilinearNet + BloomEmbedding (tests/golden/mf_hinge_bloom.npz)."""
    from oracle import mf as omf
    g = load_golden('mf_hinge_bloom')
    r = omf.mf_bloom_step(g['sd.user_embeddings.weight'], g['sd.item_embeddings.embeddings.weight'],
                          g['sd.user_biases.weight'], g['sd.item_biases.weight'], g['users'], g['items'],
                          g['negs'], 'hinge', int(g['bloom_H']), 0, np.float64)
    assert_close(float(r['loss']), float(g['loss']), 1e-6, what='loss')
    assert_close(r['pos'], g['pos'], 1e-5, what='pos')
    for k, nm in (('dWu', 'user_embeddings.weight'), ('dWi', 'item_embeddings.embeddings.weight'),
                  ('dbu', 'user_biases.weight'), ('dbi', 'item_biases.weight')):
        assert_close(r[k], g['grad.' + nm], 1e-6, atol=1e-12, what=k)

