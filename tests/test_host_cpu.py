"""CPU-only tests: host logic, the C-ABI surface, and the no-CPU-fallback rule."""

import os
import re

import numpy as np
import pytest
import torch

from conftest import ROOT, load_golden


def _header_symbols():
    text = open(os.path.join(ROOT, 'include', 'spotlight_b200.h')).read()
    text = re.sub(r'/\*.*?\*/', '', text, flags=re.S)
    return sorted(set(re.findall(r'\b(slb_[a-z0-9_]+)\s*\(', text)))


def test_library_exports_every_declared_symbol():
    import ctypes
    from spotlight_b200 import _lib
    names = _header_symbols()
    assert len(names) >= 20
    lib = ctypes.CDLL(_lib.LIB_PATH)
    for n in names:
        assert hasattr(lib, n), n
    assert sorted(_lib.EXPORTS) == names
    loaded = _lib.load()
    assert loaded.slb_version() == 100


def test_struct_layout_matches_header_field_order():
    from spotlight_b200._lib import MfStepArgs, SeqStepArgs
    text = open(os.path.join(ROOT, 'include', 'spotlight_b200.h')).read()
    for cls, tag in ((MfStepArgs, 'slb_mf_step_args'), (SeqStepArgs, 'slb_seq_step_args')):
        body = text.split('typedef struct %s {' % tag)[1].split('} %s;' % tag)[0]
        body = re.sub(r'/\*.*?\*/', '', body, flags=re.S)
        fields = []
        for decl in body.split(';'):
            decl = decl.strip()
            if not decl:
                continue
            for part in decl.split(','):
                name = re.findall(r'([A-Za-z_][A-Za-z0-9_]*)\s*$', part.strip())
                fields.append(name[0])
        assert fields == [f[0] for f in cls._fields_], tag


def test_no_cpu_path():
    from spotlight_b200 import ops
    from spotlight_b200.layers import BloomEmbedding, ScaledEmbedding
    ids = torch.arange(4)
    for layer in (ScaledEmbedding(10, 8), BloomEmbedding(100, 8)):
        with pytest.raises(RuntimeError, match='no CPU path'):
            layer(ids)
    with pytest.raises(RuntimeError, match='no CPU path'):
        ops.mf_scores(torch.zeros(4, 8), torch.zeros(4, 8), torch.zeros(4, 1), torch.zeros(4, 1),
                      ids, ids)


def test_product_never_imports_oracle():
    bad = []
    for dirpath, _, files in os.walk(os.path.join(ROOT, 'spotlight_b200')):
        for f in files:
            if f.endswith('.py'):
                src = open(os.path.join(dirpath, f)).read()
                if re.search(r'^\s*(from|import)\s+oracle', src, flags=re.M):
                    bad.append(f)
    assert not bad, bad


def test_layer_parameter_names_and_init():
    from spotlight_b200.factorization.representations import BilinearNet
    from spotlight_b200.layers import BloomEmbedding, ScaledEmbedding, ZeroEmbedding
    net = BilinearNet(30, 20, 16)
    shapes = {k: tuple(v.shape) for k, v in net.state_dict().items()}
    assert shapes == {'user_embeddings.weight': (30, 16), 'item_embeddings.weight': (20, 16),
                      'user_biases.weight': (30, 1), 'item_biases.weight': (20, 1)}
    assert float(ZeroEmbedding(5, 1).weight.abs().sum()) == 0.0
    e = ScaledEmbedding(2000, 64, padding_idx=0)
    assert float(e.weight[0].abs().sum()) == 0.0
    assert abs(float(e.weight[1:].std()) - 1.0 / 64) < 2e-3          # std 1/D, not 1/sqrt(D)
    b = BloomEmbedding(1000, 8, compression_ratio=0.25, num_hash_functions=3)
    assert b.compressed_num_embeddings == 250 and tuple(b.embeddings.weight.shape) == (250, 8)
    with pytest.raises(ValueError):
        BloomEmbedding(10, 4, num_hash_functions=25)
    with pytest.raises(NotImplementedError):
        BloomEmbedding(10, 4, bag=True)


def test_interactions_and_to_sequence():
    from spotlight_b200.interactions import Interactions
    g = load_golden('to_sequence')
    it = Interactions(g['users'], g['items'], timestamps=g['ts'])
    for tag, kw in [('a', dict(max_sequence_length=7)),
                    ('b', dict(max_sequence_length=5, step_size=1)),
                    ('c', dict(max_sequence_length=6, min_sequence_length=3, step_size=2))]:
        s = it.to_sequence(**kw)
        assert s.sequences.dtype == np.int32
        assert (s.sequences == g['seq_' + tag]).all() and (s.user_ids == g['uid_' + tag]).all()
    # the reference's two known-answer cases (tests/test_interactions.py:67-100)
    it = Interactions(np.zeros(5), np.arange(5) + 1, timestamps=np.arange(5))
    assert (it.to_sequence(max_sequence_length=5, step_size=1).sequences == np.array(
        [[1, 2, 3, 4, 5], [0, 1, 2, 3, 4], [0, 0, 1, 2, 3], [0, 0, 0, 1, 2], [0, 0, 0, 0, 1]])).all()
    assert (it.to_sequence(max_sequence_length=5, step_size=2).sequences == np.array(
        [[1, 2, 3, 4, 5], [0, 0, 1, 2, 3], [0, 0, 0, 0, 1]])).all()
    with pytest.raises(ValueError):
        Interactions(np.arange(3), np.arange(3), num_users=2)
    with pytest.raises(ValueError):
        Interactions(np.arange(3), np.arange(3)).to_sequence()          # no timestamps
    assert it.tocsr().shape == (1, 6)


def test_shuffle_and_minibatch_follow_the_stream():
    from spotlight_b200.torch_utils import minibatch, shuffle
    a, b = np.arange(100), np.arange(100) * 2
    r1, r2 = np.random.RandomState(3), np.random.RandomState(3)
    sa, sb = shuffle(a, b, random_state=r1)
    order = np.arange(100)
    r2.shuffle(order)
    assert (sa == a[order]).all() and (sb == b[order]).all()
    assert r1.get_state()[2] == r2.get_state()[2]
    chunks = list(minibatch(torch.arange(10), torch.arange(10), batch_size=4))
    assert [len(c[0]) for c in chunks] == [4, 4, 2]
    with pytest.raises(ValueError):
        shuffle(a, b[:5])


def test_fast_host_shuffle_is_bit_exact():
    """csrc/host_shuffle.cpp vs RandomState.shuffle: permutation and final state."""
    from spotlight_b200.torch_utils import shuffled_order
    for n in (0, 1, 2, 3, 100, 1000, 65537, 300_001):
        a, b = np.random.RandomState(5), np.random.RandomState(5)
        a.randint(0, 9, 11)
        b.randint(0, 9, 11)
        x = np.arange(n)
        a.shuffle(x)
        y = shuffled_order(n, b)
        assert (x == y).all(), n
        sa, sb = a.get_state(), b.get_state()
        assert (sa[1] == sb[1]).all() and sa[2] == sb[2], n
        assert (a.randint(0, 1000, 20) == b.randint(0, 1000, 20)).all()


def test_sample_items_host_path_is_numpy():
    from spotlight_b200.sampling import sample_items
    r1, r2 = np.random.RandomState(9), np.random.RandomState(9)
    assert (sample_items(1683, (4, 5), r1) == r2.randint(0, 1683, (4, 5), dtype=np.int64)).all()


def test_shuffle_stream_budget_covers_consumption():
    """rng.shuffle_begin sizes the stream as E[words] + 8 sigma: check the expectation and
    the margin against the words RandomState.shuffle really consumes (oracle/shuffle.py)."""
    import math
    from oracle import shuffle as osh
    from spotlight_b200.rng import _shuffle_expected_words
    for n in (2, 3, 10, 1000, 4097, 65537, 300000):
        used = []
        for seed in range(6):
            rs = np.random.RandomState(seed)
            words = rs.randint(0, 2 ** 32, 2 * n + 64, dtype=np.uint64).astype(np.uint32)
            used.append(osh.resolve_draws(words, n)[1])
        budget = _shuffle_expected_words(n) + 8.0 * math.sqrt(2.0 * n) + 64
        assert max(used) <= budget
        assert abs(np.mean(used) - _shuffle_expected_words(n)) <= 4.0 * math.sqrt(2.0 * n / 6) + 2


def test_every_entry_point_is_documented():
    """Each exported slb_* symbol is declared in include/spotlight_b200.h and has a row in
    INTEGRATION.md's entry-point table (what it replaces in the reference)."""
    import re
    from conftest import ROOT
    from spotlight_b200 import _lib
    header = open(os.path.join(ROOT, 'include', 'spotlight_b200.h')).read()
    doc = open(os.path.join(ROOT, 'INTEGRATION.md')).read()
    declared = set(re.findall(r'\b(slb_[a-z0-9_]+)\s*\(', header))
    assert set(_lib.EXPORTS) <= declared
    prefixes = re.findall(r'`(slb_[a-z_]+_)`', doc)          # the workspace_bytes family row
    undocumented = [name for name in _lib.EXPORTS if name not in doc and
                    not (name.endswith('_workspace_bytes') and
                         any(name == p + 'workspace_bytes' for p in prefixes))]
    assert not undocumented, undocumented


def test_fused_adam_schedule_and_dense_fallback():
    """FusedAdam (row-wise lazy-exact Adam, the reference's default optimizer at O(batch)): the
    per-step scalar table the kernels replay with, and the dense step() fallback, against
    torch.optim.Adam on CPU tensors (implicit.py:143-148)."""
    import numpy as np
    import torch
    from spotlight_b200.optim import FusedAdam
    torch.manual_seed(0)
    W1 = torch.nn.Parameter(torch.randn(7, 4))
    b1 = torch.nn.Parameter(torch.randn(7, 1))
    W2 = torch.nn.Parameter(W1.detach().clone())
    b2 = torch.nn.Parameter(b1.detach().clone())
    mine = FusedAdam([W1, b1], lr=1e-2, weight_decay=1e-3)
    ref = torch.optim.Adam([W2, b2], lr=1e-2, weight_decay=1e-3)
    sched = mine.schedule(10, torch.device('cpu')).reshape(-1, 2).numpy()
    for t in (1, 2, 7, 10):
        assert abs(sched[t, 0] - 1e-2 / (1 - 0.9 ** t)) < 1e-7 * sched[t, 0] + 1e-12
        assert abs(sched[t, 1] - np.sqrt(1 - 0.999 ** t)) < 1e-6
    for _ in range(5):
        g, gb = torch.randn(7, 4), torch.randn(7, 1)
        W1.grad, b1.grad, W2.grad, b2.grad = g.clone(), gb.clone(), g.clone(), gb.clone()
        mine.step()
        ref.step()
    assert mine.steps_taken == 5
    assert torch.allclose(W1, W2, rtol=1e-5, atol=1e-7) and torch.allclose(b1, b2, rtol=1e-5, atol=1e-7)
    assert int(mine.state[W1]['last'].min()) == 5



def test_reference_arm_prints_the_contract_line():
    """`bench.py --impl reference` (the CPU arm timed beside ours): runs the
    reference's own fit loop (oracle/_ref when installed, else the oracle port) on the
    host cores and prints one JSON line with the contract's keys.  Tiny workload here."""
    import json
    import subprocess
    import sys
    cmd = [sys.executable, os.path.join(ROOT, 'bench.py'), '--impl', 'reference', '--steps', '2', '--warmup', '1',
           '--batch', '2048', '--users', '5000', '--items', '2000', '--dim', '16']
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=300, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    assert line['impl'] == 'reference' and 'unavailable' not in line
    for key in ('metric', 'value', 'unit', 'n_gpus', 'steps', 'warmup', 'ms_per_step', 'higher_is_better',
                'scaling', 'dtype', 'data', 'config', 'cpu_baseline', 'e2e'):
        assert key in line, key
    assert line['steps'] == 2 and line['warmup'] == 1 and line['n_gpus'] == 1
    assert line['value'] > 0 and line['higher_is_better'] is True
    cb = line['cpu_baseline']
    # the unmodified reference whenever build() installed it; the torch restatement only without it
    installed = os.path.isdir(os.path.join(ROOT, 'oracle', '_ref', 'spotlight'))
    assert cb['kind'] == ('reference' if installed else 'port')
    assert cb['cores'] >= 1 and cb['value'] == line['value']
    assert line['e2e']['value'] == line['value']
    assert line['e2e']['h2d_bytes_per_step'] == 0 and line['e2e']['d2h_bytes_per_step'] == 0
    assert 'workload' in line['config'] and 'model' not in line['config']
