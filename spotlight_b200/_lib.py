"""ctypes binding of the C-ABI library (include/spotlight_b200.h).

The library is resolved lazily through this module-level loader so that models
stay picklable (``torch.save(model)``, reference tests/test_serialization.py:
29-30): no ctypes handle ever lives in a model's ``__dict__``.

There is no CPU fallback: if ``libspotlight_b200.so`` is missing the first use
raises, loudly.
"""

import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get('SLB_LIBRARY') or os.path.join(_HERE, 'libspotlight_b200.so')

c_i32, c_i64, c_f32 = ctypes.c_int32, ctypes.c_int64, ctypes.c_float
c_vp, c_sz = ctypes.c_void_p, ctypes.c_size_t

LOSS_KIND = {'pointwise': 0, 'bpr': 1, 'hinge': 2, 'adaptive_hinge': 3}
GRAD_DENSE, GRAD_COMPACT = 0, 1
OPT_NONE, OPT_SGD, OPT_ADAGRAD, OPT_ADAM = 0, 1, 2, 3

# every symbol include/spotlight_b200.h declares
EXPORTS = (
    'slb_version', 'slb_last_error', 'slb_sm_count', 'slb_workspace_init',
    'slb_mt19937_fill', 'slb_mt19937_fill_parallel', 'slb_mt19937_direct_slots',
    'slb_mt19937_fill_direct', 'slb_host_shuffle_order',
    'slb_sample_workspace_bytes', 'slb_sample_bounded', 'slb_sample_bounded_chain',
    'slb_shuffle_workspace_bytes', 'slb_shuffle_order', 'slb_permute_ids',
    'slb_embedding_forward', 'slb_bloom_rows',
    'slb_embedding_backward_workspace_bytes', 'slb_embedding_backward',
    'slb_mf_scores', 'slb_mf_scores_backward', 'slb_rank_pairs', 'slb_mf_step_workspace_bytes', 'slb_mf_fused_workspace_bytes', 'slb_mf_compact_rows',
    'slb_mf_train_step', 'slb_mf_train_step_phases', 'slb_mf_plan_copy', 'slb_mf_fused_layout', 'slb_mf_fit_epoch', 'slb_mf_fit_epoch_events', 'slb_adam_flush',
    'slb_mf_bloom_workspace_bytes', 'slb_mf_bloom_train_step',
    'slb_bias_sparse_workspace_bytes', 'slb_bias_sparse_apply',
    'slb_unique_workspace_bytes', 'slb_unique_bucket', 'slb_shard_gather_batch', 'slb_adagrad_dense',
    'slb_loss_workspace_bytes', 'slb_pairwise_loss',
    'slb_seq_step_workspace_bytes', 'slb_seq_train_step', 'slb_seq_representation',
)


class MfStepArgs(ctypes.Structure):
    """struct slb_mf_step_args."""
    _fields_ = [
        ('batch', c_i64), ('users', c_vp), ('items', c_vp), ('negs', c_vp),
        ('loss', c_i32), ('n_neg', c_i32),
        ('num_users', c_i64), ('num_items', c_i64), ('dim', c_i32),
        ('Wu', c_vp), ('Wi', c_vp), ('bu', c_vp), ('bi', c_vp),
        ('loss_out', c_vp), ('pos_out', c_vp), ('neg_out', c_vp),
        ('grad_mode', c_i32),
        ('dWu', c_vp), ('dWi', c_vp), ('dbu', c_vp), ('dbi', c_vp),
        ('urows', c_vp), ('gWu', c_vp), ('gbu', c_vp),
        ('irows', c_vp), ('gWi', c_vp), ('gbi', c_vp),
        ('compact_counts', c_vp),
        ('opt', c_i32), ('lr', c_f32), ('weight_decay', c_f32), ('eps', c_f32),
        ('state_Wu', c_vp), ('state_Wi', c_vp), ('state_bu', c_vp), ('state_bi', c_vp),
        ('norm_batch', c_i64), ('opt_users_only', c_i32),
        ('workspace', c_vp), ('workspace_bytes', c_sz),
        ('fused_workspace', c_vp), ('fused_workspace_bytes', c_sz), ('plan_stream', c_vp),
        ('beta1', c_f32), ('beta2', c_f32), ('one_minus_beta1', c_f32), ('one_minus_beta2', c_f32),
        ('state2_Wu', c_vp), ('state2_Wi', c_vp), ('state2_bu', c_vp), ('state2_bi', c_vp),
        ('last_u', c_vp), ('last_i', c_vp), ('adam_sched', c_vp), ('adam_step', c_i64),
    ]


class MfBloomArgs(ctypes.Structure):
    """struct slb_mf_bloom_args."""
    _fields_ = [
        ('base', MfStepArgs),
        ('user_rows', c_i64), ('item_rows', c_i64),
        ('user_hashes', c_i32), ('item_hashes', c_i32),
        ('user_seeds', ctypes.c_uint32 * 24), ('item_seeds', ctypes.c_uint32 * 24),
        ('user_padding_idx', c_i64), ('item_padding_idx', c_i64),
        ('pair_ids_u', c_vp), ('pair_g_u', c_vp), ('pair_ids_i', c_vp), ('pair_g_i', c_vp),
    ]


class SeqStepArgs(ctypes.Structure):
    """struct slb_seq_step_args."""
    _fields_ = [
        ('batch', c_i64), ('seq_len', c_i32), ('seqs', c_vp), ('negs', c_vp),
        ('loss', c_i32), ('n_neg', c_i32),
        ('num_items', c_i64), ('dim', c_i32),
        ('E', c_vp), ('bias', c_vp),
        ('n_layers', c_i32), ('kernel_width', c_vp), ('dilation', c_vp),
        ('nonlinearity', c_i32), ('residual', c_i32),
        ('conv_w', c_vp), ('conv_b', c_vp), ('dconv_w', c_vp), ('dconv_b', c_vp),
        ('loss_out', c_vp), ('pos_out', c_vp), ('neg_out', c_vp),
        ('dE', c_vp), ('dbias', c_vp),
        ('norm_count', c_vp),
        ('workspace', c_vp), ('workspace_bytes', c_sz),
        ('opt', c_i32), ('lr', c_f32), ('weight_decay', c_f32), ('eps', c_f32),
        ('state_E', c_vp), ('state_bias', c_vp),
    ]


_lib = None


class LibraryError(RuntimeError):
    pass


def _declare(lib):
    P = ctypes.POINTER
    lib.slb_version.restype = c_i32
    lib.slb_last_error.restype = ctypes.c_char_p
    lib.slb_sm_count.restype = c_i32
    lib.slb_workspace_init.argtypes = [c_vp, c_sz, c_vp]
    lib.slb_mt19937_fill.argtypes = [c_vp, c_i64, c_vp]
    lib.slb_mt19937_fill_parallel.argtypes = [c_vp, c_i64, c_vp, c_i32, c_vp, c_vp]
    lib.slb_mt19937_direct_slots.argtypes = [c_i64, c_i32]
    lib.slb_mt19937_direct_slots.restype = c_i64
    lib.slb_mt19937_fill_direct.argtypes = [c_vp, c_i64, c_vp, c_i32, c_vp, c_i32, c_i32, c_vp, c_i64, c_vp]
    lib.slb_sample_bounded_chain.argtypes = [c_vp, c_i64, c_vp, ctypes.c_uint32, c_i64, c_vp, c_vp, c_sz, c_vp]
    lib.slb_host_shuffle_order.argtypes = [c_vp, c_vp, c_i64, c_i32, c_vp]
    lib.slb_shuffle_workspace_bytes.argtypes = [c_i64, c_i64]
    lib.slb_shuffle_workspace_bytes.restype = c_sz
    lib.slb_shuffle_order.argtypes = [c_vp, c_i64, c_vp, c_i64, c_i64, c_i32, c_i32, c_vp, c_vp, c_sz, c_vp]
    lib.slb_permute_ids.argtypes = [c_vp, c_i64, c_vp, c_vp, c_i32, c_vp, c_vp, c_vp]
    lib.slb_sample_workspace_bytes.argtypes = [c_i64]
    lib.slb_sample_workspace_bytes.restype = c_sz
    lib.slb_sample_bounded.argtypes = [c_vp, c_i64, c_vp, ctypes.c_uint32, c_i64, c_vp, c_vp, c_sz, c_vp]
    lib.slb_embedding_forward.argtypes = [c_vp, c_i64, c_i32, c_vp, c_i64, c_i32, c_vp, c_i64, c_vp, c_vp]
    lib.slb_bloom_rows.argtypes = [c_vp, c_i64, c_i32, c_vp, c_i64, c_i64, c_vp, c_vp]
    lib.slb_embedding_backward_workspace_bytes.argtypes = [c_i64, c_i64]
    lib.slb_embedding_backward_workspace_bytes.restype = c_sz
    lib.slb_embedding_backward.argtypes = [c_vp, c_vp, c_i64, c_i32, c_vp, c_i64, c_i32, c_i64,
                                           c_vp, c_vp, c_sz, c_vp]
    lib.slb_mf_scores.argtypes = [c_vp, c_vp, c_vp, c_vp, c_i32, c_vp, c_vp, c_i64, c_i32, c_vp, c_vp]
    lib.slb_mf_scores_backward.argtypes = [c_vp, c_vp, c_vp, c_i64, c_i32, c_vp, c_vp, c_i64, c_i64, c_i32,
                                           c_vp, c_vp, c_vp, c_vp, c_vp, c_sz, c_vp]
    lib.slb_rank_pairs.argtypes = [c_vp, c_i64, c_i64, c_vp, c_vp, c_i64, c_vp, c_vp]
    lib.slb_mf_step_workspace_bytes.argtypes = [c_i64, c_i32, c_i32, c_i64, c_i64]
    lib.slb_mf_step_workspace_bytes.restype = c_sz
    lib.slb_mf_fused_workspace_bytes.argtypes = [c_i64, c_i64, c_i64, c_i32]
    lib.slb_mf_fused_workspace_bytes.restype = c_sz
    lib.slb_mf_compact_rows.argtypes = [c_i64, c_i32, c_i32, c_i32]
    lib.slb_mf_compact_rows.restype = c_i64
    lib.slb_mf_train_step.argtypes = [P(MfStepArgs), c_vp]
    lib.slb_mf_train_step_phases.argtypes = [P(MfStepArgs), c_i32, c_vp]
    lib.slb_mf_fused_layout.argtypes = [P(MfStepArgs), c_vp, c_i32]
    lib.slb_mf_fused_layout.restype = c_i32
    lib.slb_mf_plan_copy.argtypes = [P(MfStepArgs), c_i32, c_i64, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp]
    lib.slb_mf_bloom_workspace_bytes.argtypes = [P(MfBloomArgs)]
    lib.slb_mf_bloom_workspace_bytes.restype = c_sz
    lib.slb_mf_bloom_train_step.argtypes = [P(MfBloomArgs), c_vp]
    lib.slb_bias_sparse_workspace_bytes.argtypes = [c_i64]
    lib.slb_bias_sparse_workspace_bytes.restype = c_sz
    lib.slb_bias_sparse_apply.argtypes = [c_vp, c_vp, c_i64, c_vp, c_vp, c_i32, c_f32, c_f32, c_f32, c_vp, c_sz, c_vp]
    lib.slb_mf_fit_epoch.argtypes = [P(MfStepArgs), c_vp, c_vp, c_vp, c_i64, c_vp, c_vp]
    lib.slb_mf_fit_epoch_events.argtypes = [P(MfStepArgs), c_vp, c_vp, c_vp, c_i64, c_vp, c_vp, c_vp, c_vp, c_i32]
    lib.slb_adam_flush.argtypes = [c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_i64, c_i32, c_vp, c_i64,
                                   c_f32, c_f32, c_f32, c_f32, c_f32, c_f32, c_vp]
    lib.slb_unique_workspace_bytes.argtypes = [c_i64, c_i64]
    lib.slb_unique_workspace_bytes.restype = c_sz
    lib.slb_unique_bucket.argtypes = [c_vp, c_i64, c_i64, c_i64, c_i32, c_vp, c_vp, c_vp, c_vp, c_sz, c_vp]
    lib.slb_shard_gather_batch.argtypes = [c_vp, c_i64, c_vp, c_vp, c_vp, c_i64, c_i32, c_i64, c_vp, c_vp, c_vp, c_vp]
    lib.slb_adagrad_dense.argtypes = [c_vp, c_vp, c_vp, c_i64, c_f32, c_f32, c_vp]
    lib.slb_loss_workspace_bytes.argtypes = [c_i64]
    lib.slb_loss_workspace_bytes.restype = c_sz
    lib.slb_pairwise_loss.argtypes = [c_i32, c_vp, c_vp, c_vp, c_i64, c_i32, c_vp, c_vp, c_vp,
                                      c_vp, c_sz, c_vp]
    lib.slb_seq_step_workspace_bytes.argtypes = [P(SeqStepArgs)]
    lib.slb_seq_step_workspace_bytes.restype = c_sz
    lib.slb_seq_train_step.argtypes = [P(SeqStepArgs), c_vp]
    lib.slb_seq_representation.argtypes = [P(SeqStepArgs), c_vp, c_vp]
    for name in EXPORTS:
        fn = getattr(lib, name)
        if fn.restype is ctypes.c_int:   # default -> status code
            fn.restype = c_i32


def load():
    """Return the loaded library; raise (no CPU fallback) if it is missing."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise LibraryError(
                'spotlight_b200: %s not found. Build it with '
                '`python -c "import __graft_entry__ as g; g.build()"` (needs nvcc, sm_100a). '
                'There is no CPU fallback.' % LIB_PATH)
        lib = ctypes.CDLL(LIB_PATH)
        missing = [n for n in EXPORTS if not hasattr(lib, n)]
        if missing:
            raise LibraryError('spotlight_b200: library lacks symbols %s' % missing)
        _declare(lib)
        if lib.slb_version() != 100:
            raise LibraryError('spotlight_b200: ABI version mismatch')
        _lib = lib
    return _lib


def check(rc, what=''):
    """Raise on a negative status code with the library's message."""
    if rc != 0:
        msg = load().slb_last_error().decode('utf-8', 'replace')
        if rc == -1:
            raise ValueError('%s: %s' % (what or 'spotlight_b200', msg))
        raise LibraryError('%s failed (%d): %s' % (what or 'spotlight_b200', rc, msg))
