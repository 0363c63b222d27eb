"""CPU oracle for the implicit-feedback fit() hot path.

TEST INFRASTRUCTURE ONLY.  Nothing under ``spotlight_b200/`` may import this
package; only ``tests/``, ``__graft_entry__.smoke()`` and ``bench.py``'s
``cpu_baseline`` / ``--impl reference`` legs do, and there only as the checker
or the timed CPU baseline -- never as the product path.

Contents (every function cites the reference file:line it restates):

* ``mt19937``   -- NumPy-legacy ``RandomState`` stream (MT19937 + masked
                   rejection) that drives ``sample_items`` and ``shuffle``.
* ``murmur``    -- MurmurHash3_x86_32 as used by ``BloomEmbedding``.
* ``mf``        -- BilinearNet forward / the four losses / closed-form backward.
* ``seq``       -- PoolNet and CNNNet forward / backward closed forms.
* ``shuffle``   -- ``RandomState.shuffle`` (Fisher-Yates on the same stream).
* ``adam``      -- the row-wise lazy-exact Adam scheme (catch-up before the forward, real step,
                   flush), pinned against the reference's recorded default-Adam trajectory.
* ``torch_port``-- the reference's fit() loop restated on stock torch CPU ops
                   (the timed ``cpu_baseline`` "port", used by bench.py only when
                   the unmodified reference is not installed under
                   ``oracle/_ref``).
* ``reference`` -- installs that unmodified reference under ``oracle/_ref``.

The reference is pure Python (no C sources to compile into ``oracle/_ref``); the
restatements are NumPy, so there is no C build step for the oracle.

Parity pinning: the restatements are checked (tests/test_oracle_*.py) against
golden vectors produced by the *live* reference (``tests/golden/make_golden.py``
imports a checkout of it), against NumPy's own ``RandomState`` and against
``sklearn.utils.murmurhash3_32`` (recorded there too).
"""
