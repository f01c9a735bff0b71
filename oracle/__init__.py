"""TEST INFRASTRUCTURE ONLY -- CPU oracle for the VI-HMC hot path.

Nothing under ``oracle/`` is part of the product.  Only ``tests/``,
``__graft_entry__.smoke()`` and ``bench.py``'s CPU-baseline / ``--impl reference``
legs may import it, and there only as the checker (or as the timed CPU arm),
never as the thing shipped.  The product path (``vi-hmc_b200/``) never imports
this package and fails loudly when its CUDA library is missing.

Contents
--------
closures.py             torch-CPU restatement of the reference's log-posterior
                        closures (BNN VI-HMC, BNN full HMC, DeepONet, split).
hamiltorch_restated.py  restatement of the third-party sampler the reference
                        calls (hamiltorch, unpinned git HEAD, absent here).
philox_ref.py           numpy Philox4x32-10 + uniform/normal transforms.
ref_loader.py           imports the REAL reference closures from a checkout in
                        oracle/_ref/ or VIHMC_REFERENCE_ROOT (not in this repository).
make_golden.py          writes tests/golden/* from the real reference closures.

Parity status
-------------
* log-posterior value + gradient: PINNED against the reference's own closures
  (tests/golden/*.npz were produced by importing the original project).
* sampler arithmetic (hamiltorch): PARITY UNPINNED -- the package is not on
  disk and not pinned by the reference; the restatement is the spec.
"""
