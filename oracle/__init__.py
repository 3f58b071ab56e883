"""CPU oracle for the A2C caption-training hot path.

TEST INFRASTRUCTURE ONLY.  Nothing under ``oracle/`` is product code: only
``tests/``, ``__graft_entry__.smoke()`` and ``bench.py``'s CPU-baseline /
``--impl reference`` legs may import it, and only as the checker or as the CPU
baseline being timed.  The product path (``icrl_b200``) never imports it and has
no CPU fallback.

Parity status: the reference (pratikpv/image-captioning-through-rl) ships no tests
and no golden vectors (SURVEY.md §4, §8c), so this oracle is pinned against the
reference *itself*, executed unmodified in the build container by
``oracle/gen_golden.py`` (committed) which writes ``tests/golden/*.npz``.  The
oracle is checked against those fixtures by ``tests/test_oracle_golden.py`` on
every CPU run.

Where the reference's sources are present, ``__graft_entry__.build()`` copies its
four flat, unmodified modules into the git-ignored ``oracle/_ref/`` (it has no
setup.py / pyproject.toml to install from), so that ``tests/test_gpu_boundary.py``
can run the reference's own training loop on the drop-in modules wherever this
tree is run, and ``oracle/gen_golden.py`` can regenerate the fixtures.

Modules
-------
synth        re-export of icrl_b200.synth (seeded synthetic weights / inputs; lives product-side so that
             bench.py's GPU arm imports nothing from oracle/)
ref_port     the reference algorithm *as executed* (per-step prefix re-runs, the
             batch-as-time value/reward RNN calls with carried state) on torch
             CPU library layers -- the CPU baseline that bench.py times
single_pass  the verified single-pass restatement (SURVEY.md §8c) with the cell
             arithmetic written out -- what the CUDA kernels are checked against
"""

import os as _os

REFERENCE_SRC = _os.environ.get("ICRL_REFERENCE_DIR", "/root/reference")      # a checkout of the reference
REFERENCE_INSTALL = _os.path.join(_os.path.dirname(_os.path.abspath(__file__)), "_ref")
REFERENCE_MODULES = ("trainers.py", "utilities.py", "metrics.py", "models.py")


def reference_dir():
    """The installed copy oracle/_ref/, else the checkout itself; None where neither holds the reference's modules."""
    for d in (REFERENCE_INSTALL, REFERENCE_SRC):
        if all(_os.path.exists(_os.path.join(d, m)) for m in REFERENCE_MODULES):
            return d
    return None
