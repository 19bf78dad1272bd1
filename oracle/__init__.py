"""TEST INFRASTRUCTURE ONLY -- the parity oracle for the NFP hot path.

Nothing under ``oracle/`` is part of the product.  Only ``tests/``,
``__graft_entry__.smoke()`` and the CPU-baseline / ``--impl reference`` legs of
``bench.py`` may import it, and there only as the checker or as the timed CPU
baseline -- never as a fallback for the CUDA path.

Parity status: **pinned**.  The reference ships no tests or golden vectors
(SURVEY.md section 4), so the oracle is pinned by executing the reference's own
Python modules where a checkout of it exists (``oracle/check_against_reference.py``)
and by the committed fixtures under ``tests/golden/`` generated from the
reference by ``oracle/make_golden.py``.
"""
