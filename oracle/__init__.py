"""oracle/ -- TEST INFRASTRUCTURE ONLY.

CPU restatement of the reference hot path (wvangansbeke/LaneDetection_End2End:
ERFNet -> activation/mask -> weighted least-squares layer -> loss on beta).

Nothing in the product package (``lanedetection_end2end_b200``) may import this
package.  Only ``tests/``, ``__graft_entry__.smoke()`` and ``bench.py``'s
``cpu_baseline`` / ``--impl reference`` legs use it, and only as the checker or
as the reported CPU baseline -- never as the measured GPU path.

Pinning status: the reference ships no tests and no golden vectors (SURVEY.md
section 8c), so the oracle is pinned against outputs of the reference ITSELF,
imported through ``oracle/reference_import.py`` by
``oracle/make_golden.py`` (committed), which writes ``tests/golden/*.npz``.
``tests/test_oracle_vs_golden.py`` checks the restatement against those
fixtures on every run.
"""
