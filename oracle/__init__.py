"""CPU oracle for the clustering / memory / loss / scoring hot path.

TEST INFRASTRUCTURE ONLY.  Nothing under ``oracle/`` is part of the product:
only ``tests/``, ``__graft_entry__.smoke()`` and ``bench.py``'s CPU-baseline /
``--impl reference`` legs may import it, and there only as the checker (or as
the timed CPU baseline), never as something the CUDA path routes through.

* ``np_oracle``  – numpy restatement of the reference algorithms (fp32 in the
  reference's operation order by default, fp64 on request for adjudicating
  near-ties).  Every function cites the reference ``file:line`` it follows.
* ``ref_loader`` – imports the UNMODIFIED reference (the checkout named by ``VADC_REFERENCE_ROOT``, or the staged
  copy ``baseline/_ref``) with stubs for its absent, unused dependencies: the reference arm of bench.py (``kind:
  "reference"``), its ``gpu_reference`` leg and the model-level drop-in test use the reference's own classes.
* ``ref_port``   – the same op chain written with torch CPU ops, used as the
  timed CPU baseline (the reference itself is a torch program, so this is the
  closest thing to "the reference's own CPU implementation" that can travel
  to the GPU box, where ``/root/reference`` does not exist).

Pinning: the reference ships no tests or golden vectors (SURVEY.md §4), so the
oracle is pinned against outputs of the reference's own modules imported from
``/root/reference`` in the build container: ``tests/golden/make_golden.py``
generated the fixtures in ``tests/golden/*.npz`` and ``tests/test_oracle_*``
checks both oracles against them.
"""
