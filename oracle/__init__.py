"""CPU oracle for the VNect per-frame hot path.

TEST INFRASTRUCTURE ONLY.  Nothing under ``vnect_b200/`` may import this package; only ``tests/``,
``__graft_entry__.smoke()`` and the ``cpu_baseline`` / ``--impl reference`` legs of ``bench.py`` do, and there only
as the checker or as the CPU baseline being timed, never as the product path.

What it restates (reference = XinArkh/VNect, read-only from the checkout VNECT_REFERENCE_ROOT names, see ref_shim):

* ``oracle.forward``   -- the CNN of ``src/vnect_model.py:27-217`` as a torch-CPU fp32/fp64 graph (TensorFlow 1.x is not
  installable here; TF1 layer defaults are documented in SURVEY.md section 8c).
* ``oracle.prepost``   -- ``src/estimator.py:70-142``, ``src/utils.py:13-21,58-219`` and ``src/OneEuroFilter.py:13-75`` in
  numpy, including an integer restatement of OpenCV's 8-bit INTER_LINEAR resize.
* ``oracle.weights``   -- seeded random-init weights in the reference's pickle interchange format
  (``src/caffe2pkl.py:57-76``).

Pinning: the reference ships no tests, golden vectors or weights (SURVEY.md section 4), so the CNN restatement is
"parity unpinned" against TensorFlow itself.  Everything else is pinned: ``tests/golden/make_golden.py`` imports the
reference's own ``src/utils.py``, ``src/OneEuroFilter.py`` and ``src/estimator.py`` unchanged from that checkout
(with a stub ``tensorflow`` whose ``Session.run`` calls ``oracle.forward``) and commits their outputs under
``tests/golden/``; ``tests/test_oracle_*.py`` check the numpy restatement against those fixtures and against cv2.
"""
