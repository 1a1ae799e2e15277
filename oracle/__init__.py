"""CPU oracle for the Allegro per-edge hot path.  TEST INFRASTRUCTURE ONLY.

This package is a plain-PyTorch/numpy restatement of the reference algorithm
(mir-group/allegro v0.7.1, files cited per function) plus the un-vendored
arithmetic it depends on (e3nn: Wigner 3j, spherical harmonics, Irreps;
nequip: ScalarMLPFunction, scatter, Bessel/cutoff embedding, scale/shift).

Only ``tests/``, ``__graft_entry__.smoke()`` and the ``cpu_baseline`` /
``--impl reference`` legs of ``bench.py`` may import it.  The product package
``allegro_b200`` never imports it; its CUDA path raises if the extension is
missing instead of falling back here.

PARITY -- what is pinned and what is not:

* PINNED to the reference's own code: everything mir-group/allegro implements itself
  (allegro/nn/_strided/_contract.py, _channels.py, allegro/nn/_allegro.py, tensorembed.py,
  _edgeembed.py, scalarembed.py, edgewise.py and the assembly in allegro/model/allegro_models.py).
  ``tests/golden/make_reference_vectors.py`` EXECUTES those unmodified modules from a
  checkout of the reference and records inputs, state_dicts and outputs in
  ``tests/golden/ref_models_<k>.pt`` / ``ref_ops_<k>.pt``; ``tests/test_reference_golden.py`` checks this
  oracle against them (strict state_dict load, 1e-12 relative in fp64) on every box.
* PARITY UNPINNED for the third-party primitives those modules import: e3nn (wigner_3j,
  SphericalHarmonics, Irreps) and nequip (ScalarMLPFunction, Bessel/cutoff embedding,
  scale/shift, force output).  Neither package is installable in this image and the reference's
  tests hold no golden vectors for them (they compare with e3nn at run time,
  tests/nn/test_contract_basic.py:120-211, tests/nn/test_weighter.py:12-54), so while the
  fixtures above were generated the imports resolved to stand-ins backed by THIS oracle's
  restatements (tests/golden/_stubs/).  Independent implementations available in this image pin part
  of them: the spherical harmonics equal scipy's Y_l^m in the standard real basis with e3nn's axis
  convention (y polar), exactly and for every (l, m) up to l = 4, and the real Wigner 3j are
  proportional, triple by triple, to sympy's real Gaunt integrals (tests/test_oracle_o3.py).  What
  stays unpinned: the overall sign of each 3j block and the odd-sum blocks (absorbed by the path
  weights; matters only for loading trained checkpoints) and nequip's MLP normalisation constants.
  Beyond that the primitives are pinned only by the known-answer
  values and identities in ``tests/golden/o3_known_answers.json`` (SURVEY.md section 8c) and by
  the property tests the reference uses (equivariance, gradcheck, strict locality).
"""
