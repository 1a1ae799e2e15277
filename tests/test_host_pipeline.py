"""The product's HOST logic, end to end, on a CPU-only box.

The ctypes wrappers of the CUDA kernels (allegro_b200/_lib.py) are replaced by the executable specification in
tests/kernel_spec.py (what include/allegro_b200.h says each kernel computes, in torch), and the whole product path --
AllegroModel state_dict loading, weight folding / packing / column permutations, segment views, the forward and both
backward orchestrations, CSR and edge permutations, scale/shift, stress -- is compared with vectors produced by the
reference's own code (tests/golden/ref_models_<k>.pt).  A mismatch here is a bug in the Python side of the product (or in the
kernel contract), independent of any CUDA kernel; the kernels themselves are checked on the GPU.
"""
import pytest
import torch

import kernel_spec
from golden_util import load_models, model_case_ids, unpack_state_dict

MODELS = {r["name"]: r for r in load_models()}


@pytest.fixture()
def spec_kernels(monkeypatch):
    from allegro_b200 import _lib
    from allegro_b200.model.allegro_models import FusedAllegroEnergy
    from allegro_b200.nn._pipeline import AllegroCore, UpstreamPack

    for name in kernel_spec.ALL:
        monkeypatch.setattr(_lib, name, getattr(kernel_spec, name))

    def core(self):  # FusedAllegroEnergy.core without the "must live on a CUDA device" gate
        return self._core_for(torch.device("cpu"))

    monkeypatch.setattr(FusedAllegroEnergy, "core", core)


def _rel(a, b):
    a, b = a.detach().double(), b.detach().double()
    assert a.shape == b.shape, (a.shape, b.shape)
    if b.numel() == 0:
        return 0.0
    den = float(b.abs().max())
    return float((a - b).abs().max()) / (den if den > 0 else 1.0)


def _run(name, stress=True):
    from allegro_b200.model import AllegroModel

    rec = MODELS[name]
    model = AllegroModel(**rec["kwargs"])
    model.load_state_dict(unpack_state_dict(rec["state_dict"]), strict=True)
    return rec, model.model._energy_and_forces(dict(rec["data"]), stress)


@pytest.mark.parametrize("fold", ["1", "0"], ids=["fold", "nofold"])
@pytest.mark.parametrize("name", model_case_ids())
def test_host_pipeline_reproduces_reference(name, fold, spec_kernels, monkeypatch):
    monkeypatch.setenv("ALLEGRO_B200_FOLD_EMBED", fold)
    rec, out = _run(name)
    tol = 1e-10 if rec["kwargs"]["model_dtype"] == "float64" else 5e-5
    for key in ("atomic_energy", "forces", "edge_energy", "edge_features", "total_energy"):
        if key in rec:
            assert _rel(out[key], rec[key]) < tol, (key, _rel(out[key], rec[key]))


@pytest.mark.parametrize("env", [{"ALLEGRO_B200_FOLD_RADIAL": "0"}, {"ALLEGRO_B200_RADIAL_PQ": "0"}, {"ALLEGRO_B200_FOLD_RADIAL": "0", "ALLEGRO_B200_FOLD_EMBED": "0"}],
                         ids=["pq_nofold", "product_embed_kernel", "pq_nofold_noembedfold"])
@pytest.mark.parametrize("name", ["c2_lmax2_L2", "c5_lmax3_L3_5species", "per_edge_type_cutoff"])
def test_host_pipeline_radial_variants(name, env, spec_kernels, monkeypatch):
    """The upstream scalar track with the first MLP layer folded into the radial kernel (default), with the per-type-pair
    kernel but no fold, and with the round-1 product-embedding kernel: same energies and forces."""
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    rec, out = _run(name)
    assert _rel(out["forces"], rec["forces"]) < 1e-10 and _rel(out["atomic_energy"], rec["atomic_energy"]) < 1e-10


@pytest.mark.parametrize("name", ["c2_lmax2_L2", "c5_lmax3_L3_5species", "shared_irrep_weights", "spline_embed_reftest_cfg"])
def test_host_pipeline_plain_backward_plan(name, spec_kernels, monkeypatch):
    """The alternative backward orchestration (producer-side SiLU', concat-K block gradients) gives the same forces."""
    monkeypatch.setenv("ALLEGRO_B200_PLAIN_BWD", "1")
    rec, out = _run(name)
    assert _rel(out["forces"], rec["forces"]) < 1e-10


def test_host_pipeline_stress_matches_oracle(spec_kernels):
    from oracle.model_ref import AllegroOracle

    rec, out = _run("c5_lmax3_L3_5species", stress=True)
    oracle = AllegroOracle(**rec["kwargs"])
    oracle.load_state_dict(unpack_state_dict(rec["state_dict"]), strict=True)
    ref = oracle(dict(rec["data"]))
    assert _rel(out["stress"], ref["stress"]) < 1e-10 and _rel(out["virial"], ref["virial"]) < 1e-10
    _, out2 = _run("c5_lmax3_L3_5species", stress=False)
    assert "stress" not in out2


def test_host_pipeline_under_the_md_driver(spec_kernels, monkeypatch):
    """AllegroCalculator (Verlet skin list, eager mode) driving the product model: equals the reference-pinned oracle on
    exact r_max lists along a short random walk, including the stress."""
    from allegro_b200 import data as D
    from allegro_b200.calculator import AllegroCalculator
    from allegro_b200.model import AllegroModel
    from allegro_b200.model.allegro_models import FusedAllegroEnergy
    from oracle.model_ref import AllegroOracle

    monkeypatch.setattr(FusedAllegroEnergy, "energy_and_forces", lambda self, data, stress=False: self._energy_and_forces(data, stress))
    rec = MODELS["per_edge_type_cutoff"]
    sd = unpack_state_dict(rec["state_dict"])
    model = AllegroModel(**rec["kwargs"])
    model.load_state_dict(sd, strict=True)
    oracle = AllegroOracle(**rec["kwargs"])
    oracle.load_state_dict(sd, strict=True)
    d = rec["data"]
    pos, cell, types = d[D.POSITIONS_KEY], d[D.CELL_KEY], d[D.ATOM_TYPE_KEY]
    calc = AllegroCalculator(model, rec["kwargs"]["r_max"], skin=0.5, use_graph=False, compute_stress=True)
    g = torch.Generator().manual_seed(8)
    p = pos.clone()
    for _ in range(3):
        out = calc.compute(p, cell, types)
        ei, sh = D.neighbor_list(p, rec["kwargs"]["r_max"], cell, (True, True, True))
        ref = oracle({D.POSITIONS_KEY: p, D.CELL_KEY: cell, D.ATOM_TYPE_KEY: types, D.EDGE_INDEX_KEY: ei, D.EDGE_CELL_SHIFT_KEY: sh})
        assert _rel(out["forces"], ref["forces"]) < 1e-10
        assert _rel(out["atomic_energy"], ref["atomic_energy"]) < 1e-10
        assert _rel(out["stress"], ref["stress"]) < 1e-10
        p = p + 0.1 * torch.randn(p.shape, generator=g, dtype=p.dtype)
    assert calc.n_rebuilds >= 1 and calc.n_evaluations == 3


@pytest.mark.parametrize("plain", [False, True], ids=["legacy_bwd", "plain_bwd"])
@pytest.mark.parametrize("name", model_case_ids())
def test_host_pipeline_with_folded_embed_linears(name, plain, spec_kernels, monkeypatch):
    """ALLEGRO_B200_FOLD_EMBED=1: the two linear maps that consume the two-body embedding are folded into the last layer
    of the scalar-embed MLP (one GEMM less per direction).  Same energies, forces and per-edge outputs."""
    monkeypatch.setenv("ALLEGRO_B200_FOLD_EMBED", "1")
    if plain:
        monkeypatch.setenv("ALLEGRO_B200_PLAIN_BWD", "1")
    rec, out = _run(name)
    tol = 1e-10 if rec["kwargs"]["model_dtype"] == "float64" else 5e-5
    for key in ("atomic_energy", "forces", "edge_energy", "edge_features"):
        if key in rec:
            assert _rel(out[key], rec[key]) < tol, (key, _rel(out[key], rec[key]))


def test_prepared_csr_with_owned_centres_only(spec_kernels):
    """A prepared CSR may hold rows for the first n_c atoms only (the owned centres of a slab; neighbours index owned + ghost
    atoms, halo.py / _compile.py:41-61): energies come back for those centres, forces for every atom.  Reference: the oracle on
    the same frame restricted to the edges centred on the first n_c atoms (strict locality makes that the same function).
    Regression test for the multi-GPU path (r2k: the scale/shift was applied with the types of ALL atoms)."""
    from allegro_b200 import data as D
    from allegro_b200 import systems
    from allegro_b200.model import AllegroModel
    from oracle.model_ref import AllegroOracle

    d = systems.make_system("c3", 3)
    n = d[D.POSITIONS_KEY].shape[0]
    nc = 17
    ei, sh = d[D.EDGE_INDEX_KEY], d[D.EDGE_CELL_SHIFT_KEY]
    keep = ei[0] < nc
    kw = systems.model_kwargs("c3", ei.shape[1] / n, "float64")
    kw.update(num_scalar_features=16, num_tensor_features=8, radial_chemical_embed_dim=16, scalar_embed_mlp_hidden_layers_width=16,
              allegro_mlp_hidden_layers_width=16, readout_mlp_hidden_layers_width=16, per_type_energy_scales=[0.7, 1.3, 0.9],
              per_type_energy_shifts=[0.1, -0.2, 0.3])
    oracle = AllegroOracle(**kw)
    model = AllegroModel(**kw)
    model.load_state_dict(oracle.state_dict())
    d_sub = dict(d)
    d_sub[D.EDGE_INDEX_KEY], d_sub[D.EDGE_CELL_SHIFT_KEY] = ei[:, keep].contiguous(), sh[keep].contiguous()
    ref = oracle(d_sub)
    csr = D.build_csr(d_sub[D.EDGE_INDEX_KEY], nc)
    assert csr.perm is None and csr.num_atoms == nc
    shift_vec = d_sub[D.EDGE_CELL_SHIFT_KEY].double() @ d[D.CELL_KEY].view(3, 3)
    data = {D.POSITIONS_KEY: d[D.POSITIONS_KEY], D.ATOM_TYPE_KEY: d[D.ATOM_TYPE_KEY], D.CELL_KEY: d[D.CELL_KEY], D.CSR_KEY: csr,
            D.EDGE_SHIFT_VEC_KEY: shift_vec}
    out = model.model._energy_and_forces(data, False)
    assert out[D.PER_ATOM_ENERGY_KEY].shape[0] == nc and out[D.FORCE_KEY].shape[0] == n
    assert _rel(out[D.PER_ATOM_ENERGY_KEY], ref[D.PER_ATOM_ENERGY_KEY][:nc]) < 1e-10
    assert _rel(out[D.FORCE_KEY], ref[D.FORCE_KEY]) < 1e-10
