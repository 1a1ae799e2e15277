"""Oracle and product host logic against vectors produced by the REFERENCE'S OWN CODE.

tests/golden/ref_models_<k>.pt / ref_ops_<k>.pt were written by tests/golden/make_reference_vectors.py, which
executes the reference's unmodified allegro/nn + allegro/model modules (third-party e3nn / nequip
calls resolved to stand-ins backed by the oracle's primitives, tests/golden/_stubs/README.md).  These
tests therefore pin the oracle's restatement -- and the product's table / irreps / state_dict logic --
to the reference implementation itself, on every machine (no reference checkout needed at test time).

fp64 cases must agree to rounding (1e-12 relative), the fp32 case to 1e-5.
"""
import pytest
import torch

from golden_util import load_models, load_ops, model_case_ids, unpack_state_dict
from oracle import nn_ref as R
from oracle.model_ref import AllegroOracle
from oracle.o3_ref import Irreps as OIrreps

MODELS = {r["name"]: r for r in load_models()}
OPS = load_ops()


def _rel(a, b):
    a, b = a.detach().double(), b.detach().double()
    assert a.shape == b.shape, (a.shape, b.shape)
    if b.numel() == 0:
        return 0.0
    den = float(b.abs().max())
    return float((a - b).abs().max()) / (den if den > 0 else 1.0)  # all-zero reference (isolated atoms): absolute error


# ---------------------------------------------------------------------------------------
# whole model: oracle == reference
# ---------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", model_case_ids())
def test_oracle_reproduces_reference_model(name):
    rec = MODELS[name]
    oracle = AllegroOracle(**rec["kwargs"])
    res = oracle.load_state_dict(unpack_state_dict(rec["state_dict"]), strict=True)  # same keys, same shapes
    assert not res.missing_keys and not res.unexpected_keys
    out = oracle(dict(rec["data"]))
    tol = 1e-12 if rec["kwargs"]["model_dtype"] == "float64" else 1e-5
    for key in ("total_energy", "atomic_energy", "forces", "edge_energy", "edge_features"):
        if key in rec:
            assert out[key].shape == rec[key].shape, key
            assert _rel(out[key], rec[key]) < tol, (key, _rel(out[key], rec[key]))
    # module order of the reference's SequentialGraphNetwork (allegro_models.py:222-297)
    assert rec["modules"] == ["edge_norm", "radial_chemical_embed", "scalar_embed_mlp", "tensor_embed", "allegro", "edge_readout",
                              "edge_eng_sum", "per_type_energy_scale_shift", "total_energy_sum"]


@pytest.mark.parametrize("name", model_case_ids())
def test_product_model_accepts_reference_state_dict(name):
    """The product's parameter holders have the reference's state_dict: keys, shapes, and an identical
    dense w3j buffer built by the product's own Wigner-3j code (no kernels involved)."""
    from allegro_b200.model import AllegroModel

    rec = MODELS[name]
    model = AllegroModel(**rec["kwargs"])
    own = {k: v.clone() for k, v in model.state_dict().items()}
    sd = unpack_state_dict(rec["state_dict"])
    res = model.load_state_dict(sd, strict=True)
    assert not res.missing_keys and not res.unexpected_keys
    for k, v in sd.items():
        if k.endswith("w3j"):
            assert own[k].shape == v.shape
            assert (own[k].double() - v.double()).abs().max() < (1e-12 if v.dtype == torch.float64 else 1e-6), k
    tps = model.model.allegro.tps
    assert [(repr(tp.irreps_in1), repr(tp.irreps_in2), repr(tp.irreps_out), tp.num_paths) for tp in tps] == [tuple(t) for t in rec["tp_irreps"]]


# ---------------------------------------------------------------------------------------
# layer irreps build + pruning (allegro/nn/_allegro.py:101-160) and table sizes
# ---------------------------------------------------------------------------------------
@pytest.mark.parametrize("case", OPS["layers"], ids=lambda c: f"l{c['lmax']}_{'p' if c['parity'] else 'np'}_L{c['num_layers']}")
def test_layer_irreps_and_tables_match_reference(case):
    from allegro_b200 import o3

    lmax, L = case["lmax"], case["num_layers"]
    sh = o3.Irreps.spherical_harmonics(lmax)
    allowed = o3.Irreps([(1, (l, p)) for l in range(lmax + 1) for p in (1, -1)]) if case["parity"] else sh
    for mod, IR in ((o3, o3.Irreps), (R, OIrreps)):  # product host code and oracle
        shm = IR.spherical_harmonics(lmax)
        alm = IR([(1, (l, p)) for l in range(lmax + 1) for p in (1, -1)]) if case["parity"] else shm
        ins, outs = mod.allegro_layer_irreps(shm, alm, L)
        assert len(ins) == L
        for (i1, i2, io, n_paths, nnz, diag), a, b in zip(case["tps"], ins, outs):
            assert (repr(a), repr(shm), repr(b)) == (i1, i2, io)
    ins, outs = o3.allegro_layer_irreps(sh, allowed, L)
    for (i1, i2, io, n_paths, nnz, diag), a, b in zip(case["tps"], ins, outs):
        tab = o3.build_coupling_table(a, sh, b, None, "component")
        assert tab.num_paths == n_paths
        assert len(tab.entries) == nnz
        assert bool(tab.is_ij_diagonal) == diag
    # latent MLP shapes: [S(l+1)+U] -> W -> [S + n_ir U (not in the last layer)]   (_allegro.py:192-213)
    S, U, n_ir = 4, 2, lmax + 1
    for layer, dims in enumerate(case["latent_dims"]):
        assert dims[0] == S * (layer + 1) + U
        assert dims[-1] == S + (n_ir * U if layer < L - 1 else 0)


# ---------------------------------------------------------------------------------------
# operators: Contracter (forward + both input gradients) and MakeWeightedChannels
# ---------------------------------------------------------------------------------------
def _contracter_kwargs(c):
    return dict(irreps_in1=c["irreps_in1"], irreps_in2=c["irreps_in2"], irreps_out=c["irreps_out"], mul=c["mul"],
                instructions=c["instructions"], path_channel_coupling=c["path_channel_coupling"], scatter_factor=c["scatter_factor"])


@pytest.mark.parametrize("i", range(len(OPS["contracter"])))
def test_oracle_contracter_matches_reference(i):
    c = OPS["contracter"][i]
    prev = torch.get_default_dtype()
    torch.set_default_dtype(torch.float64)
    try:
        tp = R.Contracter(**_contracter_kwargs(c))
    finally:
        torch.set_default_dtype(prev)
    assert tp.num_paths == c["num_paths"] and bool(tp.w3j_is_ij_diagonal) == c["w3j_is_ij_diagonal"]
    own_w3j = tp.w3j.clone()
    sd = unpack_state_dict(c["state_dict"])
    tp.load_state_dict(sd, strict=True)
    assert (own_w3j - sd["w3j"]).abs().max() < 1e-12  # the oracle's own table == the reference's buffer
    x1, x2 = c["x1"].clone().requires_grad_(True), c["x2"].clone().requires_grad_(True)
    out = tp(x1, x2, c["idx"], c["n_atoms"])
    assert _rel(out, c["out"]) < 1e-12
    g1, g2 = torch.autograd.grad(out, (x1, x2), c["gout"])
    assert _rel(g1, c["gx1"]) < 1e-12 and _rel(g2, c["gx2"]) < 1e-12


@pytest.mark.parametrize("i", range(len(OPS["contracter"])))
def test_product_contracter_tables_match_reference(i):
    """allegro_b200.nn.Contracter (the kernel plug-in): same w3j buffer, weight shape and path count as the
    reference module, and the sparse kernel table x weights reproduces the reference's dense ww3j."""
    from allegro_b200.nn import Contracter

    c = OPS["contracter"][i]
    prev = torch.get_default_dtype()
    torch.set_default_dtype(torch.float64)
    try:
        tp = Contracter(**_contracter_kwargs(c))
    finally:
        torch.set_default_dtype(prev)
    sd = unpack_state_dict(c["state_dict"])
    assert (tp.w3j.double() - sd["w3j"]).abs().max() < 1e-12
    tp.load_state_dict(sd, strict=True)
    assert tp.num_paths == c["num_paths"] and bool(tp.w3j_is_ij_diagonal) == c["w3j_is_ij_diagonal"]
    # dense ww3j[u][i][j][k] as the reference forms it (_contract.py:213-222) from its own buffers ...
    w3j, w = sd["w3j"], sd["weights"]
    P, U = c["num_paths"], c["mul"]
    w3j_p = w3j if P > 1 else w3j.unsqueeze(0)
    if c["w3j_is_ij_diagonal"]:
        full = torch.zeros(P, tp.base_dim1, tp.base_dim2, tp.base_dim_out, dtype=torch.float64)
        ii = torch.arange(tp.base_dim1)
        full[:, ii, ii, :] = w3j_p
        w3j_p = full
    wp = w if P > 1 else w.unsqueeze(-1)
    wp = wp if c["path_channel_coupling"] else wp.unsqueeze(0).expand(U, P)
    dense = torch.einsum("up,pijk->uijk", wp, w3j_p)
    # ... equals the scatter of the product's sorted sparse table times cgw (what the kernels consume)
    ijk, _, _ = tp.sparse_table()
    cgw = tp.cgw(torch.float64, "cpu")  # [nnz][U]
    mine = torch.zeros_like(dense)
    for n, (a, b, k) in enumerate(ijk.tolist()):
        mine[:, a, b, k] += cgw[n]
    assert (mine - dense).abs().max() < 1e-12
    keys = [(a, k, b) for a, b, k in ijk.tolist()]
    assert keys == sorted(keys)  # (i, k, j) order required by ab2_tp_fwd


@pytest.mark.parametrize("i", range(len(OPS["channels"])))
def test_oracle_weighted_channels_match_reference(i):
    c = OPS["channels"][i]
    m = R.MakeWeightedChannels(OIrreps.spherical_harmonics(c["lmax"]), c["mul"], weight_individual_irreps=c["weight_individual_irreps"])
    assert m.weight_numel == c["weight_numel"]
    assert _rel(m(c["edge_attr"], c["weights"]), c["out"]) < 1e-12


def test_shared_irrep_weights_column_replication():
    """weight_individual_irreps=False on the kernels = individual weights with the U columns replicated over the
    irreps (nn/_pipeline.py:_env_perm): checked against the reference's MakeWeightedChannels output."""
    from allegro_b200.nn._pipeline import _env_perm

    c = [c for c in OPS["channels"] if not c["weight_individual_irreps"]][0]
    U, n_ir = c["mul"], c["lmax"] + 1
    perm = _env_perm(U, n_ir, individual=False)
    w_int = c["weights"][:, perm].view(-1, n_ir, U)  # internal layout w[z][r][u]
    Y = c["edge_attr"]
    out = torch.empty(Y.shape[0], U, Y.shape[1], dtype=Y.dtype)
    for l in range(n_ir):
        out[:, :, l * l : (l + 1) * (l + 1)] = Y[:, None, l * l : (l + 1) * (l + 1)] * w_int[:, l, :, None]
    assert _rel(out, c["out"]) < 1e-12
    # and the individual-weight gather is the [u][r] -> [r][u] transpose
    ci = [c for c in OPS["channels"] if c["weight_individual_irreps"] and c["lmax"] == 2][0]
    U, n_ir = ci["mul"], 3
    w_int = ci["weights"][:, _env_perm(U, n_ir)].view(-1, n_ir, U)
    assert torch.equal(w_int, ci["weights"].view(-1, U, n_ir).transpose(1, 2))


def test_product_spline_embedding_matches_reference_weights_and_oracle_gradient():
    """allegro_b200/nn/_spline.py (device-agnostic torch ops, hand-written adjoint) with the reference's spline weights:
    forward == the reference-pinned oracle module, adjoint == autograd through it; includes edges beyond the cutoff."""
    from allegro_b200.nn import TwoBodySplineScalarEmbed
    from allegro_b200.nn._spline import spline_backward, spline_forward

    rec = MODELS["spline_embed_per_edge_type_cutoff"]
    sd = {k[len("model.radial_chemical_embed."):]: v for k, v in unpack_state_dict(rec["state_dict"]).items() if "radial_chemical_embed" in k}
    names = rec["kwargs"]["type_names"]
    cfg = dict(rec["kwargs"]["radial_chemical_embed"])
    cfg.pop("_target_")
    S = rec["kwargs"]["num_scalar_features"]
    mine = TwoBodySplineScalarEmbed(names, module_output_dim=S, **cfg)
    mine.load_state_dict(sd, strict=True)
    ora = R.TwoBodySplineScalarEmbed(names, module_output_dim=S, **cfg)
    ora.load_state_dict(sd, strict=True)
    g = torch.Generator().manual_seed(0)
    E, T = 500, len(names)
    vec = torch.randn(E, 3, generator=g, dtype=torch.float64) * 2.2  # lengths 0..~8 A: inside and beyond r_max = 4
    tc, tn = torch.randint(0, T, (E,), generator=g), torch.randint(0, T, (E,), generator=g)
    rmax = torch.full((T, T), 4.0, dtype=torch.float64)
    rmax[0, :] = 2.0
    rmax[1, 0], rmax[1, 1], rmax[1, 2] = 4.0, 3.5, 3.7
    sp = mine.spline
    e0, saved = spline_forward(vec, tc, tn, rmax, sp.lower, sp.upper, sp._const, sp.flat_weights(), T, torch.float64)
    v = vec.clone().requires_grad_(True)
    x = (v.norm(dim=-1) / rmax[tc, tn]).unsqueeze(-1)
    ref = ora({R.NORM_LENGTH_KEY: x, R.EDGE_TYPE_KEY: torch.stack([tc, tn])}, torch.float64)[R.EDGE_EMBEDDING_KEY]
    assert _rel(e0, ref) < 1e-13
    assert float(e0[(x.squeeze(-1) >= 1.0).detach()].abs().max()) == 0.0  # beyond the cutoff: exactly zero
    gout = torch.randn(ref.shape, generator=g, dtype=torch.float64)
    (gv,) = torch.autograd.grad(ref, v, gout)
    assert _rel(spline_backward(saved, gout, sp.flat_weights(), T), gv) < 1e-12
    # module forward used by the torch-autograd path of the product model
    out = mine(x.detach().squeeze(-1), tc, tn, torch.float32)
    assert out.dtype == torch.float32 and _rel(out, ref) < 1e-6
