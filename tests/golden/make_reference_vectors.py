"""Generate golden vectors by EXECUTING THE REFERENCE'S OWN CODE (needs a checkout of the reference).

    python tests/golden/make_reference_vectors.py REFERENCE_CHECKOUT

What runs: the unmodified `allegro/nn/*.py` and `allegro/model/allegro_models.py` from a checkout
of mir-group/allegro v0.7.1.  Its third-party imports (e3nn, nequip, hydra) are not
installable in this image, so they resolve to the stand-ins under `tests/golden/_stubs/`, which
forward to the oracle's restatements of the published algorithms (see `_stubs/README.md` for
exactly what that does and does not pin).  The reference's package `__init__` (which pulls in the
nequip-compile tooling) is bypassed by registering a bare parent package; every `allegro.nn` /
`allegro.model` module is executed as is.

Outputs (committed; each collection is split over numbered files below MAX_FILE_BYTES,
tests/golden_util.py joins them):
  tests/golden/ref_models_<k>.pt   whole-model cases: ctor kwargs, inputs, reference state_dict, outputs
  tests/golden/ref_ops_<k>.pt      operator cases: Contracter / MakeWeightedChannels inputs+outputs,
                                   per-layer irreps of Allegro_Module for a grid of (l_max, parity, L),
                                   and a reference model's Contracters as enable_B200Contracter sees them
"""
import io
import os
import sys
import types

import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
MAX_FILE_BYTES = 900_000
sys.path.insert(0, os.path.join(HERE, "_stubs"))
sys.path.insert(0, ROOT)

REF = sys.argv[1] if len(sys.argv) > 1 else ""
if not os.path.isdir(os.path.join(REF, "allegro")):
    sys.exit("usage: make_reference_vectors.py REFERENCE_CHECKOUT (a mir-group/allegro v0.7.1 source tree)")
_pkg = types.ModuleType("allegro")
_pkg.__path__ = [os.path.join(REF, "allegro")]
sys.modules["allegro"] = _pkg

import allegro.model  # noqa: E402  (reference code)
import allegro.nn  # noqa: E402  (reference code)
from allegro.nn._strided import Contracter, MakeWeightedChannels  # noqa: E402  (reference code)
from e3nn.o3 import Irreps  # noqa: E402  (stand-in)

from allegro_b200 import data as D  # noqa: E402
from allegro_b200 import systems  # noqa: E402

BESSEL = {"_target_": "allegro.nn.TwoBodyBesselScalarEmbed", "num_bessels": 8, "polynomial_cutoff_p": 6}


def pack_state_dict(sd):
    """Dense `w3j` buffers (mostly zeros, MBs at l_max=3) are stored as (shape, indices, values);
    tests/test_reference_golden.py::unpack_state_dict restores them exactly."""
    out = {}
    for k, v in sd.items():
        if k.endswith("w3j"):
            nz = v.nonzero()
            out[k] = {"w3j_shape": tuple(v.shape), "idx": nz.to(torch.int16), "val": v[tuple(nz.T)].clone(), "dtype": v.dtype}
        else:
            out[k] = v.clone()
    return out


def save_parts(stem, collections):
    """Write ``collections`` (a dict of lists) as <stem>_1.pt, <stem>_2.pt, ...: records are taken in order and a
    new file is started before one would exceed MAX_FILE_BYTES.  Returns the file names."""
    def size(part):
        buf = io.BytesIO()
        torch.save(part, buf)
        return buf.tell()

    parts = [{}]
    for key, records in collections.items():
        for rec in records:
            trial = {k: list(v) for k, v in parts[-1].items()}
            trial.setdefault(key, []).append(rec)
            if parts[-1] and size(trial) > MAX_FILE_BYTES:
                parts.append({key: [rec]})
            else:
                parts[-1] = trial
    names = []
    for k, part in enumerate(parts, 1):
        assert size(part) <= MAX_FILE_BYTES, f"one {stem} record alone exceeds {MAX_FILE_BYTES} bytes"
        names.append(f"{stem}_{k}.pt")
        torch.save(part, os.path.join(HERE, names[-1]))
    return names


def _cluster(n, box, seed):
    """Open-boundary cluster, edges in shuffled (not centre-sorted) order."""
    g = torch.Generator().manual_seed(seed)
    pos = torch.rand(n, 3, generator=g, dtype=torch.float64) * box
    types = torch.randint(0, 2, (n,), generator=g)
    ei, _ = D.neighbor_list(pos, 3.5, None, (False, False, False))
    perm = torch.randperm(ei.shape[1], generator=g)
    return {D.POSITIONS_KEY: pos, D.ATOM_TYPE_KEY: types, D.EDGE_INDEX_KEY: ei[:, perm].contiguous()}


def model_cases():
    small = dict(num_scalar_features=16, num_tensor_features=8, radial_chemical_embed_dim=16, scalar_embed_mlp_hidden_layers_width=16,
                 allegro_mlp_hidden_layers_width=16, readout_mlp_hidden_layers_width=8)
    cases = []

    def add(name, data, dtype="float64", **kw):
        n, e = data[D.POSITIONS_KEY].shape[0], data[D.EDGE_INDEX_KEY].shape[1]
        base = dict(seed=7 + len(cases), model_dtype=dtype, radial_chemical_embed=dict(BESSEL), avg_num_neighbors=e / n)
        base.update(kw)
        cases.append((name, base, data))

    c1 = systems.make_system("c1", 1)  # 8-atom Si cell, r_max 4
    add("c1_lmax1_L1", c1, type_names=["Si"], r_max=4.0, l_max=1, num_layers=1, **small)
    c2 = systems.make_system("c2", 2)  # 32-atom Cu FCC, r_max 5
    add("c2_lmax2_L2", c2, type_names=["Cu"], r_max=5.0, l_max=2, num_layers=2, **small)
    add("c2_lmax2_L2_f32", c2, dtype="float32", type_names=["Cu"], r_max=5.0, l_max=2, num_layers=2, **small)
    add("c2_arch_S64_U32", c2, type_names=["Cu"], r_max=5.0, l_max=2, num_layers=2, num_scalar_features=64, num_tensor_features=32,
        radial_chemical_embed_dim=64, scalar_embed_mlp_hidden_layers_width=64, allegro_mlp_hidden_layers_width=64,
        readout_mlp_hidden_layers_width=64)
    add("noparity_lmax2_L2", c2, type_names=["Cu"], r_max=5.0, l_max=2, num_layers=2, parity=False, **small)
    add("shared_paths_lmax2_L3", c2, type_names=["Cu"], r_max=5.0, l_max=2, num_layers=3, tp_path_channel_coupling=False, **small)
    add("shared_irrep_weights", c2, type_names=["Cu"], r_max=5.0, l_max=2, num_layers=2, weight_individual_irreps=False, **small)
    add("deep_mlps_nolatent_nonlin", c2, type_names=["Cu"], r_max=5.0, l_max=1, num_layers=2, allegro_mlp_hidden_layers_depth=2,
        scalar_embed_mlp_hidden_layers_depth=0, readout_mlp_hidden_layers_depth=0, **small)
    c5 = systems.make_system("c5", 2)  # 32 atoms, 5 species
    add("c5_lmax3_L3_5species", c5, type_names=["A", "B", "C", "D", "E"], r_max=5.0, l_max=3, num_layers=3,
        per_type_energy_scales=[1.0, 0.5, 2.0, 1.5, 0.25], per_type_energy_shifts=[0.1, -0.2, 0.3, 0.0, 1.0], **small)
    add("per_edge_type_cutoff", c5, type_names=["A", "B", "C", "D", "E"], r_max=5.0, l_max=2, num_layers=2,
        per_edge_type_cutoff={"A": 4.0, "B": {"A": 3.5, "B": 4.5, "C": 5.0, "D": 5.0, "E": 4.0}}, **small)
    add("cluster_open_unsorted", _cluster(20, 6.0, 3), type_names=["X", "Y"], r_max=3.5, l_max=2, num_layers=2, **small)
    # ragged / empty inputs: atoms without any neighbour in the middle of the index range, and a frame with no edge at all
    cl = _cluster(22, 6.0, 5)
    far = torch.tensor([[90.0, 0, 0], [0, 95.0, 0], [0, 0, 99.0]], dtype=torch.float64)
    pos = torch.cat([cl[D.POSITIONS_KEY][:4], far[:1], cl[D.POSITIONS_KEY][4:15], far[1:2], cl[D.POSITIONS_KEY][15:], far[2:]], 0)
    types = torch.cat([cl[D.ATOM_TYPE_KEY][:4], torch.tensor([1]), cl[D.ATOM_TYPE_KEY][4:15], torch.tensor([0]), cl[D.ATOM_TYPE_KEY][15:], torch.tensor([1])])
    ei, _ = D.neighbor_list(pos, 3.5, None, (False, False, False))
    ragged = {D.POSITIONS_KEY: pos, D.ATOM_TYPE_KEY: types, D.EDGE_INDEX_KEY: ei}
    add("isolated_atoms_ragged_rows", ragged, type_names=["X", "Y"], r_max=3.5, l_max=2, num_layers=2, avg_num_neighbors=9.0,
        per_type_energy_shifts=[0.5, -1.0], **small)
    ei0, _ = D.neighbor_list(far, 3.5, None, (False, False, False))
    assert ei0.shape[1] == 0
    add("no_edges_at_all", {D.POSITIONS_KEY: far, D.ATOM_TYPE_KEY: torch.tensor([0, 1, 1]), D.EDGE_INDEX_KEY: ei0}, type_names=["X", "Y"],
        r_max=3.5, l_max=2, num_layers=2, avg_num_neighbors=9.0, per_type_energy_shifts=[0.5, -1.0], **small)
    # the reference's own model-test configuration (tests/model/test_allegro.py:27-44: 3 types, r_max 4, avgN 20, L 2,
    # l_max 2, S 32, U 4, latent depth 2) with the SPLINE two-body embedding (:76-117 grid), with and without
    # per-edge-type cutoffs
    c3 = systems.make_system("c3", 3)  # 27 atoms, 3 species, r_max 6 list ...
    ei, sh = D.neighbor_list(c3[D.POSITIONS_KEY], 4.0, c3[D.CELL_KEY], (True, True, True))  # ... re-listed at r_max 4
    c3 = dict(c3)
    c3[D.EDGE_INDEX_KEY], c3[D.EDGE_CELL_SHIFT_KEY] = ei, sh
    ref_cfg = dict(type_names=["H", "C", "O"], r_max=4.0, l_max=2, num_layers=2, num_scalar_features=32, num_tensor_features=4,
                   allegro_mlp_hidden_layers_depth=2, allegro_mlp_hidden_layers_width=32, scalar_embed_mlp_hidden_layers_width=32,
                   readout_mlp_hidden_layers_width=8)
    spline = {"_target_": "allegro.nn.TwoBodySplineScalarEmbed", "num_splines": 8, "spline_span": 6}
    add("spline_embed_reftest_cfg", c3, radial_chemical_embed=dict(spline), **ref_cfg)
    add("spline_embed_per_edge_type_cutoff", c3, radial_chemical_embed=dict(spline), per_edge_type_cutoff={"H": 2.0, "C": {"H": 4.0, "C": 3.5, "O": 3.7}, "O": 3.9},
        tp_path_channel_coupling=False, **ref_cfg)
    add("spline_embed_f32", c3, dtype="float32", radial_chemical_embed=dict(spline), **ref_cfg)
    return cases


def run_models():
    out = []
    for name, kw, data in model_cases():
        model = allegro.model.AllegroModel(**kw)  # reference builder -> ForceStressOutput(SequentialGraphNetwork)
        res = model(dict(data))
        rec = {
            "name": name,
            "kwargs": kw,
            "data": data,
            "state_dict": pack_state_dict(model.state_dict()),
            "total_energy": res["total_energy"],
            "atomic_energy": res["atomic_energy"],
            "forces": res["forces"],
            "edge_energy": res["edge_energy"],
            "modules": [n for n, _ in model.model.named_children()],
            "tp_irreps": [(repr(tp.irreps_in1), repr(tp.irreps_in2), repr(tp.irreps_out), tp.num_paths) for tp in model.model.allegro.tps],
        }
        if res["edge_features"].numel() <= 10_000:
            rec["edge_features"] = res["edge_features"]
        out.append(rec)
        print(f"{name:28s} atoms {data['pos'].shape[0]:3d} edges {data['edge_index'].shape[1]:5d} E {float(res['total_energy']):+.6f} "
              f"max|F| {float(res['forces'].abs().max()):.4f}")
    return save_parts("ref_models", {"models": out})


def run_ops():
    torch.manual_seed(99)
    prev = torch.get_default_dtype()
    torch.set_default_dtype(torch.float64)
    contract = []
    sh = lambda l: repr(Irreps.spherical_harmonics(l))  # noqa: E731
    full = lambda l: "+".join(f"1x{k}{p}" for k in range(l + 1) for p in "eo")  # noqa: E731
    specs = [
        # (irreps_in1, irreps_in2, irreps_out, mul, instructions, path_channel_coupling, scatter_factor)
        (sh(1), sh(1), "1x0e", 4, None, True, None),
        (sh(2), sh(2), full(2), 8, None, True, 0.2),
        (full(2), sh(2), full(2), 8, None, True, 0.3),
        (full(2), sh(2), "1x0e", 8, None, False, 0.3),
        (full(3), sh(3), full(3), 3, None, True, 1.0),
        (sh(2), sh(2), "1x0e+1x1o+1x2e", 5, [(0, 0, 0), (1, 1, 0), (1, 2, 1), (2, 2, 2)], True, None),
        ("1x1o", "1x1o", "1x1e", 2, None, True, None),          # single path: weights (mul,)
        ("1x0e+1x1o", "1x0e+1x1o", "1x0e+1x1o", 6, [(0, 0, 0), (1, 1, 0)], False, 0.5),
        (sh(4), sh(4), "1x0e", 2, None, True, 0.1),
    ]
    g = torch.Generator().manual_seed(5)
    for i1, i2, io, mul, ins, pcc, sf in specs:
        tp = Contracter(irreps_in1=Irreps(i1), irreps_in2=Irreps(i2), irreps_out=Irreps(io), mul=mul, instructions=ins,
                        path_channel_coupling=pcc, scatter_factor=sf)
        n_atoms, n_edges = 7, 40
        idx = torch.randint(0, n_atoms, (n_edges,), generator=g)
        x1 = torch.randn(n_edges, mul, tp.base_dim1, generator=g)
        x2 = torch.randn(n_edges, mul, tp.base_dim2, generator=g)
        x1r, x2r = x1.clone().requires_grad_(True), x2.clone().requires_grad_(True)
        out = tp(x1r, x2r, idx, n_atoms)
        gout = torch.randn(out.shape, generator=g)
        g1, g2 = torch.autograd.grad(out, (x1r, x2r), gout)
        contract.append(dict(irreps_in1=i1, irreps_in2=i2, irreps_out=io, mul=mul, instructions=ins, path_channel_coupling=pcc,
                             scatter_factor=sf, state_dict=pack_state_dict(tp.state_dict()), idx=idx, n_atoms=n_atoms,
                             x1=x1, x2=x2, out=out.detach(), gout=gout, gx1=g1, gx2=g2, num_paths=tp.num_paths,
                             w3j_is_ij_diagonal=bool(tp.w3j_is_ij_diagonal)))
    channels = []
    for lmax, mul, wi in [(1, 4, True), (2, 8, True), (3, 3, True), (2, 5, False)]:
        ir = Irreps.spherical_harmonics(lmax)
        m = MakeWeightedChannels(irreps_in=ir, multiplicity_out=mul, weight_individual_irreps=wi)
        ea = torch.randn(11, ir.dim, generator=g)
        w = torch.randn(11, m.weight_numel, generator=g)
        channels.append(dict(lmax=lmax, mul=mul, weight_individual_irreps=wi, edge_attr=ea, weights=w, out=m(ea, w), weight_numel=m.weight_numel))
    layers = []
    for lmax in range(0, 5):
        for parity in (True, False):
            for L in (1, 2, 3, 4):
                sh_ir = Irreps.spherical_harmonics(lmax)
                allowed = Irreps([(1, (l, p)) for l in range(lmax + 1) for p in (1, -1)]) if parity else sh_ir
                am = allegro.nn.Allegro_Module(
                    num_layers=L, num_scalar_features=4, num_tensor_features=2, tensor_track_allowed_irreps=allowed, avg_num_neighbors=10.0,
                    irreps_in={"edge_attrs": sh_ir, "edge_features": sh_ir, "edge_embedding": Irreps("4x0e")})
                layers.append(dict(lmax=lmax, parity=parity, num_layers=L,
                                   tps=[(repr(tp.irreps_in1), repr(tp.irreps_in2), repr(tp.irreps_out), tp.num_paths,
                                         int((tp.w3j != 0).sum()), bool(tp.w3j_is_ij_diagonal)) for tp in am.tps],
                                   latent_dims=[tuple(int(w.shape[0]) for w in lat.weights) + (int(lat.weights[-1].shape[1]),) for lat in am.latents]))
    torch.set_default_dtype(prev)
    print(f"operators: {len(contract)} Contracter, {len(channels)} MakeWeightedChannels, {len(layers)} layer-irreps cases")
    return save_parts("ref_ops", dict(contracter=contract, channels=channels, layers=layers, modifier=[run_modifier()]))


def run_modifier():
    """A model assembled by the reference's builders, as allegro_b200's enable_B200Contracter finds it: the constructor
    state of every Contracter, the module tree and the state_dict (tests/test_reference_modifier.py)."""
    kw = dict(seed=3, model_dtype="float64", r_max=4.0, type_names=["H", "C", "O"], l_max=2, num_layers=3, num_scalar_features=16,
              num_tensor_features=4, avg_num_neighbors=20.0, radial_chemical_embed={"_target_": "allegro.nn.TwoBodyBesselScalarEmbed"})
    model = allegro.model.AllegroModel(**kw)
    tps = [dict(irreps_in1=repr(tp.irreps_in1), irreps_in2=repr(tp.irreps_in2), irreps_out=repr(tp.irreps_out), mul=tp.mul,
                instructions=tp.instructions, path_channel_coupling=tp.path_channel_coupling, scatter_factor=tp.scatter_factor,
                irrep_normalization=tp.irrep_normalization, num_paths=tp.num_paths, w3j_is_ij_diagonal=bool(tp.w3j_is_ij_diagonal))
           for tp in model.model.allegro.tps]
    return dict(kwargs=kw, tps=tps, state_dict=pack_state_dict(model.state_dict()),
                modules=[(name, type(m).__name__) for name, m in model.named_modules()])


if __name__ == "__main__":
    for f in run_models() + run_ops():
        print(f, os.path.getsize(os.path.join(HERE, f)) // 1024, "KiB")
