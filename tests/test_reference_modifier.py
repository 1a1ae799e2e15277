"""The kernel plug-in point against a model assembled by the REFERENCE'S OWN builders.

`Contracter.enable_B200Contracter(model)` is the analogue of the reference's `enable_TritonContracter` /
`enable_CuEquivarianceContracter` model modifiers (allegro/nn/_strided/_contract.py:253-310).  The reference model
(seed 3, fp64, l_max 2, 3 layers) was built by tests/golden/make_reference_vectors.py, which recorded the constructor
state of its three Contracters, its module tree and its state_dict (tests/golden/ref_ops_<k>.pt, key "modifier").
Here the oracle's restatement of that model is loaded with the reference's state_dict and must hold the recorded
Contracters; after the modifier every Contracter must be the B200 operator with the reference's constructor state and
`state_dict`, and nothing else may change.  (The forward of the replaced operator needs a GPU:
tests/test_zx_gpu_reference_golden.py.)
"""
import pytest
import torch

from golden_util import load_ops, unpack_state_dict

REC = load_ops()["modifier"][0]
CTOR = ("irreps_in1", "irreps_in2", "irreps_out", "mul", "instructions", "path_channel_coupling", "scatter_factor", "irrep_normalization",
        "num_paths", "w3j_is_ij_diagonal")


def _ctor_state(tp):
    return {k: (repr(getattr(tp, k)).replace(" ", "") if k.startswith("irreps") else getattr(tp, k)) for k in CTOR}


def _expected(rec):
    return {k: (v.replace(" ", "") if k.startswith("irreps") else v) for k, v in rec.items()}


def test_enable_b200_contracter_on_reference_model():
    from allegro_b200.nn import B200Contracter
    from oracle.model_ref import AllegroOracle

    sd = unpack_state_dict(REC["state_dict"])
    model = AllegroOracle(**REC["kwargs"])
    res = model.load_state_dict(sd, strict=True)
    assert not res.missing_keys and not res.unexpected_keys
    old = list(model.model.allegro.tps)
    # the model holds the reference model's Contracters: same constructor state, same places in the module tree
    assert [_ctor_state(tp) for tp in old] == [_expected(t) for t in REC["tps"]]
    ref_tp_paths = [name for name, cls in REC["modules"] if cls == "Contracter"]
    assert [name for name, m in model.named_modules() if type(m).__name__ == "Contracter"] == ref_tp_paths

    def others():
        return [(name, type(m)) for name, m in model.named_modules() if not any(name == p or name.startswith(p + ".") for p in ref_tp_paths)]

    before_sd = {k: v.clone() for k, v in model.state_dict().items()}
    before_mods = others()
    out = B200Contracter.enable_B200Contracter(model)
    assert out is model
    new = list(model.model.allegro.tps)
    assert len(new) == len(old) and all(isinstance(tp, B200Contracter) for tp in new)
    for a, b, rec in zip(old, new, REC["tps"]):
        assert _ctor_state(b) == _expected(rec)
        assert b.w3j.dtype == a.w3j.dtype and torch.equal(b.w3j, a.w3j) and torch.equal(b.weights, a.weights)
    after = model.state_dict()
    assert list(after.keys()) == list(before_sd.keys())
    assert all(torch.equal(after[k], before_sd[k]) for k in before_sd)
    assert set(after) == set(sd) and all(torch.equal(after[k], sd[k]) for k in sd)  # the reference's state_dict, unchanged
    # every other module of the model is untouched
    assert others() == before_mods
    # the replaced operator refuses CPU tensors instead of silently falling back
    tp = new[0]
    with pytest.raises(RuntimeError):
        tp(torch.zeros(2, tp.mul, tp.base_dim1, dtype=torch.float64), torch.zeros(2, tp.mul, tp.base_dim2, dtype=torch.float64),
           torch.zeros(2, dtype=torch.long), 2)
