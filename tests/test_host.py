"""Host-side logic that needs no GPU: the module contract, the config surface, and that the C-ABI
library loads and exports every symbol include/voicesplit_b200.h declares."""
import ctypes
import json
import os
import re

import numpy as np
import pytest
import torch

from conftest import ROOT
from voicesplit_b200 import _cabi, config, synth


def _model(cls_name="VoiceSplit", dims=None):
    from models.voicefilter.model import VoiceFilter
    from models.voicesplit.model import VoiceSplit
    cls = {"VoiceSplit": VoiceSplit, "VoiceFilter": VoiceFilter}[cls_name]
    dims = dims or synth.make_dims(33, 16, 24, 40)
    return cls(config.AttrDict(synth.make_config_dict(dims))), dims


def test_state_dict_contract_native_shapes():
    # SURVEY.md section 8(b): keys/shapes of the shipped config (num_freq 601)
    m, dims = _model(dims=synth.make_dims())
    sd = m.state_dict()
    assert sd["conv.1.weight"].shape == (64, 1, 1, 7)
    assert sd["conv.5.weight"].shape == (64, 64, 7, 1)
    for i in (9, 13, 17, 21, 25):
        assert sd[f"conv.{i}.weight"].shape == (64, 64, 5, 5)
    assert sd["conv.28.weight"].shape == (8, 64, 1, 1)
    assert sd["conv.29.running_var"].shape == (8,)
    assert sd["conv.2.num_batches_tracked"].dtype == torch.int64
    assert sd["lstm.weight_ih_l0"].shape == (1600, 5064)
    assert sd["lstm.weight_hh_l0_reverse"].shape == (1600, 400)
    assert sd["fc1.weight"].shape == (600, 800) and sd["fc2.weight"].shape == (601, 600)
    assert sum(p.numel() for p in m.parameters()) == 18876001
    ref = synth.make_state_dict(dims)
    assert set(ref) == set(sd)


def _reference_layouts():
    # written by tests/golden/make_reference_checks_golden.py from the unmodified reference classes
    with open(os.path.join(ROOT, "tests", "golden", "reference_layouts.json")) as f:
        return json.load(f)


@pytest.mark.parametrize("name", ["VoiceSplit", "VoiceFilter"])
def test_state_dict_round_trips_with_reference_class(name):
    ref = _reference_layouts()[name]
    mine, dims = _model(name)
    assert ref["dims"] == [dims[k] for k in ("num_freq", "emb_dim", "lstm_dim", "fc1_dim")]
    msd = mine.state_dict()
    assert [k for k, _, _ in ref["state_dict"]] == list(msd.keys())
    for k, shape, dtype in ref["state_dict"]:
        assert tuple(msd[k].shape) == tuple(shape) and msd[k].dtype == getattr(torch, dtype), k
    # a state_dict laid out like the reference's loads strictly (reference checkpoint -> this repo); the way back needs exactly
    # the key / shape equality checked above
    rsd = {k: torch.zeros(shape, dtype=getattr(torch, dtype)) for k, shape, dtype in ref["state_dict"]}
    mine.load_state_dict(rsd, strict=True)
    # Adam can drive the parameters (train.py:34)
    opt = torch.optim.Adam(mine.parameters(), lr=1e-2)
    assert len(opt.param_groups[0]["params"]) == ref["n_parameters"]


def test_forward_refuses_cpu_and_train_mode():
    m, dims = _model()
    x, emb = synth.make_inputs(1, 4, dims)
    with pytest.raises(RuntimeError, match="no CPU"):
        m.eval()(torch.from_numpy(x), torch.from_numpy(emb))


def test_config_loader_strips_comments(tmp_path):
    p = tmp_path / "c.json"
    p.write_text('{\n "model_name":"voicesplit", // comment\n "model":{"lstm_dim": 400, // x\n "emb_dim": 256}\n}\n')
    c = config.load_config(str(p))
    assert c.model_name == "voicesplit" and c.model["lstm_dim"] == 400


def test_reference_config_json_builds_module():
    c = config.load_config(os.path.join(ROOT, "tests", "golden", "reference_config.json"))
    from models.voicesplit.model import VoiceSplit
    m = VoiceSplit(c)
    assert m.dims == synth.make_dims(601, 256, 400, 600, 601)
    # the restated loader reads the reference's own config.json to the same dict as the reference's load_config
    assert _reference_layouts()["config_json"] == dict(c)


def test_cabi_exports_every_declared_symbol():
    header = open(os.path.join(ROOT, "include", "voicesplit_b200.h")).read()
    body = re.sub(r"/\*.*?\*/", "", header, flags=re.S)
    declared = set(re.findall(r"\b(vs_[a-z0-9_]+)\s*\(", body))
    assert declared == set(_cabi.SIGNATURES), declared ^ set(_cabi.SIGNATURES)
    lib = _cabi.load()     # loads without a GPU (static cudart, driver entry points resolved lazily)
    for name in declared:
        assert hasattr(lib, name), name
    assert lib.vs_abi_version() == 2


def test_cabi_create_fails_loudly_without_gpu():
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    lib = _cabi.load()
    d = _cabi.VsDims(33, 16, 24, 40, 33, 0)
    h = ctypes.c_void_p()
    rc = lib.vs_engine_create(ctypes.byref(d), ctypes.byref(h))
    assert rc != 0 and lib.vs_last_error()


def test_synth_is_deterministic():
    d = synth.make_dims(33, 16, 24, 40)
    a, b = synth.make_state_dict(d, 3, "stress"), synth.make_state_dict(d, 3, "stress")
    assert all(np.array_equal(a[k], b[k]) for k in a)
    x1, e1 = synth.make_inputs(2, 5, d, 9)
    x2, e2 = synth.make_inputs(2, 5, d, 9)
    assert np.array_equal(x1, x2) and np.array_equal(e1, e2) and x1.min() >= 0 and x1.max() <= 1


def test_module_deepcopy_and_pickle_drop_the_engine_handle():
    import copy
    import pickle
    m, _ = _model()
    m._engine = object()          # stand-in for a live ctypes handle
    c = copy.deepcopy(m)
    assert c._engine is None and c._packed_sig is None
    r = pickle.loads(pickle.dumps(m))
    assert r._engine is None and list(r.state_dict()) == list(m.state_dict())
