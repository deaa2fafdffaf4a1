"""CPU: the C-ABI library loads, exports every symbol include/saceo.h declares, answers layout queries without
a GPU, validates configurations like the reference does, and REFUSES to run without a device (no CPU fallback)."""
import ctypes as C
import os
import re

import pytest

import __graft_entry__ as G
from sac_expert_b200 import lib as L
from sac_expert_b200.population import PopulationSpec

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def lib():
    G.build()
    return L.load()


def header_symbols():
    txt = open(os.path.join(ROOT, "include", "saceo.h")).read()
    txt = re.sub(r"/\*.*?\*/", "", txt, flags=re.S)
    return sorted(set(re.findall(r"\b(saceo_[a-z_0-9]+)\s*\(", txt)))


def test_every_declared_symbol_is_exported(lib):
    syms = header_symbols()
    assert len(syms) >= 18
    for s in syms:
        assert hasattr(lib, s), s
    assert sorted(L.EXPORTS) == syms
    assert lib.saceo_abi_version() == L.ABI_VERSION


def test_layout_query_without_gpu(lib):
    spec = PopulationSpec(n_agents=256, S=27, A=8)
    lay = L.query_layout(spec.to_config())
    S, A, H, Hm = 27, 8, 256, 512
    assert lay.na == S * H + H + H * H + H + H * 2 * A + 2 * A
    assert lay.nc == (S + A) * H + H + H * H + H + H + 1
    assert lay.nm == (S + A) * Hm + Hm + Hm * Hm + Hm + Hm * (S + 1) + (S + 1)
    assert lay.na_stride % 32 == 0 and lay.na_stride > lay.na
    assert lay.row_words % 4 == 0 and lay.off_d % 2 == 0 and lay.off_d >= 2 * S + A + 1
    assert lay.workspace_bytes > 0
    hop = L.query_layout(PopulationSpec(n_agents=1, S=11, A=3).to_config())
    assert hop.row_words * 4 == 112          # Hopper row: 26 words + f64 done flag, 16-byte aligned


def test_config_validation_mirrors_reference_errors(lib):
    bad = PopulationSpec(n_agents=1, S=4, A=2, E=7, num_models=2).to_config()     # odd E with two models
    lay = L.Layout()
    assert lib.saceo_query_layout(C.byref(bad), C.byref(lay)) == -1
    assert b"even" in lib.saceo_last_error()
    with pytest.raises(ValueError):
        PopulationSpec(n_agents=1, S=4, A=2, actor_acts=("gelu", "relu")).to_config()
    three = PopulationSpec(n_agents=1, S=4, A=2, num_models=3).to_config()
    assert lib.saceo_query_layout(C.byref(three), C.byref(lay)) == -1
    for slot in (3, 4, 7):          # switches without a meaning: only 0 is accepted
        cfg = PopulationSpec(n_agents=1, S=4, A=2).to_config()
        cfg.reserved[slot] = 1
        assert lib.saceo_query_layout(C.byref(cfg), C.byref(lay)) == -1


def test_create_refuses_without_device(lib):
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    cfg = PopulationSpec(n_agents=1, S=4, A=2).to_config()
    ctx = C.c_void_p()
    rc = lib.saceo_create(C.byref(cfg), C.byref(ctx))
    assert rc == -3 and b"no CPU fallback" in lib.saceo_last_error()
    from sac_expert_b200.population import Population
    with pytest.raises(L.SaceoError):
        Population(PopulationSpec(n_agents=1, S=4, A=2))


def test_unbound_network_objects_fail_loudly():
    from sac_expert_b200.sac_eo.actors.init_actor import init_actor
    from sac_expert_b200.sac_eo.envs.synthetic import SyntheticEnv
    actor = init_actor(SyntheticEnv(4, 2), [8, 8], ["tanh"], 0.01, 1.0, "orthogonal", False, None, True, True, False)
    ws = actor.get_weights()
    assert [w.shape for w in ws] == [(4, 8), (8,), (8, 8), (8,), (8, 4), (4,)]
    actor.set_weights(actor.get_weights(flat=True), from_flat=True)
    with pytest.raises(L.SaceoError):
        actor.sample([0, 0, 0, 0])           # no device population bound: there is no CPU forward
