"""CPU-side checks: the C-ABI library loads and exports every symbol declared in include/orlg.h
(no compute call: there is no GPU here), host topology pre-processing, and the product never
touching the oracle."""
import ctypes
import os
import re

import numpy as np
import pytest

import helpers

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def header_symbols():
    text = open(os.path.join(ROOT, "include", "orlg.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(orlg_[a-z_]+)\s*\(", text)))


def test_library_exports_every_declared_symbol():
    from optical_rl_gym_b200 import _native

    lib = _native.lib()
    syms = header_symbols()
    assert len(syms) >= 20
    for s in syms:
        assert hasattr(lib, s), "liborlg.so does not export %s" % s
    assert sorted(_native.EXPORTED) == syms, "python binding list and header disagree"
    assert lib.orlg_version() == 1


def test_struct_layouts_match_header():
    """The ctypes mirrors must have the C layout of orlg_config / orlg_tables / orlg_request."""
    from optical_rl_gym_b200 import _native

    assert ctypes.sizeof(_native.Config) == 104          # 2*i32, i64, 12*i32, u64, 4*f64 (with padding)
    assert _native.Config.seed.offset % 8 == 0 and _native.Config.env_id_base.offset == 8
    assert ctypes.sizeof(_native.Tables) == 6 * 4 + 15 * 8
    assert ctypes.sizeof(_native.KernelInfo) == 7 * 4
    assert _native.REQUEST_DTYPE.itemsize == 32
    assert [_native.REQUEST_DTYPE.fields[n][1] for n in ("arrival", "holding", "src", "dst", "bit_rate")] == [0, 8, 16, 20, 24]


def test_create_fails_cleanly_without_gpu_or_with_bad_arguments():
    from optical_rl_gym_b200 import _native

    lib = _native.lib()
    out = ctypes.c_void_p()
    assert lib.orlg_create(None, None, 0, ctypes.byref(out)) == -1
    assert b"null" in lib.orlg_last_error()
    cfg = _native.Config(kind=7, num_envs=4)
    tab = _native.Tables()
    assert lib.orlg_create(ctypes.byref(cfg), ctypes.byref(tab), 0, ctypes.byref(out)) == -1


def test_product_fails_loudly_without_cuda():
    torch = pytest.importorskip("torch")
    if torch.cuda.is_available():
        pytest.skip("this check is for the GPU-less container")
    from optical_rl_gym_b200 import OpticalVecEnv, _native

    with pytest.raises(_native.NativeError):
        OpticalVecEnv("DeepRMSA-v0", 4, helpers.golden_tables())


def test_product_never_imports_the_oracle():
    pkg = os.path.join(ROOT, "optical-rl-gym_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                text = open(os.path.join(dirpath, f)).read()
                assert "oracle" not in text.lower() or f == "orlg_device.cuh" and "oracle reproduces" in text, \
                    "%s mentions the oracle" % os.path.join(dirpath, f)


def test_nsfnet_tables_equal_reference_pickle_tables():
    """optical_rl_gym_b200.topology.nsfnet() (own link list + NetworkX KSP) == tables extracted from the
    reference's nsfnet_chen_5-paths_6-modulations.h5 (tests/golden/nsfnet_tables.npz)."""
    import dataclasses

    from optical_rl_gym_b200.topology import nsfnet

    a, b = nsfnet(), helpers.golden_tables()
    assert (a.num_nodes, a.num_links, a.num_paths, a.k_paths) == (14, 22, 455, 5)
    for f in dataclasses.fields(a):
        if f.name == "name":
            continue
        x, y = getattr(a, f.name), getattr(b, f.name)
        assert np.array_equal(x, y) if isinstance(x, np.ndarray) else x == y, f.name
    # SURVEY.md section 8 facts
    assert a.path_hops.min() == 1 and a.path_hops.max() == 9
    assert int((a.path_se == 1).sum()) == 372


def test_topology_roundtrip_and_synthetic(tmp_path):
    from optical_rl_gym_b200.topology import TopologyTables, synthetic_ring_chords

    t = synthetic_ring_chords(num_nodes=12, num_chords=10, k_paths=3, seed=3)
    assert t.num_links == 22 and t.num_nodes == 12 and t.k_paths == 3
    assert (t.pair_count[t.pair_first >= 0] >= 1).all()
    p = tmp_path / "t.npz"
    t.save(p)
    u = TopologyTables.load(p)
    assert np.array_equal(t.path_links, u.path_links) and u.node_names == t.node_names
    for row in range(t.num_paths):                      # CSR consistency: hops == number of links, links chain the nodes
        links = t.links_of(row)
        assert len(links) == t.path_hops[row]


def test_number_of_slots_integer_form_matches_reference_float_expression():
    """SURVEY a6: ceil(b / (SE*12.5)) + 1 == (2b + 25SE - 1)//(25SE) + 1 for every table entry the library builds."""
    import math

    for se in range(1, 7):
        for b in range(1, 1024):
            assert math.ceil(b / (se * 12.5)) + 1 == (2 * b + 25 * se - 1) // (25 * se) + 1


def test_integration_md_stub_matches_the_header_structs():
    """The ctypes stub printed in INTEGRATION.md section 2 is what a maintainer would copy: its Config / Tables
    must have exactly the layout of include/orlg.h (a short Tables hands orlg_create a garbage link_order pointer)."""
    import ctypes as C
    import re

    from optical_rl_gym_b200 import _native

    text = open(os.path.join(ROOT, "INTEGRATION.md")).read()
    block = re.search(r"```python\nimport ctypes as C, numpy as np, torch\n(.*?)```", text, re.S).group(1)
    classes = block[block.index("class Config"):block.index("class BatchedDeepRMSA")]
    ns = {"C": C}
    exec(classes, ns)
    for name in ("Config", "Tables"):
        doc, real = ns[name], getattr(_native, name)
        assert [f[0] for f in doc._fields_] == [f[0] for f in real._fields_], name
        assert C.sizeof(doc) == C.sizeof(real), name
        for f in real._fields_:
            assert getattr(doc, f[0]).offset == getattr(real, f[0]).offset, (name, f[0])


def test_spaces_sample_seed_contains():
    """gym 0.21 space protocol of the stand-ins (what SB3's VecEnv consumers call): seed() makes sample() reproducible, samples
    are members, shapes / dtypes as the reference declares them (deeprmsa_env.py:38-43, rmsa_env.py:138-149, rmcsa_env.py:181-188)."""
    from optical_rl_gym_b200 import spaces

    d = spaces.Discrete(6)
    d.seed(3)
    a = [d.sample() for _ in range(200)]
    d.seed(3)
    assert a == [d.sample() for _ in range(200)] and set(a) == set(range(6)) and all(x in d for x in a)
    assert 6 not in d and -1 not in d and 2.5 not in d
    m = spaces.MultiDiscrete((6, 101))
    m.seed(1)
    xs = np.stack([m.sample() for _ in range(500)])
    assert xs.dtype == np.int64 and xs.shape == (500, 2) and (xs >= 0).all() and (xs < [6, 101]).all() and xs[:, 1].max() > 90
    assert m.contains(xs[0]) and not m.contains(np.array([6, 0])) and not m.contains(np.array([1, 2, 3]))
    b = spaces.Box(0, 1, (54,), np.float32)
    b.seed(0)
    y = b.sample()
    assert y.shape == (54,) and y.dtype == np.float32 and b.contains(y) and not b.contains(y + 2)
    dd = spaces.Dict({"a": spaces.Discrete(3), "b": spaces.Box(0, 1, (2,), np.uint8)})
    dd.seed(5)
    s = dd.sample()
    assert dd.contains(s) and s["b"].dtype == np.uint8


def test_policy_loader_shared_and_separate_trunks():
    """MlpPolicy.from_state_dict: the SB3 < 1.8 layout (shared trunk: the shipped best_model.zip) and the >= 1.8 layout with
    separate actor / critic trunks -- the value must come from the critic's own trunk (ADVICE round 1)."""
    import torch

    from optical_rl_gym_b200.policy import MlpPolicy

    torch.manual_seed(0)
    obs_dim, width, n_act = 54, 16, 5

    def lin(i, o):
        return torch.nn.Linear(i, o)

    pi = [lin(obs_dim, width), lin(width, width)]
    vf = [lin(obs_dim, width), lin(width, width)]
    act, val = lin(width, n_act), lin(width, 1)
    x = torch.randn(7, obs_dim)

    def trunk(ls, v):
        for layer in ls:
            v = torch.tanh(layer(v))
        return v

    sd = {"action_net.weight": act.weight, "action_net.bias": act.bias, "value_net.weight": val.weight, "value_net.bias": val.bias}
    for j, layer in enumerate(pi):
        sd["mlp_extractor.policy_net.%d.weight" % (2 * j)] = layer.weight
        sd["mlp_extractor.policy_net.%d.bias" % (2 * j)] = layer.bias
    for j, layer in enumerate(vf):
        sd["mlp_extractor.value_net.%d.weight" % (2 * j)] = layer.weight
        sd["mlp_extractor.value_net.%d.bias" % (2 * j)] = layer.bias
    pol = MlpPolicy.from_state_dict({k: v.detach() for k, v in sd.items()})
    logits, value = pol(x)
    assert torch.allclose(logits, act(trunk(pi, x)), atol=1e-6) and torch.allclose(value, val(trunk(vf, x)).squeeze(-1), atol=1e-6)
    assert not torch.allclose(value, val(trunk(pi, x)).squeeze(-1), atol=1e-3)
    shared = {"action_net.weight": act.weight, "action_net.bias": act.bias, "value_net.weight": val.weight, "value_net.bias": val.bias}
    for j, layer in enumerate(pi):
        shared["mlp_extractor.shared_net.%d.weight" % (2 * j)] = layer.weight
        shared["mlp_extractor.shared_net.%d.bias" % (2 * j)] = layer.bias
    pol2 = MlpPolicy.from_state_dict({k: v.detach() for k, v in shared.items()})
    l2, v2 = pol2(x)
    assert pol2.critic_net is None and torch.allclose(l2, logits, atol=1e-6) and torch.allclose(v2, val(trunk(pi, x)).squeeze(-1), atol=1e-6)
