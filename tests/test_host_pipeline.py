"""Rows f3 / f4 of SURVEY.md section 8: host topology pipeline (file readers, k-shortest paths, pickle loader, cache),
the SB3-format episode monitor and the MLP policy loader.  CPU tests unless marked gpu."""
import dataclasses
import io
import os
import zipfile

import numpy as np
import pytest

import helpers
from optical_rl_gym_b200 import topology as T

GOLD = helpers.GOLDEN_DIR


def assert_same_tables(a, b, skip=("name",)):
    for f in dataclasses.fields(T.TopologyTables):
        if f.name in skip:
            continue
        x, y = getattr(a, f.name), getattr(b, f.name)
        if isinstance(x, np.ndarray):
            assert np.array_equal(x, y, equal_nan=x.dtype.kind == "f"), f.name
        else:
            assert x == y, f.name


@pytest.mark.parametrize("src,gold,k", [("topo_small.txt", "topo_small_txt_tables.npz", 4),
                                        ("topo_small.xml", "topo_small_xml_tables.npz", 3)])
def test_file_readers_reproduce_reference_get_topology(src, gold, k, tmp_path):
    """Our reader + Yen pipeline on a .txt / SNDlib .xml file == the reference's create_topology.get_topology on the
    same file (golden recorded by tests/golden/make_golden_topology.py): every path, hop list, length, modulation."""
    want = T.TopologyTables.load(os.path.join(GOLD, gold))
    got = T.get_topology(os.path.join(GOLD, src), k_paths=k, cache_dir=str(tmp_path))
    assert_same_tables(got, want)
    assert len(os.listdir(tmp_path)) == 1                      # cached ...
    again = T.get_topology(os.path.join(GOLD, src), k_paths=k, cache_dir=str(tmp_path))
    assert_same_tables(again, got, skip=())                    # ... and the cache round-trips (name included)


def test_sndlib_lengths_are_rounded_haversine():
    names, links = T.read_sndlib_topology(os.path.join(GOLD, "topo_small.xml"))
    assert names[0] == "Aveiro" and len(names) == 10 and len(links) == 15
    want = T.TopologyTables.load(os.path.join(GOLD, "topo_small_xml_tables.npz"))
    assert np.array_equal(np.array([l for _, _, l in links]), want.link_length)
    assert all(round(l, 3) == l for _, _, l in links)


def test_txt_reader_edge_cases(tmp_path):
    p = tmp_path / "t.txt"
    p.write_text("# comment\n# another\n3\n3\n1 2 10\n2 3 20\n\n1 3 40\n")
    names, links = T.read_txt_file(p)
    assert names == ("1", "2", "3") and links == [("1", "2", 10), ("2", "3", 20), ("1", "3", 40)]
    t = T.get_topology(p, k_paths=2)
    assert t.num_paths == 6 and list(t.path_length[t.rows_of(0, 2)]) == [30.0, 40.0]
    with pytest.raises(ValueError):
        T.get_topology(str(tmp_path / "t.csv"))
    bad = tmp_path / "bad.txt"
    bad.write_text("2\n1\n1 5 10\n")
    with pytest.raises(ValueError):
        T.get_topology(bad)


def test_germany50_golden_is_consistent():
    t = T.TopologyTables.load(os.path.join(GOLD, "topo_germany50_tables.npz"))
    assert (t.num_nodes, t.num_links, t.k_paths, t.num_paths) == (50, 88, 5, 6125)
    for row in (0, 17, 6124):
        links = t.links_of(row)
        assert len(links) == t.path_hops[row]
        assert abs(t.link_length[links].sum() - t.path_length[row]) < 1e-9
        assert t.path_length[row] <= t.mod_reach[t.path_mod[row]]


# ---------------------------------------------------------------------------------------------- MLP policy
def _fake_sb3_zip(path, rng, shared=True):
    import torch

    dims = [54, 128, 128, 128, 128, 128]
    sd = {}
    trunk = "mlp_extractor.shared_net." if shared else "mlp_extractor.policy_net."
    for i in range(5):
        sd["%s%d.weight" % (trunk, 2 * i)] = torch.tensor(rng.normal(0, 0.2, (dims[i + 1], dims[i])), dtype=torch.float32)
        sd["%s%d.bias" % (trunk, 2 * i)] = torch.tensor(rng.normal(0, 0.1, dims[i + 1]), dtype=torch.float32)
    sd["action_net.weight"] = torch.tensor(rng.normal(0, 0.2, (5, 128)), dtype=torch.float32)
    sd["action_net.bias"] = torch.tensor(rng.normal(0, 0.1, 5), dtype=torch.float32)
    sd["value_net.weight"] = torch.tensor(rng.normal(0, 0.2, (1, 128)), dtype=torch.float32)
    sd["value_net.bias"] = torch.tensor(rng.normal(0, 0.1, 1), dtype=torch.float32)
    buf = io.BytesIO()
    torch.save(sd, buf)
    with zipfile.ZipFile(path, "w") as z:
        z.writestr("policy.pth", buf.getvalue())
        z.writestr("data", "{}")
    return {k: v.numpy().astype(np.float64) for k, v in sd.items()}, trunk


@pytest.mark.parametrize("shared", [True, False])
def test_mlp_policy_loads_sb3_archive_and_matches_numpy_forward(tmp_path, shared):
    torch = pytest.importorskip("torch")
    from optical_rl_gym_b200.policy import MlpPolicy

    rng = np.random.default_rng(3)
    sd, trunk = _fake_sb3_zip(tmp_path / "model.zip", rng, shared)
    pol = MlpPolicy.from_sb3_zip(tmp_path / "model.zip")
    obs = helpers.load_golden("deeprmsa_default_random")["obs"][0, :256]
    x = obs.copy()
    for i in range(5):
        x = np.tanh(x @ sd["%s%d.weight" % (trunk, 2 * i)].T + sd["%s%d.bias" % (trunk, 2 * i)])
    logits = x @ sd["action_net.weight"].T + sd["action_net.bias"]
    value = (x @ sd["value_net.weight"].T + sd["value_net.bias"])[:, 0]
    got_l, got_v = pol(torch.as_tensor(obs))
    np.testing.assert_allclose(got_l.detach().numpy(), logits, rtol=2e-4, atol=2e-5)
    np.testing.assert_allclose(got_v.detach().numpy(), value, rtol=2e-4, atol=2e-5)
    a = pol.act(torch.as_tensor(obs)).numpy()
    assert a.shape == (256, 1) and a.dtype == np.int32
    margin = np.sort(logits, axis=1)
    clear = (margin[:, -1] - margin[:, -2]) > 1e-3
    assert np.array_equal(a[clear, 0], logits.argmax(1)[clear])
    s = pol.act(torch.as_tensor(obs), deterministic=False, generator=torch.Generator().manual_seed(1))
    assert s.min() >= 0 and s.max() < 5


def test_monitor_file_format_matches_sb3(tmp_path):
    """load_monitor_csv reads the layout SB3 writes (header line + r,l,t,<keywords>)."""
    from optical_rl_gym_b200.monitor import load_monitor_csv

    p = tmp_path / "x.monitor.csv"
    p.write_text('#{"t_start": 1650000000.0, "env_id": "DeepRMSA-v0"}\nr,l,t,episode_service_blocking_rate\n'
                 "-12.0,50,1.5,0.62\n-8.0,50,3.25,0.58\n")
    header, cols = load_monitor_csv(p)
    assert header["env_id"] == "DeepRMSA-v0" and list(cols) == ["r", "l", "t", "episode_service_blocking_rate"]
    assert cols["r"].tolist() == [-12.0, -8.0] and cols["l"].tolist() == [50.0, 50.0]


@pytest.mark.gpu
def test_vec_monitor_and_policy_rollout_on_device(tmp_path):
    """VecMonitor over the CUDA env: per-episode return / length / info keywords equal a host recomputation from the
    step outputs; the monitor file parses; an MLP policy drives the env without leaving the device."""
    import torch

    from optical_rl_gym_b200 import OpticalVecEnv
    from optical_rl_gym_b200.monitor import VecMonitor, load_monitor_csv
    from optical_rl_gym_b200.policy import MlpPolicy

    n, L = 64, 30
    base = OpticalVecEnv("DeepRMSA-v0", n, helpers.golden_tables(), seed=4, episode_length=L)
    keys = ("episode_service_blocking_rate", "episode_bit_rate_blocking_rate")
    env = VecMonitor(base, str(tmp_path / "train"), info_keywords=keys)
    torch.manual_seed(0)
    pol = MlpPolicy(base.obs_dim, base.action_space.n).to("cuda")
    obs = env.reset()
    ret = np.zeros(n)
    want_r, want_l, want_b = [], [], []
    for t in range(3 * L):
        a = pol.act(obs, deterministic=False)
        obs, reward, done, info = env.step(a)
        ret += reward.cpu().numpy()
        d = done.cpu().numpy().astype(bool)
        if d.any():
            want_r += ret[d].tolist()
            want_l += [L - 1] * int(d.sum())              # SURVEY App. B-1: episodes are episode_length - 1 steps
            want_b += info[keys[0]].cpu().numpy()[d].tolist()
            ret[d] = 0
    assert len(want_r) == 3 * n and env.get_episode_rewards() == want_r and env.get_episode_lengths() == want_l
    assert env.episode_infos[keys[0]] == want_b
    env.close()
    header, cols = load_monitor_csv(str(tmp_path / "train.monitor.csv"))
    assert header["env_id"] == "DeepRMSA-v0" and list(cols) == ["r", "l", "t"] + list(keys)
    assert cols["r"].tolist() == want_r and cols["l"].tolist() == [float(x) for x in want_l]
    assert np.array_equal(cols[keys[0]], np.array(want_b))
