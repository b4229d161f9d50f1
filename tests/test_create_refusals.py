"""orlg_create refuses every unsupported configuration with its documented code and message, before it allocates anything.

Each case changes one field of an otherwise valid NSFNET configuration.  The checks before the device query run on any
machine; the ones after it need a device.  The checks run in a fixed order, so an input with several faults is refused for
the first of them.  On the GPU, handles whose creation fails after the first device allocation free what they allocated."""
import ctypes
import json
import os
import subprocess
import sys

import numpy as np
import pytest

import helpers

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
KIND = {"RWA": 0, "RMSA": 1, "DeepRMSA": 2, "RMCSA": 3}
OK, E_INVALID, E_UNSUPPORTED, E_CUDA, E_NOMEM = 0, -1, -2, -3, -4


@pytest.fixture(scope="module")
def lib():
    from optical_rl_gym_b200 import _native

    return _native.lib()


@pytest.fixture(scope="module")
def nsfnet():
    return helpers.golden_tables()


def create(lib, t, device=0, tables=None, **cfg):
    """orlg_create on NSFNET tables t: `cfg` overrides fields of a valid DeepRMSA-v0 configuration, `tables` fields of the
    orlg_tables struct or of the arrays behind it.  Returns (code, message); a created handle is destroyed."""
    from optical_rl_gym_b200 import _native as nat

    tables = dict(tables or {})
    c = dict(kind=KIND["DeepRMSA"], num_envs=64, num_slots=100, num_cores=1, j=1, episode_length=50, allow_rejection=0,
              bit_rate_lo=25, bit_rate_hi=100, traffic=nat.TRAFFIC_PHILOX, obs_dtype=nat.OBS_F32, auto_reset=1,
              heap_capacity=0, seed=7, channel_width=12.5, mean_holding=25.0, mean_iat=0.1, worst_xt=-84.7)
    c.update(cfg)
    bit_rates = np.asarray(tables.pop("bit_rates", [0]), np.int32)
    keep = {}

    def arr(name, dtype):
        keep[name] = np.ascontiguousarray(tables.pop(name, getattr(t, name)), dtype=dtype)
        return keep[name].ctypes.data_as(ctypes.c_void_p)

    counts = dict(num_nodes=t.num_nodes, num_links=t.num_links, k_paths=t.k_paths, num_paths=t.num_paths,
                  num_mods=len(t.mod_se), num_bit_rates=0)
    counts.update({k: tables.pop(k) for k in list(tables) if k in counts})
    keep["node_prob"] = np.full(t.num_nodes, 1.0 / t.num_nodes)
    keep["bit_rates"] = bit_rates
    keep["bit_rate_prob"] = np.full(len(bit_rates), 1.0 / len(bit_rates))
    tab = nat.Tables(**counts,
                     pair_first=arr("pair_first", np.int32), pair_count=arr("pair_count", np.int32),
                     path_hops=arr("path_hops", np.int32), path_se=arr("path_se", np.int32),
                     path_mod=arr("path_mod", np.int32), path_link_ptr=arr("path_link_ptr", np.int32),
                     path_links=arr("path_links", np.int32), path_length=arr("path_length", np.float64),
                     mod_se=arr("mod_se", np.int32), mod_osnr=arr("mod_osnr", np.float64), mod_xt=arr("mod_xt", np.float64),
                     node_prob=keep["node_prob"].ctypes.data_as(ctypes.c_void_p),
                     bit_rates=keep["bit_rates"].ctypes.data_as(ctypes.c_void_p),
                     bit_rate_prob=keep["bit_rate_prob"].ctypes.data_as(ctypes.c_void_p),
                     link_order=arr("link_order", np.int32))
    assert not tables, "unknown table fields %s" % sorted(tables)
    h = ctypes.c_void_p()
    rc = lib.orlg_create(ctypes.byref(nat.Config(**c)), ctypes.byref(tab), device, ctypes.byref(h))
    if rc != OK:
        assert not h.value
        return rc, lib.orlg_last_error().decode()
    assert h.value and lib.orlg_destroy(h) == OK
    return rc, ""


# (case, overrides of the configuration, overrides of the tables, code, message): the checks before the device query
BEFORE_DEVICE = [
    ("unknown_kind", dict(kind=4), {}, E_INVALID, "unknown env kind"),
    ("num_envs_zero", dict(num_envs=0), {}, E_INVALID, "num_envs must be positive"),
    ("num_envs_negative", dict(num_envs=-5), {}, E_INVALID, "num_envs must be positive"),
    ("slots_zero", dict(num_slots=0), {}, E_UNSUPPORTED, "1..512 slots per link"),
    ("slots_513", dict(num_slots=513), {}, E_UNSUPPORTED, "1..512 slots per link"),
    ("links_zero", {}, dict(num_links=0), E_UNSUPPORTED, "1..65535 links"),
    ("links_65536", {}, dict(num_links=65536), E_UNSUPPORTED, "1..65535 links"),
    ("nodes_one", {}, dict(num_nodes=1), E_UNSUPPORTED, "2..255 nodes"),
    ("nodes_256", {}, dict(num_nodes=256), E_UNSUPPORTED, "2..255 nodes"),
    ("k_zero", {}, dict(k_paths=0), E_UNSUPPORTED, "k_paths must be 1..16"),
    ("k_17", {}, dict(k_paths=17), E_UNSUPPORTED, "k_paths must be 1..16"),
    ("paths_2^20", {}, dict(num_paths=1 << 20), E_UNSUPPORTED, "too many paths"),
    ("cores_zero", dict(kind=KIND["RMCSA"], num_cores=0), {}, E_UNSUPPORTED, "1..31 cores"),
    ("cores_32", dict(kind=KIND["RMCSA"], num_cores=32), {}, E_UNSUPPORTED, "1..31 cores"),
    ("j_zero", dict(j=0), {}, E_INVALID, "j must be 1..16"),
    ("j_17", dict(j=17), {}, E_INVALID, "j must be 1..16"),
    ("episode_zero", dict(episode_length=0), {}, E_UNSUPPORTED, "episode_length must be < 2^22"),
    ("episode_2^22", dict(episode_length=1 << 22), {}, E_UNSUPPORTED, "episode_length must be < 2^22"),
    ("holding_zero", dict(mean_holding=0.0), {}, E_INVALID, "holding / inter-arrival times must be positive"),
    ("iat_nan", dict(mean_iat=float("nan")), {}, E_INVALID, "holding / inter-arrival times must be positive"),
    ("bit_rate_bounds", dict(kind=KIND["RMSA"], bit_rate_lo=100, bit_rate_hi=25), {}, E_INVALID,
     "bit_rate_higher_bound < bit_rate_lower_bound"),
    ("no_modulation_table", dict(kind=KIND["RMCSA"], num_cores=7), dict(num_mods=0), E_INVALID,
     "RMCSA needs a modulation table"),
    # several faults: the first check in order decides
    ("envs_before_slots", dict(num_envs=0, num_slots=0), {}, E_INVALID, "num_envs must be positive"),
    ("links_before_nodes", {}, dict(num_links=0, num_nodes=1), E_UNSUPPORTED, "1..65535 links"),
    ("j_before_times", dict(j=0, mean_holding=-1.0), {}, E_INVALID, "j must be 1..16"),
    ("configuration_before_device", dict(episode_length=0), {}, E_UNSUPPORTED, "episode_length must be < 2^22"),
]


@pytest.mark.parametrize("case,cfg,tables,code,message", BEFORE_DEVICE, ids=[c[0] for c in BEFORE_DEVICE])
def test_refusal_before_the_device_query(lib, nsfnet, case, cfg, tables, code, message):
    device = 10 ** 6 if case == "configuration_before_device" else 0
    assert create(lib, nsfnet, device=device, tables=tables, **cfg) == (code, message)


@pytest.mark.parametrize("kind", ["DeepRMSA", "RMSA", "RMCSA"])
def test_valid_configuration_reaches_the_device_query(lib, nsfnet, kind):
    """The base configurations pass every check before the device query: a device that does not exist refuses them."""
    assert create(lib, nsfnet, device=-1, kind=KIND[kind], num_cores=7) == (E_CUDA, "no such CUDA device")


def _path_link_out_of_range(t):
    links = t.path_links.copy()
    links[3] = t.num_links
    return dict(path_links=links)


def _path_link_negative(t):
    links = t.path_links.copy()
    links[0] = -1
    return dict(path_links=links)


def _hop_count(t):
    hops = t.path_hops.copy()
    hops[7] += 1
    return dict(path_hops=hops)


# the checks after the device query, in their order
AFTER_DEVICE = [
    ("bit_rate_above_65535", dict(kind=KIND["RMSA"]), lambda t: dict(num_bit_rates=2, bit_rates=[40, 70000]), E_UNSUPPORTED,
     "bit rates must be 0..65535"),
    ("observation_tile", dict(j=16, obs_dtype=1), lambda t: {}, E_UNSUPPORTED, "observation too large for the staging tile"),
    ("heap_capacity_4097", dict(heap_capacity=4097), lambda t: {}, E_UNSUPPORTED,
     "heap_capacity above 4096 live services per environment"),
    ("path_link_out_of_range", {}, _path_link_out_of_range, E_INVALID, "path link index out of range"),
    ("path_link_negative", {}, _path_link_negative, E_INVALID, "path link index out of range"),
    ("hop_count", {}, _hop_count, E_INVALID, "inconsistent path hop counts"),
    ("slots_201_continuous", dict(kind=KIND["RMSA"], num_slots=320, channel_width=0.5), lambda t: {}, E_UNSUPPORTED,
     "a request of this configuration may need 201..320 slots: at most 200 slots per service are representable"),
    ("slots_201_discrete", dict(kind=KIND["RMSA"], num_slots=300, channel_width=0.5),
     lambda t: dict(num_bit_rates=2, bit_rates=[10, 100]), E_UNSUPPORTED,
     "a request of this configuration may need 201..300 slots: at most 200 slots per service are representable"),
    # several faults: the first check in order decides
    ("tile_before_heap", dict(j=16, obs_dtype=1, heap_capacity=5000), lambda t: {}, E_UNSUPPORTED,
     "observation too large for the staging tile"),
    ("heap_before_paths", dict(heap_capacity=5000), _hop_count, E_UNSUPPORTED,
     "heap_capacity above 4096 live services per environment"),
    ("links_before_hops", {}, lambda t: dict(_path_link_out_of_range(t), **_hop_count(t)), E_INVALID,
     "path link index out of range"),
    ("paths_before_slots", dict(kind=KIND["RMSA"], num_slots=320, channel_width=0.5), _hop_count, E_INVALID,
     "inconsistent path hop counts"),
]


@pytest.mark.gpu
@pytest.mark.parametrize("case,cfg,tables,code,message", AFTER_DEVICE, ids=[c[0] for c in AFTER_DEVICE])
def test_refusal_after_the_device_query(lib, nsfnet, case, cfg, tables, code, message):
    assert create(lib, nsfnet, tables=tables(nsfnet), **cfg) == (code, message)


@pytest.mark.gpu
@pytest.mark.parametrize("kind,cfg,tables", [
    ("DeepRMSA", {}, {}),
    ("DeepRMSA", dict(j=15, obs_dtype=1, heap_capacity=4096), {}),      # the largest tile and capacity that are accepted
    ("RMSA", dict(num_slots=320, channel_width=0.6), {}),               # 100 Gb/s needs 168 slots: representable
    ("RMSA", {}, dict(num_bit_rates=3, bit_rates=[10, 40, 65535])),
    ("RMCSA", dict(num_cores=7), {}),
])
def test_base_configurations_are_accepted(lib, nsfnet, kind, cfg, tables):
    """The configurations the refusals above start from create a handle."""
    assert create(lib, nsfnet, tables=tables, kind=KIND[kind], **cfg) == (OK, "")


def leak_check_child():
    """Runs in a child process (see the test below) and prints the free device memory before and after."""
    import torch

    from optical_rl_gym_b200 import _native

    lib, t = _native.lib(), helpers.golden_tables()
    torch.cuda.init()
    huge = dict(num_envs=2 ** 31 - 1)
    small = dict(num_envs=4096, episode_length=100)
    first = [create(lib, t, **huge), create(lib, t, **small)]       # module loading and context set-up are not leaks
    torch.cuda.synchronize()
    free0 = torch.cuda.mem_get_info()[0]
    refused = [create(lib, t, **huge) for _ in range(50)]
    created = [create(lib, t, **small)[0] for _ in range(50)]
    torch.cuda.synchronize()
    free1 = torch.cuda.mem_get_info()[0]
    print(json.dumps(dict(first=first, refused=sorted(set(map(tuple, refused))), created=sorted(set(created)),
                          free0=free0, free1=free1)))


@pytest.mark.gpu
def test_failed_creates_free_what_they_allocated():
    """2^31 - 1 envs pass every configuration check; the tables upload, and the first state array (22 links x 16 bytes per
    env: ~756 GB of masks) is refused at once.  50 such creates and 50 create / destroy pairs of a 4096-env handle leave
    free device memory where it was.  In a child process: a refused cudaMalloc stays in the CUDA runtime's last error of the
    thread, where the next kernel-launch check of an unrelated test would find it."""
    env = dict(os.environ, PYTHONPATH=os.pathsep.join([os.path.join(ROOT, "optical-rl-gym_b200"), os.path.dirname(__file__),
                                                       os.environ.get("PYTHONPATH", "")]))
    flags = ["-s"] if sys.flags.no_user_site else []
    res = subprocess.run([sys.executable] + flags + ["-c", "import test_create_refusals as m; m.leak_check_child()"],
                         env=env, capture_output=True, text=True, timeout=600)
    assert res.returncode == 0, res.stderr[-4000:]
    out = json.loads(res.stdout.strip().splitlines()[-1])
    nomem = [E_NOMEM, "cudaMalloc failed for %d bytes" % (22 * 16 * (2 ** 31 - 1))]
    assert out["first"] == [nomem, [OK, ""]]
    assert out["refused"] == [nomem]
    assert out["created"] == [OK]
    assert out["free1"] == out["free0"], "device memory not returned: %d bytes" % (out["free0"] - out["free1"])
