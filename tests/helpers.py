"""Shared helpers of the parity tests: golden loading and oracle construction."""
import glob
import json
import os

import numpy as np

from optical_rl_gym_b200.topology import TopologyTables

GOLDEN_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def golden_names():
    return sorted(os.path.basename(p)[:-4] for p in glob.glob(os.path.join(GOLDEN_DIR, "*.npz"))
                  if not p.endswith("nsfnet_tables.npz") and not os.path.basename(p).startswith(("wrap_", "topo_", "traffic_")))


def load_golden(name):
    with np.load(os.path.join(GOLDEN_DIR, name + ".npz"), allow_pickle=False) as z:
        g = {k: z[k] for k in z.files}
    g["meta"] = json.loads(str(g["meta"]))
    return g


def wrapper_golden_names():
    return sorted(os.path.basename(p)[:-4] for p in glob.glob(os.path.join(GOLDEN_DIR, "wrap_*.npz")))


def golden_tables():
    return TopologyTables.load(os.path.join(GOLDEN_DIR, "nsfnet_tables.npz"))


# Non-NSFNET topologies within the non-wide kernels' limits (<= 32 links, 5 paths per pair): the kernels read their link
# count at run time there (link template 0) instead of using the 22-link NSFNET instance.
SYNTHETIC = {"E20": (12, 8), "E32": (16, 16)}       # name -> (ring nodes, chords); 20 and 32 links
_TABLES = {}


def tables(name):
    """"nsfnet" (22 links), "E20" / "E32" (seeded ring + chords graphs, k = 5, seed 3), "small_xml" (10 nodes, 15 links,
    k = 3); built once per process."""
    if name not in _TABLES:
        from optical_rl_gym_b200.topology import synthetic_ring_chords

        if name == "nsfnet":
            _TABLES[name] = golden_tables()
        elif name == "small_xml":
            _TABLES[name] = TopologyTables.load(os.path.join(GOLDEN_DIR, "topo_small_xml_tables.npz"))
        else:
            nodes, chords = SYNTHETIC[name]
            _TABLES[name] = synthetic_ring_chords(nodes, chords, k_paths=5, seed=3)
    return _TABLES[name]


def sim_kwargs(meta):
    """Reference env_args (as recorded) -> the keyword set shared by the oracle and the product
    (defaults per env class: optical_network_env.py:14-25, rmsa_env.py:29-46, deeprmsa_env.py:10-21,
    rwa_env.py:19-31, rmcsa_env.py:29-49)."""
    kind, a = meta["kind"], dict(meta["env_args"])
    kw = {}
    kw["episode_length"] = a.get("episode_length", 1000)
    if kind == "DeepRMSA-v0":
        kw["mean_holding"] = a.get("mean_service_holding_time", 25.0)
        kw["mean_iat"] = a.get("mean_service_inter_arrival_time", 0.1)
        kw["num_slots"] = a.get("num_spectrum_resources", 100)
        kw["j"] = a.get("j", 1)
        kw["allow_rejection"] = a.get("allow_rejection", False)
    else:
        hold = a.get("mean_service_holding_time", 10800.0)
        load = a.get("load", 10.0)
        kw["mean_holding"] = hold
        kw["mean_iat"] = 1 / float(load / float(hold))
        kw["num_slots"] = a.get("num_spectrum_resources", 80 if kind == "RWA-v0" else 100)
        kw["allow_rejection"] = a.get("allow_rejection", kind == "RWA-v0")
    kw["channel_width"] = a.get("channel_width", 50.0 if kind == "RWA-v0" else 12.5)
    if kind == "RMCSA-v0":
        kw["num_cores"] = a.get("num_spatial_resources", 7)
        kw["worst_xt"] = a.get("worst_xt", {7: -84.7, 12: -61.9, 19: -54.8}.get(kw["num_cores"]))
    if a.get("bit_rate_selection") == "discrete":
        kw["bit_rates"] = list(a.get("bit_rates", (10, 40, 100)))
        kw["bit_rate_prob"] = a.get("bit_rate_probabilities")
    if a.get("node_request_probabilities") is not None:
        kw["node_prob"] = np.array(a["node_request_probabilities"], np.float64)
    return kw


HEURISTIC_ID = {"sp": 0, "sp_ff": 0, "sap": 1, "sap_ff": 1, "llp_ff": 2, "sap_lf": 3, "heuristic": 1}
