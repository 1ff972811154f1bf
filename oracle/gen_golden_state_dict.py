"""tests/golden/reference_state_dict.json: key, shape and dtype of every state_dict entry of UNet2D5_dsbn
(PyMIC/pymic/net/net3d/unet2d5_dsbn.py), in order, for the authors' VS network (vs_t1s_{g,weights,S}.cfg: feature_chns
32-512, conv_dims [2, 2, 3, 3, 3]) and for the benchmark's network (ft 16-256, all 3-D)
(tests/test_integration_reference.py::test_state_dict_layout_matches_the_reference_network).

With a PyMIC source tree given, the layout is read from the reference's own class; without one, from the drop-in
fplplus_b200.net.UNet2D5_dsbn:
    python -m oracle.gen_golden_state_dict [--reference <dir holding PyMIC/>]"""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

BASE = {"net_type": "UNet2D5_dsbn", "num_domains": 2, "class_num": 2, "in_chns": 1, "dropout": [0.0, 0.0, 0.3, 0.4, 0.5],
        "bilinear": False, "deep_supervise": False, "aes": False}
NETWORKS = {"vs_shipped": dict(BASE, feature_chns=[32, 64, 128, 256, 512], conv_dims=[2, 2, 3, 3, 3]),
            "configs2": dict(BASE, feature_chns=[16, 32, 64, 128, 256], conv_dims=[3, 3, 3, 3, 3])}


def layout(state_dict):
    return [[k, list(v.shape), str(v.dtype).replace("torch.", "")] for k, v in state_dict.items()]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reference", help="directory holding the PyMIC source tree of the original project")
    args = ap.parse_args()
    if args.reference:
        sys.path.insert(0, os.path.join(args.reference, "PyMIC"))
        from pymic.net.net3d.unet2d5_dsbn import UNet2D5_dsbn
        source = "PyMIC/pymic/net/net3d/unet2d5_dsbn.py UNet2D5_dsbn"
    else:
        from fplplus_b200.net import UNet2D5_dsbn
        source = ("fplplus_b200.net.UNet2D5_dsbn, whose layout is identical to commit 731a43c's, where "
                  "tests/test_integration_reference.py matched it key for key (order, shape, dtype) to the reference class")
    out = {"source": source, "networks": {}}
    for tag, params in NETWORKS.items():
        out["networks"][tag] = {"params": params, "state_dict": layout(UNet2D5_dsbn(dict(params)).state_dict())}
    path = os.path.join(ROOT, "tests", "golden", "reference_state_dict.json")
    with open(path, "w") as f:
        json.dump(out, f, separators=(",", ":"))
    print("wrote", path)


if __name__ == "__main__":
    main()
