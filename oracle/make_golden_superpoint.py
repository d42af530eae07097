"""Generate tests/golden/sp_*.pt by running the UNMODIFIED reference SuperPoint in this container.

    python oracle/make_golden_superpoint.py [case ...]   # needs /root/reference (read-only); CPU, fp32

``lightglue/superpoint.py`` imports ``kornia.color.rgb_to_grayscale`` (absent here) and ``.utils.Extractor`` (which
imports kornia and cv2), and its constructor downloads ``superpoint_v1.pth``.  Neither is on the path this oracle
covers (grayscale input, ``forward``), so the generator provides stand-ins for exactly those three things -- a
``kornia.color`` stub that must never be called, a minimal ``Extractor`` base that only builds ``self.conf`` the
way utils.py:131-134 does, and a ``torch.hub.load_state_dict_from_url`` that returns the seeded synthetic weights
(oracle/superpoint_synth.py) -- and loads the reference file by path.  Everything else that runs is the
reference's own code.  Fixtures store the recipe, checksums of the regenerated image / weights and the outputs;
``float64/<name>.pt`` holds the keypoints and scores of the same forward in float64.
"""
from __future__ import annotations

import importlib.util
import os
import sys
import types
from types import SimpleNamespace

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from lightglue_b200 import synth  # noqa: E402
from oracle import superpoint_synth as sps  # noqa: E402

REF = "/root/reference/lightglue/superpoint.py"
OUT = os.path.join(ROOT, "tests", "golden")

CASES = {
    "sp_240x320": dict(h=240, w=320, b=1, seed=11, conf={}),
    "sp_480x640_top512": dict(h=480, w=640, b=1, seed=12, conf=dict(max_num_keypoints=512)),
    "sp_b2_top256": dict(h=240, w=320, b=2, seed=13, conf=dict(max_num_keypoints=256)),
    "sp_nms2_thr01": dict(h=160, w=240, b=1, seed=14, conf=dict(nms_radius=2, detection_threshold=0.1, remove_borders=8)),
    # neither extent a multiple of 8, odd at several pooling levels (203 -> 101 -> 50 -> 25, 317 -> 158 -> 79 -> 39)
    "sp_odd_203x317": dict(h=203, w=317, b=1, seed=17, conf={}),
}


def load_reference(weights):
    def never(*a, **k):
        raise RuntimeError("rgb_to_grayscale is outside the pinned path (grayscale inputs only)")

    kornia = types.ModuleType("kornia")
    color = types.ModuleType("kornia.color")
    color.rgb_to_grayscale = never
    kornia.color = color
    sys.modules.setdefault("kornia", kornia)
    sys.modules.setdefault("kornia.color", color)

    class Extractor(torch.nn.Module):  # utils.py:130-134: conf = default_conf overridden by kwargs
        def __init__(self, **conf):
            super().__init__()
            self.conf = SimpleNamespace(**{**self.default_conf, **conf})

    pkg = types.ModuleType("lg_ref_pkg")
    pkg.__path__ = []
    utils = types.ModuleType("lg_ref_pkg.utils")
    utils.Extractor = Extractor
    sys.modules["lg_ref_pkg"] = pkg
    sys.modules["lg_ref_pkg.utils"] = utils
    torch.hub.load_state_dict_from_url = lambda *a, **k: weights
    spec = importlib.util.spec_from_file_location("lg_ref_pkg.superpoint", REF)
    mod = importlib.util.module_from_spec(spec)
    sys.modules["lg_ref_pkg.superpoint"] = mod
    spec.loader.exec_module(mod)
    return mod


def main():
    torch.set_grad_enabled(False)
    weights = sps.make_superpoint_state_dict(0)
    ref = load_reference(weights)
    os.makedirs(OUT, exist_ok=True)
    only = set(sys.argv[1:])  # optional: names of the cases to (re)generate
    grid_sample = torch.nn.functional.grid_sample
    for name, rc in CASES.items():
        if only and name not in only:
            continue
        image = sps.make_image(rc["h"], rc["w"], rc["b"], rc["seed"])
        model = ref.SuperPoint(**rc["conf"]).eval()
        if rc["b"] == 1 or rc["conf"].get("max_num_keypoints"):
            out = model({"image": image})
            res = {k: [t.clone() for t in out[k]] for k in ("keypoints", "keypoint_scores", "descriptors")}
            # keep the fixtures small: above 600 keypoints only every 4th descriptor row is stored
            res["desc_stride"] = [4 if t.shape[0] > 600 else 1 for t in res["descriptors"]]
            res["descriptors"] = [t[::st].clone() for t, st in zip(res["descriptors"], res["desc_stride"])]
            # The same forward in float64 (float64/<name>.pt: keypoints and scores): fp32 scores depend on the
            # convolutions' summation order, which varies with the host CPU and thread count by more than the oracle
            # test's tolerance; float64 scores do not.  superpoint.py:210 casts the keypoints to float32, so the sampling
            # grid is cast to the descriptor map's dtype.
            torch.nn.functional.grid_sample = lambda inp, grid, *a, **k: grid_sample(inp, grid.to(inp.dtype), *a, **k)
            try:
                out64 = model.double()({"image": image.double()})
            finally:
                torch.nn.functional.grid_sample = grid_sample
            res64 = {k: [t.clone() for t in out64[k]] for k in ("keypoints", "keypoint_scores")}
        else:
            raise ValueError("batched cases need max_num_keypoints (the reference stacks per-image results)")
        fix = {
            "recipe": rc,
            "conf": {k: getattr(model.conf, k) for k in ("nms_radius", "max_num_keypoints", "detection_threshold", "remove_borders")},
            "image_checksum": synth.checksum(image),
            "weights_checksum": {k: synth.checksum(v) for k, v in weights.items() if k.startswith(("conv1a", "convPb", "convDb"))},
            "out": res,
        }
        torch.save(fix, os.path.join(OUT, name + ".pt"))
        os.makedirs(os.path.join(OUT, "float64"), exist_ok=True)
        torch.save(res64, os.path.join(OUT, "float64", name + ".pt"))
        print(name, [tuple(t.shape) for t in res["keypoints"]], [tuple(t.shape) for t in res["descriptors"]], "max score", float(max(t.max() for t in res["keypoint_scores"])))


if __name__ == "__main__":
    main()
