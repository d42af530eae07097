"""Generate tests/golden/*.pt by running the UNMODIFIED reference matcher in this container.

    python oracle/make_golden.py [batch_semantics]   # needs the reference checkout (REF); CPU, fp32

The reference package cannot be imported as a package here (``import lightglue`` pulls kornia, which
is absent), but ``lightglue/lightglue.py`` only needs numpy + torch, so it is loaded by file path
(SURVEY.md §8c).  ``/root/reference`` does not exist on the GPU box: nothing else in the repo reads
it; tests consume only the committed fixtures.

Each fixture stores the *recipe* (seeds, shapes, conf), checksums of the regenerated inputs/weights
(so a fixture can never silently be compared against different data) and the reference outputs.
Weights are not stored (47 MB); they are regenerated from ``lightglue_b200.synth.make_state_dict``.
"""
from __future__ import annotations

import importlib.util
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from lightglue_b200 import synth  # noqa: E402

REF = "/root/reference/lightglue/lightglue.py"
OUT = os.path.join(ROOT, "tests", "golden")

# name -> recipe.  `pruning_threshold` is written into the reference's class-level
# pruning_keypoint_thresholds["cpu"] (lightglue.py:339-344) exactly as benchmark.py:178-181 mutates it.
CASES = {
    "c1_n512": dict(n=512, d=256, b=1, seed=1000, adaptive=False),
    "ragged_b2": dict(n=512, m=300, d=256, b=2, seed=1001, adaptive=False),
    "n2048": dict(n=2048, d=256, b=1, seed=1002, adaptive=False),
    "disk_d128": dict(n=640, d=128, b=1, seed=1003, adaptive=False),
    "sift_scale_ori": dict(n=256, d=128, b=1, seed=1004, adaptive=False, scale_ori=True),
    "nosize": dict(n=384, d=256, b=1, seed=1005, adaptive=False, drop_size=True),
    "adaptive_n512": dict(n=512, d=256, b=1, seed=1006, adaptive=True, pruning_threshold=-1),
    "adaptive_n1200_th1024": dict(n=1200, m=1100, d=256, b=1, seed=1007, adaptive=True, pruning_threshold=1024),
    "depth_only_n512": dict(n=512, d=256, b=1, seed=1008, adaptive=True, width_off=True, pruning_threshold=-1),
    "width_only_n512": dict(n=512, d=256, b=1, seed=1009, adaptive=True, depth_off=True, pruning_threshold=-1),
    "empty_m0": dict(n=64, m=0, d=256, b=1, seed=1010, adaptive=False),
}


def load_reference():
    spec = importlib.util.spec_from_file_location("lg_ref", REF)
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def conf_of(rc: dict) -> dict:
    adaptive = rc.get("adaptive", False)
    depth = 0.95 if adaptive and not rc.get("depth_off") else -1
    width = 0.99 if adaptive and not rc.get("width_off") else -1
    return dict(depth_confidence=depth, width_confidence=width, filter_threshold=0.1)


def build_inputs(rc: dict):
    data, perm = synth.make_pair(
        rc["n"], d=rc["d"], b=rc["b"], seed=rc["seed"], m=rc.get("m"), scale_ori=rc.get("scale_ori", False)
    )
    if rc.get("drop_size"):
        for k in ("image0", "image1"):
            data[k].pop("image_size")
    sd = synth.make_state_dict(
        seed=0, input_dim=rc["d"], adaptive=rc.get("adaptive", False), add_scale_ori=rc.get("scale_ori", False)
    )
    return data, perm, sd


def batch_semantics(ref) -> None:
    """batch_early_exit.pt: the reference's adaptive depth on B=2 batches (tests/test_reference_batch_semantics.py).
    Weights with which pair 41 exits early alone and pair 42 does not; outputs of each pair alone, of pair 41 twice in
    one batch and of the two together."""
    rc = dict(weight_seed=2, n=192, seeds=(41, 42), depth_confidence=0.95, width_confidence=-1)
    sd = synth.make_state_dict(adaptive=True, seed=rc["weight_seed"])
    model = ref.LightGlue(features=None, depth_confidence=rc["depth_confidence"],
                          width_confidence=rc["width_confidence"]).eval()
    missing, unexpected = model.load_state_dict(sd, strict=False)
    assert not unexpected and all(k == "confidence_thresholds" for k in missing), (missing, unexpected)
    p41, p42 = (synth.make_pair(rc["n"], b=1, seed=s)[0] for s in rc["seeds"])

    def cat(pairs):
        return {k: {kk: torch.cat([p[k][kk] for p in pairs]) for kk in pairs[0][k]} for k in ("image0", "image1")}

    outs = {}
    for name, data in (("alone41", p41), ("alone42", p42), ("twice41", cat([p41, p41])), ("mixed", cat([p41, p42]))):
        out = model(data)
        outs[name] = {"stop": int(out["stop"]), "matches0": out["matches0"].to(torch.int32),
                      "matches1": out["matches1"].to(torch.int32), "matching_scores0": out["matching_scores0"],
                      "matching_scores1": out["matching_scores1"]}
        print(f"batch_early_exit/{name:8s} stop={outs[name]['stop']}")
    fix = {
        "recipe": rc,
        "weights_checksum": {k: synth.checksum(v) for k, v in list(sd.items())[:4]},
        "inputs_checksum": {s: {"k0": synth.checksum(p["image0"]["keypoints"]), "d1": synth.checksum(p["image1"]["descriptors"])}
                            for s, p in zip(rc["seeds"], (p41, p42))},
        "out": outs,
    }
    torch.save(fix, os.path.join(OUT, "batch_early_exit.pt"))


def main() -> None:
    torch.set_grad_enabled(False)
    torch.set_num_threads(os.cpu_count() or 1)
    ref = load_reference()
    os.makedirs(OUT, exist_ok=True)
    batch_semantics(ref)
    if sys.argv[1:] == ["batch_semantics"]:
        return
    for name, rc in CASES.items():
        data, perm, sd = build_inputs(rc)
        conf = conf_of(rc)
        ref.LightGlue.pruning_keypoint_thresholds["cpu"] = rc.get("pruning_threshold", -1)
        model = ref.LightGlue(
            features=None, input_dim=rc["d"], add_scale_ori=rc.get("scale_ori", False), **conf
        ).eval()
        missing, unexpected = model.load_state_dict(sd, strict=False)
        assert not unexpected and all(k == "confidence_thresholds" for k in missing), (missing, unexpected)
        layer_sums = []

        def hook(_m, _i, o, acc=layer_sums):
            acc.append((synth.checksum(o[0]), synth.checksum(o[1]), tuple(o[0].shape), tuple(o[1].shape)))

        hs = [t.register_forward_hook(hook) for t in model.transformers]
        out = model(data)
        for h in hs:
            h.remove()
        fix = {
            "recipe": rc,
            "conf": conf,
            "weights_checksum": {k: synth.checksum(v) for k, v in list(sd.items())[:4]},
            "inputs_checksum": {
                "k0": synth.checksum(data["image0"]["keypoints"]),
                "d1": synth.checksum(data["image1"]["descriptors"]),
            },
            "perm": perm.to(torch.int32),
            "layer_checksums": layer_sums,
            "out": {
                "matches0": out["matches0"].to(torch.int32),
                "matches1": out["matches1"].to(torch.int32),
                "matching_scores0": out["matching_scores0"],
                "matching_scores1": out["matching_scores1"],
                "stop": int(out["stop"]),
                "matches": [t.to(torch.int32) for t in out["matches"]],
                "scores": [t for t in out["scores"]],
                "prune0": out["prune0"],
                "prune1": out["prune1"],
                "dtypes": {k: str(v.dtype) for k, v in out.items() if torch.is_tensor(v)},
                "matches_is_tensor": torch.is_tensor(out["matches"]),
            },
        }
        nm = [int((t > -1).sum()) for t in out["matches0"]]
        correct = 0
        if rc.get("m") is None:
            m1 = out["matches1"]
            correct = int(((m1 == perm) & (m1 > -1)).sum())
        hist = torch.bincount(out["prune0"].flatten().long()).tolist()
        print(f"{name:24s} stop={out['stop']} matches={nm} correct={correct} prune0_hist={hist}")
        torch.save(fix, os.path.join(OUT, name + ".pt"))


if __name__ == "__main__":
    main()
