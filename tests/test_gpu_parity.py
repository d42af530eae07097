"""GPU parity: the CUDA path (through the C ABI) against the reference-generated golden fixtures
and against the CPU oracle on the same seeded inputs.

Tolerances (north star: "bit-exact match indices when pruning is disabled, scores within 1e-3"):
  precision="fp32"  : identical match indices, |dscore| <= 1e-4 on every fixture
  precision="bf16x3": identical match indices, |dscore| <= 1e-3
  precision="bf16"  : |dscore| <= 8e-2, index flips reported and bounded (operand rounding; SURVEY §7.3)
"""
import pytest
import torch

from lightglue_b200 import LightGlue, synth
from lightglue_b200.ragged import pad_pairs, split_outputs
from oracle import lightglue_oracle as oracle
from tests.helpers import ALL_CASES, compare_outputs, forward_kwargs, load_case

pytestmark = pytest.mark.gpu


def to_cuda(data):
    return {k: {kk: vv.cuda() for kk, vv in v.items()} for k, v in data.items()}


def build(fix, sd, precision):
    rc, conf = fix["recipe"], fix["conf"]
    m = LightGlue(
        features=None, input_dim=rc["d"], add_scale_ori=rc.get("scale_ori", False), precision=precision, **conf
    )
    m.load_state_dict(sd, strict=False)
    m = m.eval().cuda()
    # same pruning threshold the fixture was generated with (benchmark.py:178-181 mutates this dict too)
    m.pruning_keypoint_thresholds = dict(LightGlue.pruning_keypoint_thresholds, flash=rc.get("pruning_threshold", -1))
    return m


@pytest.mark.parametrize("name", ALL_CASES)
def test_fp32_path_matches_reference_fixture(name):
    fix, data, sd = load_case(name)
    m = build(fix, sd, "fp32")
    out = m(to_cuda(data))
    gold = fix["out"]
    adaptive = fix["recipe"].get("adaptive", False)
    compare_outputs(out, gold, score_tol=1e-4)
    assert str(out["prune0"].dtype) == gold["dtypes"]["prune0"]
    assert out["matches0"].dtype == torch.int64 and out["matching_scores0"].dtype == torch.float32
    assert torch.equal(out["prune0"].cpu().double(), gold["prune0"].double())
    assert torch.equal(out["prune1"].cpu().double(), gold["prune1"].double())
    assert torch.is_tensor(out["matches"]) == gold["matches_is_tensor"]
    if not gold["matches_is_tensor"]:
        for a, b, sa, sb in zip(out["matches"], gold["matches"], out["scores"], gold["scores"]):
            assert torch.equal(a.cpu().to(torch.int32), b)
            if sa.numel():
                assert float((sa.cpu() - sb).abs().max()) <= 1e-4
    del adaptive


def test_log_assignment_matrix_matches_oracle():
    torch.manual_seed(5)
    sd = synth.make_state_dict()
    m = LightGlue(features=None, precision="fp32", depth_confidence=-1, width_confidence=-1)
    m.load_state_dict(sd, strict=False)
    m = m.cuda()
    x0 = torch.randn(2, 200, 256)
    x1 = torch.randn(2, 333, 256)
    full, m0, m1, ms0, ms1 = m.log_assignment_matrix(4, x0.cuda(), x1.cuda())
    ref = oracle.log_assignment(sd, 4, x0, x1)
    assert float((full.cpu() - ref).abs().max()) < 2e-4
    r0, r1, rs0, rs1 = oracle.filter_matches(ref, 0.1)
    assert torch.equal(m0.cpu(), r0) and torch.equal(m1.cpu(), r1)
    assert float((ms0.cpu() - rs0).abs().max()) < 1e-4 and float((ms1.cpu() - rs1).abs().max()) < 1e-4


def test_batched_equals_single_and_invariants_n2048():
    """Size-independent properties at the benchmark shape (N=2048): batching does not change results,
    matches are mutual, scores obey the threshold, the compact list is ordered."""
    sd = synth.make_state_dict()
    m = LightGlue(features=None, precision="fp32", depth_confidence=-1, width_confidence=-1)
    m.load_state_dict(sd, strict=False)
    m = m.cuda()
    data, perm = synth.make_pair(2048, b=3, seed=4242)
    out = m(to_cuda(data))
    for b in range(3):
        one = {k: {kk: vv[b : b + 1] for kk, vv in v.items()} for k, v in data.items()}
        o1 = m(to_cuda(one))
        assert torch.equal(o1["matches0"][0], out["matches0"][b])
        assert float((o1["matching_scores0"][0] - out["matching_scores0"][b]).abs().max()) < 1e-6
        m0, m1 = out["matches0"][b], out["matches1"][b]
        idx = torch.where(m0 > -1)[0]
        assert torch.equal(m1[m0[idx]], idx)
        assert bool((out["matching_scores0"][b][idx] > 0.1).all())
        assert bool((out["matching_scores0"][b][m0 == -1] <= 0.1).logical_or(m0[m0 == -1] == -1).all())
        pairs = out["matches"][b]
        assert pairs.shape[0] == idx.numel() and bool((pairs[1:, 0] > pairs[:-1, 0]).all())
        # the matcher recovers the planted permutation
        good = (out["matches1"][b].cpu() == perm[b]) & (out["matches1"][b].cpu() > -1)
        assert int(good.sum()) > 300


def test_permutation_equivariance():
    sd = synth.make_state_dict()
    m = LightGlue(features=None, precision="fp32", depth_confidence=-1, width_confidence=-1)
    m.load_state_dict(sd, strict=False)
    m = m.cuda()
    data, _ = synth.make_pair(700, seed=77)
    out = m(to_cuda(data))
    g = torch.Generator().manual_seed(3)
    p = torch.randperm(700, generator=g)
    d2 = {"image0": {k: (v[:, p] if v.shape[1:2] == (700,) else v) for k, v in data["image0"].items()}, "image1": data["image1"]}
    out2 = m(to_cuda(d2))
    assert torch.equal(out2["matches0"][0].cpu(), out["matches0"][0].cpu()[p])


TC_CASES = ["c1_n512", "ragged_b2", "n2048", "disk_d128", "sift_scale_ori", "nosize"]


@pytest.mark.parametrize("name", TC_CASES)
def test_bf16x3_path_index_exact(name):
    """tcgen05 path with split-bf16 linears: identical match indices, scores within 1e-3."""
    fix, data, sd = load_case(name)
    out = build(fix, sd, "bf16x3")(to_cuda(data))
    flips, dmax = compare_outputs(out, fix["out"], score_tol=1e-3)
    print(f"[bf16x3] {name}: flips={flips} max|dscore|={dmax:.2e}")


@pytest.mark.parametrize("name", TC_CASES)
def test_bf16_path_bounded_error(name):
    """tcgen05 path with plain bf16 operands: operand rounding moves scores by O(1e-2) (SURVEY §7.3), so
    a few matches whose score sits at filter_threshold may flip; bounded and reported, not hidden."""
    fix, data, sd = load_case(name)
    out = build(fix, sd, "bf16")(to_cuda(data))
    flips, dmax = compare_outputs(out, fix["out"], score_tol=8e-2, exact_indices=False)
    npts = fix["out"]["matches0"].numel() + fix["out"]["matches1"].numel()
    print(f"[bf16] {name}: flips={flips}/{npts} max|dscore|={dmax:.2e}")
    assert flips <= max(4, npts // 50)


@pytest.mark.parametrize("prec", ["bf16x3", "bf16"])
def test_tc_adaptive_runs_and_agrees(prec):
    """Adaptive depth/width on the tensor-core path: decisions are threshold tests on fp values, so
    small arithmetic differences may move a few points; stop layer must agree, prune histograms nearly."""
    fix, data, sd = load_case("adaptive_n512")
    out = build(fix, sd, prec)(to_cuda(data))
    gold = fix["out"]
    assert abs(int(out["stop"]) - gold["stop"]) <= (0 if prec == "bf16x3" else 1)
    if int(out["stop"]) == gold["stop"]:
        diff = int((out["prune0"].cpu() != gold["prune0"]).sum())
        print(f"[{prec}] adaptive: prune0 differences {diff}/512")
        assert diff <= (4 if prec == "bf16x3" else 40)


TC_ADAPTIVE_CASES = ["adaptive_n512", "adaptive_n1200_th1024", "depth_only_n512", "width_only_n512"]


@pytest.mark.parametrize("name", TC_ADAPTIVE_CASES)
def test_index_exact_tc_modes_adaptive_identical_decisions(name):
    """Every adaptive fixture on the index-exact tensor-core path: identical stop layer, identical prune counters,
    identical match indices (no +-1, no allowance)."""
    fix, data, sd = load_case(name)
    gold = fix["out"]
    out = build(fix, sd, "bf16x3")(to_cuda(data))
    assert int(out["stop"]) == int(gold["stop"])
    assert torch.equal(out["prune0"].cpu().double(), gold["prune0"].double())
    assert torch.equal(out["prune1"].cpu().double(), gold["prune1"].double())
    compare_outputs(out, gold, score_tol=1e-3)


def test_index_exact_adaptive_n2048_default_flash_threshold():
    """BASELINE config 3 (N=2048, depth 0.95 / width 0.99, pruning threshold 1536) on the index-exact tensor-core path
    against the oracle: identical stop, prune counters and match indices."""
    sd = synth.make_state_dict(adaptive=True)
    data, _ = synth.make_pair(2048, b=1, seed=41)
    ref = oracle.forward(sd, data, depth_confidence=0.95, width_confidence=0.99, pruning_threshold=1536)
    m = LightGlue(features=None, precision="bf16x3")
    m.load_state_dict(sd, strict=False)
    out = m.cuda()(to_cuda(data))
    assert int(out["stop"]) == int(ref["stop"])
    assert torch.equal(out["prune0"].cpu(), ref["prune0"]) and torch.equal(out["prune1"].cpu(), ref["prune1"])
    assert torch.equal(out["matches0"].cpu(), ref["matches0"]) and torch.equal(out["matches1"].cpu(), ref["matches1"])
    assert float((out["matching_scores0"].cpu() - ref["matching_scores0"]).abs().max()) < 1e-3


def test_index_exact_batched_b32_equals_single_n2048():
    """BASELINE config 2 shape (B=32, N=2048) on the index-exact tensor-core path: every pair of the batch gives the
    result of its own B=1 call (bit-identical indices and scores: the kernels never mix pairs)."""
    sd = synth.make_state_dict()
    m = LightGlue(features=None, precision="bf16x3", depth_confidence=-1, width_confidence=-1)
    m.load_state_dict(sd, strict=False)
    m = m.cuda()
    data, _ = synth.make_pair(2048, b=32, seed=777)
    cd = to_cuda(data)
    out = m(cd)
    for b in (0, 13, 31):
        one = {k: {kk: vv[b : b + 1].contiguous() for kk, vv in v.items()} for k, v in cd.items()}
        o1 = m(one)
        assert torch.equal(o1["matches0"][0], out["matches0"][b]) and torch.equal(o1["matches1"][0], out["matches1"][b])
        assert float((o1["matching_scores0"][0] - out["matching_scores0"][b]).abs().max()) <= 1e-6


@pytest.mark.parametrize("prec,tol", [("fp32", 2e-4), ("bf16x3", 2e-3)])
def test_per_layer_residual_stream_against_oracle(prec, tol):
    """Block-level parity (SURVEY 4.1): the residual stream after every transformer layer (what a forward hook on the
    reference's transformers[i] sees, lightglue.py:541) against the oracle's, through lg_debug_capture_layers."""
    fix, data, sd = load_case("c1_n512")
    ref = oracle.forward(sd, data, return_layers=True)
    m = build(fix, sd, prec)
    out, layers = m.forward_with_layers(to_cuda(data))
    assert len(layers) == len(ref["layers"]) == 9
    worst = 0.0
    for i, ((a0, a1), (r0, r1)) in enumerate(zip(layers, ref["layers"])):
        scale = max(float(r0.abs().max()), 1.0)
        d = max(float((a0.cpu() - r0).abs().max()), float((a1.cpu() - r1).abs().max())) / scale
        worst = max(worst, d)
        assert d <= tol, f"layer {i}: relative deviation {d:.2e} > {tol}"
    print(f"[{prec}] per-layer max relative deviation {worst:.2e}")


@pytest.mark.parametrize("prec", ["fp32", "bf16x3"])
def test_batched_early_exit_is_decided_per_pair(prec):
    """The documented deviation for B > 1 (tests/test_reference_batch_semantics.py shows what the reference does instead):
    in one batch {pair 41, pair 41 again, pair 42} every pair exits where it exits alone -- the oracle's B = 1 result --
    and returns its own B = 1 matches; ``stop`` is the maximum, ``stops`` the per-pair list."""
    sd = synth.make_state_dict(adaptive=True, seed=2)
    pairs = [synth.make_pair(192, b=1, seed=s)[0] for s in (41, 41, 42)]
    refs = [oracle.forward(sd, p, depth_confidence=0.95, width_confidence=-1) for p in pairs]
    assert [int(r["stop"]) for r in refs] == [6, 6, 9]
    m = LightGlue(features=None, precision=prec, depth_confidence=0.95, width_confidence=-1)
    m.load_state_dict(sd, strict=False)
    m = m.cuda()
    batch = {k: {kk: torch.cat([p[k][kk] for p in pairs]) for kk in pairs[0][k]} for k in ("image0", "image1")}
    out = m(to_cuda(batch))
    assert out["stops"] == [6, 6, 9] and int(out["stop"]) == 9
    for i, r in enumerate(refs):
        assert torch.equal(out["matches0"][i].cpu(), r["matches0"][0]) and torch.equal(out["matches1"][i].cpu(), r["matches1"][0])
        assert float((out["matching_scores0"][i].cpu() - r["matching_scores0"][0]).abs().max()) < 1e-3


def test_batched_early_exit_with_odd_tile_count():
    """Pairs that exit at different layers in one tensor-core batch whose padded length is an odd number of 128-row tiles
    (the three pairs above and a 300-point pair: Lp = 384, three tiles).  final_proj takes the head of each pair's own exit
    layer and the assignment sweeps the pair's own partner, so a CTA pair must never hold tiles of two sequences: every
    pair returns its own B = 1 result."""
    sd = synth.make_state_dict(adaptive=True, seed=2)
    pairs = [synth.make_pair(n, b=1, seed=s)[0] for n, s in ((192, 41), (192, 41), (192, 42), (300, 43))]
    refs = [oracle.forward(sd, p, depth_confidence=0.95, width_confidence=-1) for p in pairs]
    assert [int(r["stop"]) for r in refs] == [6, 6, 9, 6]
    m = LightGlue(features=None, precision="bf16x3", depth_confidence=0.95, width_confidence=-1)
    m.load_state_dict(sd, strict=False)
    m = m.cuda()
    data = pad_pairs([to_cuda(p) for p in pairs])
    out = m(data)
    assert out["stops"] == [6, 6, 9, 6]
    for got, r in zip(split_outputs(out, data["image0"]["num_keypoints"], data["image1"]["num_keypoints"]), refs):
        assert torch.equal(got["matches0"].cpu(), r["matches0"]) and torch.equal(got["matches1"].cpu(), r["matches1"])
        assert float((got["matching_scores0"].cpu() - r["matching_scores0"]).abs().max()) < 1e-3


def test_pruned_to_zero_points_ends_the_pair_like_the_reference():
    """Pruning that leaves an image without points: the reference breaks at the top of the next layer and answers from
    its empty branch (lightglue.py:539-540, 568-588): nothing matched, stop = that layer + 1."""
    sd = synth.make_state_dict(adaptive=True)
    for k in list(sd):  # matchability far below any threshold: every point is pruned at the first opportunity
        if "matchability.bias" in k:
            sd[k] = sd[k] - 200.0
    data, _ = synth.make_pair(300, b=1, seed=91)
    ref = oracle.forward(sd, data, depth_confidence=-1, width_confidence=0.99, pruning_threshold=-1)
    assert int((ref["matches0"] > -1).sum()) == 0
    for prec in ("fp32", "bf16x3"):
        m = LightGlue(features=None, precision=prec, depth_confidence=-1, width_confidence=0.99)
        m.load_state_dict(sd, strict=False)
        m = m.cuda()
        m.pruning_keypoint_thresholds = dict(LightGlue.pruning_keypoint_thresholds, flash=-1)
        out = m(to_cuda(data))
        assert int(out["stop"]) == int(ref["stop"]), (prec, out["stop"], ref["stop"])
        assert bool((out["matches0"] == -1).all()) and bool((out["matches1"] == -1).all())
        assert float(out["matching_scores0"].abs().max()) == 0.0
        assert torch.equal(out["prune0"].cpu(), ref["prune0"]) and torch.equal(out["prune1"].cpu(), ref["prune1"])


def test_two_devices_in_one_process():
    """Per-device kernel setup (shared-memory opt-in, SM count): a second matcher on another GPU of the same process."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    fix, data, sd = load_case("c1_n512")
    outs = []
    for dev in (0, 1):
        m = LightGlue(features=None, precision="bf16x3", depth_confidence=-1, width_confidence=-1)
        m.load_state_dict(sd, strict=False)
        m = m.eval().to(f"cuda:{dev}")
        outs.append(m({k: {kk: vv.to(f"cuda:{dev}") for kk, vv in v.items()} for k, v in data.items()}))
    assert torch.equal(outs[0]["matches0"].cpu(), outs[1]["matches0"].cpu())
    compare_outputs(outs[1], fix["out"], score_tol=1e-3)


def test_match_stream_equals_direct_forward():
    """The pinned-host streaming API (H2D one batch ahead on a copy stream) returns what forward returns."""
    from lightglue_b200.pipeline import match_stream

    sd = synth.make_state_dict()
    m = LightGlue(features=None, precision="bf16x3", depth_confidence=-1, width_confidence=-1)
    m.load_state_dict(sd, strict=False)
    m = m.cuda()
    batches = []
    for i in range(3):
        d, _ = synth.make_pair(384, b=2, seed=500 + i)
        batches.append({k: {kk: vv.pin_memory() for kk, vv in v.items()} for k, v in d.items()})
    direct = [m(to_cuda(b)) for b in batches]
    streamed = list(match_stream(m, batches))
    assert len(streamed) == 3
    for a, b in zip(direct, streamed):
        assert torch.equal(a["matches0"].cpu(), b["matches0"]) and torch.equal(a["matches1"].cpu(), b["matches1"])
        assert torch.equal(a["matching_scores0"].cpu(), b["matching_scores0"])


@pytest.mark.parametrize("adaptive", [False, True])
def test_cuda_graph_mode_matches_eager(adaptive):
    """conf.cuda_graph replays the whole forward (incl. device-side early exit / pruning) as one graph."""
    name = "adaptive_n512" if adaptive else "c1_n512"
    fix, data, sd = load_case(name)
    rc, conf = fix["recipe"], fix["conf"]
    outs = []
    for g in (False, True):
        m = LightGlue(features=None, input_dim=rc["d"], precision="bf16x3", cuda_graph=g, **conf)
        m.load_state_dict(sd, strict=False)
        m = m.eval().cuda()
        m.pruning_keypoint_thresholds = dict(LightGlue.pruning_keypoint_thresholds, flash=rc.get("pruning_threshold", -1))
        d = to_cuda(data)
        o = m(d)
        o = m(d)  # second call replays the captured graph
        outs.append(o)
    a, b = outs
    assert a["stop"] == b["stop"]
    for k in ("matches0", "matches1", "matching_scores0", "matching_scores1", "prune0", "prune1"):
        assert torch.equal(a[k], b[k]), k
    assert all(torch.equal(x, y) for x, y in zip(a["matches"], b["matches"]))


def test_log_assignment_matrix_tensor_core_variant():
    """The materialising assignment variant on the tensor-core sweep (bf16x3): matrix within 2e-3 of the
    oracle's, identical filter_matches indices."""
    torch.manual_seed(6)
    sd = synth.make_state_dict()
    m = LightGlue(features=None, precision="bf16x3", depth_confidence=-1, width_confidence=-1)
    m.load_state_dict(sd, strict=False)
    m = m.cuda()
    x0 = torch.randn(2, 300, 256)
    x1 = torch.randn(2, 517, 256)
    full, m0, m1, ms0, ms1 = m.log_assignment_matrix(3, x0.cuda(), x1.cuda())
    ref = oracle.log_assignment(sd, 3, x0, x1)
    assert float((full.cpu() - ref).abs().max()) < 2e-3
    r0, r1, rs0, rs1 = oracle.filter_matches(ref, 0.1)
    assert torch.equal(m0.cpu(), r0) and torch.equal(m1.cpu(), r1)
    assert float((ms0.cpu() - rs0).abs().max()) < 1e-3


def test_disk_n4096_against_oracle():
    """BASELINE config 4 shape (DISK d=128, N=4096): index-exact tensor-core mode vs the CPU oracle."""
    sd = synth.make_state_dict(input_dim=128)
    data, _ = synth.make_pair(4096, d=128, b=1, seed=31)
    ref = oracle.forward(sd, data)
    m = LightGlue(features=None, input_dim=128, precision="bf16x3", depth_confidence=-1, width_confidence=-1)
    m.load_state_dict(sd, strict=False)
    out = m.cuda()(to_cuda(data))
    flips = int((out["matches0"].cpu() != ref["matches0"]).sum()) + int((out["matches1"].cpu() != ref["matches1"]).sum())
    dmax = float((out["matching_scores0"].cpu() - ref["matching_scores0"]).abs().max())
    print(f"[bf16x3] disk n4096: flips={flips} max|dscore|={dmax:.2e} matches={int((ref['matches0'] > -1).sum())}")
    assert flips == 0 and dmax < 1e-3


def test_adaptive_n2048_default_flash_threshold():
    """Adaptive depth/width at N=2048 with the reference's default CUDA+flash pruning threshold (1536, lightglue.py:
    339-344, 658-662): pruning only runs while an image has more than 1536 points.  fp32 path vs the oracle."""
    sd = synth.make_state_dict(adaptive=True)
    data, _ = synth.make_pair(2048, b=1, seed=41)
    ref = oracle.forward(sd, data, depth_confidence=0.95, width_confidence=0.99, pruning_threshold=1536)
    m = LightGlue(features=None, precision="fp32")
    m.load_state_dict(sd, strict=False)
    m = m.cuda()
    assert m.pruning_min_kpts(torch.device("cuda")) == 1536
    out = m(to_cuda(data))
    assert int(out["stop"]) == int(ref["stop"])
    assert torch.equal(out["prune0"].cpu(), ref["prune0"]) and torch.equal(out["prune1"].cpu(), ref["prune1"])
    assert torch.equal(out["matches0"].cpu(), ref["matches0"]) and torch.equal(out["matches1"].cpu(), ref["matches1"])
    assert float((out["matching_scores0"].cpu() - ref["matching_scores0"]).abs().max()) < 1e-4
    print("adaptive n2048: stop", out["stop"], "prune0 hist", torch.bincount(out["prune0"].flatten()).tolist())

