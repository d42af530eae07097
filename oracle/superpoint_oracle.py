"""CPU oracle for the SuperPoint extractor forward (SURVEY.md 8f1) -- TEST INFRASTRUCTURE ONLY.

Groundwork for the next row of the scope table: a functional restatement (plain torch ops on explicit
weight tensors, no nn.Module) of ``SuperPoint.forward`` in /root/reference/lightglue/superpoint.py,
pinned by fixtures generated from the reference file itself (``oracle/make_golden_superpoint.py`` ->
``tests/golden/sp_*.pt``; ``tests/test_superpoint_oracle_golden.py``).  No CUDA path exists for it yet; only
``tests/`` may import this module.

Line numbers below refer to /root/reference/lightglue/superpoint.py.  Not restated: image loading /
resizing (utils.py ``ImagePreprocessor``, kornia) and the RGB->gray conversion (kornia, absent here).
"""
from __future__ import annotations

from typing import Dict, List, Optional

import torch
import torch.nn.functional as F

ENCODER = ("conv1a", "conv1b", "conv2a", "conv2b", "conv3a", "conv3b", "conv4a", "conv4b")  # 137-147, 171-181
POOL_AFTER = ("conv1b", "conv2b", "conv3b")                                                   # 173, 176, 179
CELL = 8  # three 2x2 poolings: one descriptor / one 65-way detector cell per 8x8 pixels


def conv_relu(w: Dict[str, torch.Tensor], name: str, x: torch.Tensor, relu: bool = True) -> torch.Tensor:
    weight = w[f"{name}.weight"]
    y = F.conv2d(x, weight, w[f"{name}.bias"], stride=1, padding=weight.shape[-1] // 2)  # 3x3 pad 1 / 1x1 pad 0 (137-153)
    return F.relu(y) if relu else y


def encoder(w: Dict[str, torch.Tensor], image: torch.Tensor) -> torch.Tensor:
    """Shared VGG-style encoder (171-181): [B,1,H,W] -> [B,128,H/8,W/8]."""
    x = image
    for name in ENCODER:
        x = conv_relu(w, name, x)
        if name in POOL_AFTER:
            x = F.max_pool2d(x, kernel_size=2, stride=2)
    return x


def dense_scores(w: Dict[str, torch.Tensor], feat: torch.Tensor) -> torch.Tensor:
    """Detector head (184-190): 65-way softmax per cell, dustbin dropped, 64 channels unfolded to the 8x8
    pixels of the cell (channel c -> row c // 8, column c % 8) -> [B, H, W]."""
    logits = conv_relu(w, "convPb", conv_relu(w, "convPa", feat), relu=False)
    prob = torch.softmax(logits, dim=1)[:, :-1]
    b, _, hc, wc = prob.shape
    prob = prob.permute(0, 2, 3, 1).reshape(b, hc, wc, CELL, CELL)
    return prob.permute(0, 1, 3, 2, 4).reshape(b, hc * CELL, wc * CELL)


def simple_nms(scores: torch.Tensor, radius: int) -> torch.Tensor:
    """52-68: keep local maxima of a (2r+1)^2 window, then twice re-admit maxima of what is left outside the
    suppression zones of the maxima found so far."""
    def window_max(x):
        return F.max_pool2d(x, kernel_size=2 * radius + 1, stride=1, padding=radius)

    zero = torch.zeros_like(scores)
    keep = scores == window_max(scores)
    for _ in range(2):
        suppressed = window_max(keep.float()) > 0
        rest = torch.where(suppressed, zero, scores)
        keep = keep | ((rest == window_max(rest)) & ~suppressed)
    return torch.where(keep, scores, zero)


def sample_descriptors(kpts_xy: torch.Tensor, dense: torch.Tensor, cell: int = CELL) -> torch.Tensor:
    """79-96: bilinear sampling of the coarse descriptor map at pixel keypoints (x, y), then L2 norm.
    kpts_xy [K, 2], dense [C, Hc, Wc] -> [K, C]."""
    c, hc, wc = dense.shape
    k = kpts_xy - cell / 2 + 0.5
    k = k / torch.tensor([wc * cell - cell / 2 - 0.5, hc * cell - cell / 2 - 0.5]).to(k)
    k = k * 2 - 1
    out = F.grid_sample(dense[None], k.view(1, 1, -1, 2).to(dense), mode="bilinear", align_corners=True)
    return F.normalize(out.reshape(c, -1), p=2, dim=0).t().contiguous()


def forward(
    w: Dict[str, torch.Tensor],
    image: torch.Tensor,
    *,
    nms_radius: int = 4,
    max_num_keypoints: Optional[int] = None,
    detection_threshold: float = 0.0005,
    remove_borders: int = 4,
) -> Dict[str, List[torch.Tensor]]:
    """SuperPoint.forward (163-227) on a grayscale batch [B,1,H,W] (any H, W >= 8; max_pool2d floors).  Returns per-image
    lists (the reference stacks them, which needs equal counts): keypoints [K,2] (x, y), keypoint_scores [K],
    descriptors [K,256]."""
    feat = encoder(w, image)
    scores = simple_nms(dense_scores(w, feat), nms_radius)
    if remove_borders:  # 193-198
        p = remove_borders
        scores[:, :p] = -1
        scores[:, :, :p] = -1
        scores[:, -p:] = -1
        scores[:, :, -p:] = -1
    dense = F.normalize(conv_relu(w, "convDb", conv_relu(w, "convDa", feat), relu=False), p=2, dim=1)  # 220-222
    kpts, kscores, descs = [], [], []
    for b in range(image.shape[0]):
        ys, xs = torch.where(scores[b] > detection_threshold)  # 201-208: row-major order
        sc = scores[b][ys, xs]
        if max_num_keypoints is not None and max_num_keypoints < sc.numel():  # 71-76: top-k, sorted by score
            sc, idx = torch.topk(sc, max_num_keypoints, dim=0, sorted=True)
            ys, xs = ys[idx], xs[idx]
        xy = torch.stack([xs, ys], dim=-1).float()  # 217-218: (h, w) -> (x, y)
        kpts.append(xy)
        kscores.append(sc)
        descs.append(sample_descriptors(xy, dense[b]))
    return {"keypoints": kpts, "keypoint_scores": kscores, "descriptors": descs}
