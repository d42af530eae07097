"""Small forwards of every precision mode / adaptive setting, meant to run under compute-sanitizer."""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from lightglue_b200 import LightGlue, synth
torch.set_grad_enabled(False)
for prec in ("bf16", "bf16x3", "fp32"):
    for adaptive in (False, True):
        sd = synth.make_state_dict(adaptive=adaptive)
        kw = {} if adaptive else dict(depth_confidence=-1, width_confidence=-1)
        m = LightGlue(features=None, precision=prec, **kw); m.load_state_dict(sd, strict=False); m = m.cuda()
        m.pruning_keypoint_thresholds = dict(LightGlue.pruning_keypoint_thresholds, flash=-1)
        # (300, 200): three 128-row tiles per sequence -> final_proj and the assignment sweeps give every sequence a
        # fourth, dead row slot, so that no CTA pair straddles two sequences; (512, 512): an even number of tiles
        for n, mm in ((300, 200), (512, 512)):
            d, _ = synth.make_pair(n, m=mm, b=2, seed=5)
            out = m({k: {kk: vv.cuda() for kk, vv in v.items()} for k, v in d.items()})
            torch.cuda.synchronize()
            print(prec, adaptive, (n, mm), int((out["matches0"] > -1).sum()), out["stop"], "timeout", hex(m.debug_timeout_code()), flush=True)
m = LightGlue(features=None, precision="bf16x3", depth_confidence=-1, width_confidence=-1).cuda()
full = m.log_assignment_matrix(2, torch.randn(1, 260, 256).cuda(), torch.randn(1, 300, 256).cuda())[0]
torch.cuda.synchronize()
print("matrix", tuple(full.shape), flush=True)
