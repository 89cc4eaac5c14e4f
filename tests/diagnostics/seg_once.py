"""One normalize + U-Net + instances pass on a 2048 x 2048 field (for ncu launch lists / captures of the
segmentation kernels).  The (prob, dist) maps of the instance step are the ellipse maps of the parity tests."""
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
from oracle import stardist as sd                      # noqa: E402
import test_gpu_stardist as T                          # noqa: E402
from cell_image_analysis_b200.stardist import StarDist2D   # noqa: E402
from cell_image_analysis_b200 import synth             # noqa: E402

H = W = int(os.environ.get("SEG_SIDE", "2048"))
w = sd.random_model(T.CFG, seed=11)
m = StarDist2D.from_arrays(T.CFG, w, {"prob": 0.479071, "nms": 0.3})
for opt in ("seg_conv_tma", "seg_conv_ws"):      # A/B runs: SEG_CONV_TMA=0 etc.
    if os.environ.get(opt.upper()):
        m.engine.set_option(opt, float(os.environ[opt.upper()]))
green, _ = synth.make_field(0, 2048, 2048, *synth.FIELD_CONFIGS["config1"][2:])
green = np.ascontiguousarray(green[:H, :W])
cells = T._ellipse_field(H, W, max(2, int(23 * H / 2048)), 3)
prob, dist = sd.star_maps_from_ellipses(H, W, 2, cells)
pd, dd = torch.from_numpy(prob).cuda(), torch.from_numpy(dist).cuda()
for _ in range(int(os.environ.get("SEG_REPS", "2"))):
    x = m.normalize_device(green)
    m.predict(x)
    labels, n = m.instances_from_prediction((H, W), pd, dd)
torch.cuda.synchronize()
print("instances", n)
