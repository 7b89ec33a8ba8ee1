"""Times the fused Bottleneck kernel at the network's shapes (XRSEG_DBG_TIME=1 prints the last of five launches)."""
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
os.environ["XRSEG_DBG_TIME"] = "1"
from xr_image_segmentation_b200 import inference as I  # noqa: E402

rng = np.random.default_rng(0)
for (B, c1, cm, c2, h, w) in [(64, 16, 8, 16, 160, 160), (64, 32, 16, 32, 80, 80), (64, 32, 16, 32, 160, 160)]:
    x = rng.standard_normal((B, c1, h, w), dtype=np.float32)
    w1 = rng.standard_normal((cm, c1, 3, 3), dtype=np.float32) * 0.1
    w2 = rng.standard_normal((c2, cm, 3, 3), dtype=np.float32) * 0.1
    y = I.debug_bottleneck(x, w1, np.zeros(cm, np.float32), w2, np.zeros(c2, np.float32), residual=True)
    print(B, c1, cm, c2, h, w, "finite", bool(np.isfinite(y).all()), flush=True)
