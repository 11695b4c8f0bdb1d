#!/usr/bin/env python
"""Hardware probe for the window kernel: max error of a few layer shapes against torch fp32.
   python scripts/win_probe.py"""
import os
import sys

import numpy as np
import torch
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import gpu_util as G  # noqa: E402

CASES = [("c64", 2, 20, 20, 64, 64, 3), ("c32", 2, 20, 20, 32, 32, 3), ("c16", 2, 20, 20, 16, 16, 3),
         ("c128s", 2, 20, 20, 128, 128, 3), ("1x1_64", 2, 20, 20, 64, 64, 1), ("1x1_48", 2, 20, 20, 48, 32, 1)]
for name, B, H, W, cin, cout, k in CASES:
    rng = np.random.default_rng(1)
    x = G.bf16_round_np(rng.normal(0, 1, (B, H, W, cin)))
    w = G.bf16_round_np(rng.normal(0, 1.0 / np.sqrt(cin * k * k), (cout, cin, k, k)))
    b = rng.normal(0, 0.5, cout).astype(np.float32)
    try:
        got = G.conv2d(torch.from_numpy(x).to(G.DEV).to(torch.bfloat16), w, b, k, 1, 0).float().cpu().numpy()
    except Exception as e:  # noqa: BLE001
        print("%-8s FAILED: %s" % (name, e))
        break
    want = F.conv2d(torch.from_numpy(x).permute(0, 3, 1, 2), torch.from_numpy(w), torch.from_numpy(b),
                    padding=k // 2).permute(0, 2, 3, 1).numpy()
    err = np.abs(got - want)
    print("%-8s max err %.4f  frac>0.05: %.4f" % (name, err.max(), (err > 0.05).mean()))
