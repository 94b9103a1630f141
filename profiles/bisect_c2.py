"""Bisect helper: the shipping pipeline on the C2 clip against the reference golden under one configuration per process.

    python profiles/bisect_c2.py <tag> [umma=0|1] [wif=N] [calls=K] [attn=mma]

Prints per-call wall time and the PSNR of the composited video inside the holes vs the sample of them that
tests/golden/c2_80x240x432_ellipse_it20.npz holds."""
import os
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle import ops_ref  # noqa: E402
from propainter_b200 import config, ops, synth  # noqa: E402
from propainter_b200.inference_propainter import InferenceConfig, ProPainterPipeline  # noqa: E402

tag = sys.argv[1]
opts = dict(a.split("=") for a in sys.argv[2:])
config.UMMA_CONV = bool(int(opts.get("umma", "1")))
if opts.get("attn") == "mma":
    _orig = ops.sparse_window_attn
    ops.sparse_window_attn = lambda *a, **k: _orig(*a, **{**k, "impl": "mma"})
g = np.load(os.path.join(ROOT, "tests", "golden", "c2_80x240x432_ellipse_it20.npz"))
u8, fm, md = synth.make_clip(80, 240, 432, mask="ellipse", seed=0)
hole = md[0, :, 0].numpy() > 0
ref = g["comp_holes"]
pipe = ProPainterPipeline(device="cuda")
cfg = InferenceConfig()
if "wif" in opts:
    cfg.windows_in_flight = int(opts["wif"])
for call in range(int(opts.get("calls", "3"))):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    comp = pipe(torch.from_numpy(u8), fm, md, cfg)
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    a = comp.cpu().numpy()[hole][::int(g["hole_step"])]
    print(f"[{tag}] call {call}: {dt * 1e3:8.1f} ms  PSNR in the holes {ops_ref.psnr_u8(a, ref):6.2f} dB  "
          f"max|d| {np.abs(a.astype(int) - ref.astype(int)).max()}", flush=True)
