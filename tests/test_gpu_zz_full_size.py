"""Full-size tests of the shipping pipeline at the benchmarked configuration (BASELINE.json configs[1] = C2, and the
80-frame border-mask clip of configs[2] = C3); collected after the op / module parity files.

  * vs the REFERENCE: tests/golden/c{2,3}_80x240x432_*.npz hold the outputs of the unmodified reference modules for exactly
    these clips (tests/golden/make_golden.py, ~10 min of CPU each): RAFT flows, completed flows and propagated frames
    (every 2nd frame, every 16th row and column), the propagated masks, and a sample of the composited uint8 video
    inside the holes (outside them the video is the input, which is checked bit-exactly).  The shipping defaults (TF32
    tensor-core products, CUDA graphs, autotuned plans) are compared stage by stage; bars are ~10x the error measured on
    B200 (printed by the test).
  * the oracle itself is pinned at full size by running it on the GPU in strict fp32 against the same golden.
  * size-independent properties (zero mask = identity, replay determinism, the hole never grows)."""
import os

import numpy as np
import pytest
import torch

from oracle import pipeline_ref

pytestmark = pytest.mark.gpu
DEV = "cuda"
GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
GOLD80 = {"c2": ("c2_80x240x432_ellipse_it20", "ellipse"), "c3": ("c3_80x240x432_border_it20", "border")}


def _load80(key):
    from propainter_b200 import synth
    name, mask = GOLD80[key]
    g = np.load(os.path.join(GOLD, name + ".npz"))
    u8, fm, md = synth.make_clip(80, 240, 432, mask=mask, seed=0)
    hole = md[0, :, 0].numpy() > 0
    return g, u8, fm, md, hole


def _video_errors(g, a, u8, hole):
    """PSNR of the whole video and of the holes alone against the reference's composited video, and the differences at
    the sampled hole pixels.  The fixture holds every hole_step-th hole pixel (np.nonzero order); outside the holes the
    reference video is the input clip, so the error there is exact and only the holes' mean squared error is sampled."""
    d_h = a[hole][::int(g["hole_step"])].astype(np.float64) - g["comp_holes"]
    d_o = a[~hole].astype(np.float64) - u8[~hole]
    mse = (np.mean(d_h ** 2) * a[hole].size + np.sum(d_o ** 2)) / a.size
    psnr = 20.0 * np.log10(255.0 / np.sqrt(mse)) if mse else float("inf")
    psnr_hole = 20.0 * np.log10(255.0 / np.sqrt(np.mean(d_h ** 2))) if d_h.any() else float("inf")
    return psnr, psnr_hole, np.abs(d_h), np.abs(d_o).max(initial=0)


def _stage_errors(g, st):
    s, f = int(g["stride"]), int(g["frame_step"])
    sub = lambda z: z[:, ::f, :, ::s, ::s].float().cpu().numpy()
    out = {}
    for key, val in (("gt_f", st["gt_flows"][0]), ("gt_b", st["gt_flows"][1]), ("pred_f", st["pred_flows"][0]),
                     ("pred_b", st["pred_flows"][1])):
        ref = g[key]
        out[key] = float(np.abs(sub(val) - ref).max() / max(np.abs(ref).max(), 1e-12))
    um = np.unpackbits(g["upd_m"])[:st["updated_masks"].numel()].reshape(st["updated_masks"].shape)
    out["upd_m_mismatch"] = float((um != (st["updated_masks"].cpu().numpy() > 0.5)).mean())
    out["upd_f_mismatch"] = float((np.abs(sub(st["updated_frames"]) - g["upd_f"]) > 1e-4).mean())
    return out


@pytest.mark.shipping
@pytest.mark.parametrize("key", ["c2", "c3"])
def test_full_size_vs_reference_golden(key):
    """The benchmarked pipeline (shipping defaults, 80 x 240 x 432, raft_iter 20) against the reference modules' outputs."""
    from propainter_b200.inference_propainter import InferenceConfig, ProPainterPipeline
    g, u8, fm, md, hole = _load80(key)
    pipe = ProPainterPipeline(device=DEV)
    comp, st = pipe(torch.from_numpy(u8), fm, md, InferenceConfig(), return_stages=True)
    a = comp.cpu().numpy()
    e = _stage_errors(g, st)
    psnr, psnr_hole, d, _ = _video_errors(g, a, u8, hole)
    print(f"{key}: " + " ".join(f"{k}={v:.2e}" for k, v in e.items()) +
          f" | PSNR {psnr:.2f} dB (holes only {psnr_hole:.2f} dB), max |diff| {d.max()}, >1 level in the holes: "
          f"{(d > 1).mean():.2e}")
    assert np.array_equal(a[~hole], u8[~hole])
    # measured on B200 (round 2): flows 1.4e-3 / 1.5e-3 (TF32 library convs in RAFT), masks and propagated frames exact,
    # PSNR 72.1 dB (C2) / 67.2 dB (C3), 61.1 dB inside the holes, max |diff| 1 level
    assert e["gt_f"] < 1e-2 and e["gt_b"] < 1e-2 and e["pred_f"] < 1e-2 and e["pred_b"] < 1e-2
    assert e["upd_m_mismatch"] < 1e-3 and e["upd_f_mismatch"] < 1e-3
    assert psnr_hole > 52.0 and psnr > 60.0 and d.max() <= 4


def test_oracle_pinned_at_full_size():
    """The oracle (run on the GPU in strict fp32: no TF32 anywhere) reproduces the reference's C2 golden: the CPU suite can
    only afford this check at 8-23 frames (tests/test_oracle_golden.py)."""
    g, u8, fm, md, hole = _load80("c2")
    from propainter_b200 import schemas
    from propainter_b200._params import ParamNet
    sds = {k: {n: v.to(DEV) for n, v in ParamNet(sch, seed=sd).state_dict().items()}
           for k, sch, sd in (("raft", schemas.raft_schema(), 1), ("rfc", schemas.rfc_schema(), 2), ("gen", schemas.generator_schema(), 3))}
    a, b = torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32
    torch.backends.cudnn.allow_tf32 = torch.backends.cuda.matmul.allow_tf32 = False
    try:
        comp, st = pipeline_ref.run_pipeline(sds, u8, fm.to(DEV), md.to(DEV), raft_iter=20, return_stages=True)
    finally:
        torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = a, b
    e = _stage_errors(g, st)
    psnr, _, d, d_out = _video_errors(g, comp, u8, hole)
    print("oracle@gpu fp32 vs golden: " + " ".join(f"{k}={v:.2e}" for k, v in e.items()) +
          f" | max |diff| {max(d.max(), d_out)}, changed in the holes {(d > 0).mean():.2e}")
    assert max(e["gt_f"], e["gt_b"]) < 1e-3 and max(e["pred_f"], e["pred_b"]) < 1e-3 and e["upd_m_mismatch"] < 1e-4
    assert psnr > 60.0


def test_full_size_properties():
    """BASELINE.json configs[1] at full size (80 x 240 x 432, shipping defaults) through properties that need no
    oracle run: (i) outside the dilated mask the composite is the input, bit-exact (inference_propainter.py:437-444);
    (ii) an all-zero mask returns the input video and leaves the RAFT flows untouched by completion (combine_flow,
    recurrent_flow_completion.py:340-347); (iii) replaying the captured graphs is bit-deterministic; (iv) the filled
    region changes when the mask moves (the fill is actually computed); (v) image propagation never grows the hole and
    only touches masked pixels (propainter.py:155-161)."""
    from propainter_b200 import synth
    from propainter_b200.inference_propainter import InferenceConfig, ProPainterPipeline
    T, H, W = 80, 240, 432
    u8, fm, md = synth.make_clip(T, H, W, mask="ellipse", seed=0)
    pipe = ProPainterPipeline(device=DEV)
    cfg = InferenceConfig()
    x = torch.from_numpy(u8)
    comp, st = pipe(x, fm, md, cfg, return_stages=True)
    a = comp.cpu().numpy()
    hole = md[0, :, 0].bool().numpy()
    assert a.shape == u8.shape and a.dtype == np.uint8
    assert np.array_equal(a[~hole], u8[~hole])                                           # (i)
    assert (a[hole] != u8[hole]).mean() > 0.5                                            # (iv) the hole was re-synthesised
    assert np.array_equal(pipe(x, fm, md, cfg).cpu().numpy(), a)                         # (iii)
    um = st["updated_masks"][0, :, 0].cpu().numpy() > 0.5
    assert not (um & ~hole).any() and um.sum() <= hole.sum()                             # (v) the hole never grows
    frames = pipeline_ref.to_float_frames(u8)[0]
    uf = st["updated_frames"][0].cpu()
    keep = ~torch.from_numpy(hole)[:, None].expand(-1, 3, -1, -1)
    assert torch.equal(uf[keep], frames[keep])
    zero = torch.zeros_like(md)
    comp0, st0 = pipe(x, zero, zero, cfg, return_stages=True)
    assert np.array_equal(comp0.cpu().numpy(), u8)                                       # (ii)
    for k in (0, 1):                                                                     # 0*pred + 1*flow == flow wherever pred is finite
        fin = torch.isfinite(st0["pred_flows"][k])
        assert torch.equal(st0["pred_flows"][k][fin], st0["gt_flows"][k][fin])
