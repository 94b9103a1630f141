"""Generates tests/golden/*.npz by running the UNMODIFIED reference modules, imported read-only from a checkout of
sczhou/ProPainter.  The tests only read the committed fixtures; this script is how they were made.

    PYTHONDONTWRITEBYTECODE=1 python tests/golden/make_golden.py --reference <ProPainter checkout> [--cases ...]

Weights: the seeded synthetic state_dicts of the product's ParamNets (seeds 1/2/3), loaded into the
reference modules with strict=True -- which also proves the state_dict schema is identical.
The driver loop below re-types inference_propainter.py:298-452 around the reference's own modules
(the script itself is not importable: logic under __main__, needs imageio).
"""
import argparse
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

from propainter_b200 import schemas, synth  # noqa: E402
from propainter_b200._params import ParamNet  # noqa: E402


def build_reference(ref_dir):
    sys.path.insert(1, ref_dir)
    from RAFT import RAFT as RefRAFT
    from model.propainter import InpaintGenerator as RefGen
    from model.recurrent_flow_completion import RecurrentFlowCompleteNet as RefRFC
    sds = {"raft": ParamNet(schemas.raft_schema(), seed=1).state_dict(),
           "rfc": ParamNet(schemas.rfc_schema(), seed=2).state_dict(),
           "gen": ParamNet(schemas.generator_schema(), seed=3).state_dict()}
    raft = RefRAFT(argparse.Namespace(small=False, mixed_precision=False, alternate_corr=False)).eval()
    raft.load_state_dict(sds["raft"], strict=True)
    rfc = RefRFC(None).eval()
    rfc.load_state_dict(sds["rfc"], strict=True)
    gen = RefGen(model_path=None).eval()
    gen.load_state_dict(sds["gen"], strict=True)
    return raft, rfc, gen


def raft_bi(raft, frames, iters):
    """model/modules/flow_comp_raft.py:39-55 around the reference RAFT (RAFT_bi itself needs a checkpoint file)."""
    b, l, c, h, w = frames.shape
    a, bb = frames[:, :-1].reshape(-1, c, h, w), frames[:, 1:].reshape(-1, c, h, w)
    _, fw = raft(a, bb, iters=iters, test_mode=True)
    _, bw = raft(bb, a, iters=iters, test_mode=True)
    return fw.view(b, l - 1, 2, h, w), bw.view(b, l - 1, 2, h, w)


def get_ref_index(mid, nb, length, ref_stride=10, ref_num=-1):     # inference_propainter.py:159-173 verbatim semantics
    ref_index = []
    if ref_num == -1:
        for i in range(0, length, ref_stride):
            if i not in nb:
                ref_index.append(i)
    else:
        s = max(0, mid - ref_stride * (ref_num // 2))
        e = min(length, mid + ref_stride * (ref_num // 2))
        for i in range(s, e, ref_stride):
            if i not in nb:
                if len(ref_index) > ref_num:
                    break
                ref_index.append(i)
    return ref_index


@torch.no_grad()
def reference_pipeline(nets, u8, flow_masks, masks_dilated, raft_iter=20, neighbor_length=10, ref_stride=10, subvideo_length=80):
    raft, rfc, gen = nets
    T, H, W = u8.shape[:3]
    frames = (torch.from_numpy(u8).permute(0, 3, 1, 2).contiguous().float().div(255) * 2 - 1).unsqueeze(0)
    clip = 12 if W <= 640 else 8 if W <= 720 else 4 if W <= 1280 else 2
    if T > clip:
        ff, bb = [], []
        for f in range(0, T, clip):
            e = min(T, f + clip)
            a, b = raft_bi(raft, frames[:, f:e] if f == 0 else frames[:, f - 1:e], raft_iter)
            ff.append(a), bb.append(b)
        gt = (torch.cat(ff, 1), torch.cat(bb, 1))
    else:
        gt = raft_bi(raft, frames, raft_iter)
    L = gt[0].size(1)
    if L > subvideo_length:
        pf, pb, pad = [], [], 5
        for f in range(0, L, subvideo_length):
            s, e = max(0, f - pad), min(L, f + subvideo_length + pad)
            ps, pe = max(0, f) - s, e - min(L, f + subvideo_length)
            sub, _ = rfc.forward_bidirect_flow((gt[0][:, s:e], gt[1][:, s:e]), flow_masks[:, s:e + 1])
            sub = rfc.combine_flow((gt[0][:, s:e], gt[1][:, s:e]), sub, flow_masks[:, s:e + 1])
            pf.append(sub[0][:, ps:e - s - pe]), pb.append(sub[1][:, ps:e - s - pe])
        pred = (torch.cat(pf, 1), torch.cat(pb, 1))
    else:
        pred, _ = rfc.forward_bidirect_flow(gt, flow_masks)
        pred = rfc.combine_flow(gt, pred, flow_masks)
    masked = frames * (1 - masks_dilated)
    sub_ip = min(100, subvideo_length)
    if T > sub_ip:
        uf, um, pad = [], [], 10
        for f in range(0, T, sub_ip):
            s, e = max(0, f - pad), min(T, f + sub_ip + pad)
            ps, pe = max(0, f) - s, e - min(T, f + sub_ip)
            b, t = 1, e - s
            prop, ul = gen.img_propagation(masked[:, s:e], (pred[0][:, s:e - 1], pred[1][:, s:e - 1]), masks_dilated[:, s:e], "nearest")
            upd = frames[:, s:e] * (1 - masks_dilated[:, s:e]) + prop.view(b, t, 3, H, W) * masks_dilated[:, s:e]
            uf.append(upd[:, ps:e - s - pe]), um.append(ul.view(b, t, 1, H, W)[:, ps:e - s - pe])
        upd_f, upd_m = torch.cat(uf, 1), torch.cat(um, 1)
    else:
        prop, ul = gen.img_propagation(masked, pred, masks_dilated, "nearest")
        upd_f = frames * (1 - masks_dilated) + prop.view(1, T, 3, H, W) * masks_dilated
        upd_m = ul.view(1, T, 1, H, W)
    comp = [None] * T
    ns = neighbor_length // 2
    ref_num = subvideo_length // ref_stride if T > subvideo_length else -1
    first_window = None
    for f in range(0, T, ns):
        nb = [i for i in range(max(0, f - ns), min(T, f + ns + 1))]
        refs = get_ref_index(f, nb, T, ref_stride, ref_num)
        ids = nb + refs
        p = gen(upd_f[:, ids], (pred[0][:, nb[:-1]], pred[1][:, nb[:-1]]), masks_dilated[:, ids], upd_m[:, ids], len(nb))
        if first_window is None:
            first_window = p.clone()
        p = p.view(-1, 3, H, W)
        p = ((p + 1) / 2).cpu().permute(0, 2, 3, 1).numpy() * 255
        bm = masks_dilated[0, nb].cpu().permute(0, 2, 3, 1).numpy().astype(np.uint8)
        for i in range(len(nb)):
            idx = nb[i]
            img = np.array(p[i]).astype(np.uint8) * bm[i] + u8[idx] * (1 - bm[i])
            comp[idx] = img if comp[idx] is None else comp[idx].astype(np.float32) * 0.5 + img.astype(np.float32) * 0.5
            comp[idx] = comp[idx].astype(np.uint8)
    return np.stack(comp, 0), dict(gt_f=gt[0], gt_b=gt[1], pred_f=pred[0], pred_b=pred[1], upd_f=upd_f, upd_m=upd_m, win0=first_window)


def summarize(name, comp, st, out_dir, u8, md=None, stride=4, frame_step=1, hole_step=1):
    """stride / frame_step: spatial / temporal subsampling of the stage tensors.  With `md` (the dilated masks) only the
    pixels of the composited video inside the holes are stored, every `hole_step`-th of them in np.nonzero order
    (`comp_holes`): outside them the video equals the input clip, which the test regenerates from the seed.  The steps
    keep every fixture under 1 MB."""
    sub = lambda z: z[:, ::frame_step, :, ::stride, ::stride].contiguous().numpy()
    if md is not None:
        sel = md[0, :, 0].numpy() > 0
        assert np.array_equal(comp[~sel], u8[~sel])
        extra = dict(comp_holes=comp[sel][::hole_step], stride=np.array(stride), frame_step=np.array(frame_step),
                     hole_step=np.array(hole_step))
    else:
        extra = dict(comp=comp)
    np.savez_compressed(
        os.path.join(out_dir, name + ".npz"), **extra,
        gt_f=sub(st["gt_f"]), gt_b=sub(st["gt_b"]), pred_f=sub(st["pred_f"]), pred_b=sub(st["pred_b"]),
        upd_f=sub(st["upd_f"]), upd_m=np.packbits(st["upd_m"].numpy().astype(np.uint8)), win0=sub(st["win0"]),
        sums=np.array([st[k].double().abs().sum().item() for k in ("gt_f", "gt_b", "pred_f", "pred_b", "upd_f", "win0")]))


CASES = {
    # BASELINE.json configs[0]: 8-frame 128x128 clip + square mask (reduced RAFT iterations keep it CPU-cheap)
    "c1_8x128x128_square_it6": dict(T=8, H=128, W=128, mask="square", raft_iter=6, sub=80),
    # T > subvideo_length: halo chunking of stages 2/3 and bounded ref selection
    "chunk_23x128x128_ellipse_it2_sub10": dict(T=23, H=128, W=128, mask="ellipse", raft_iter=2, sub=10, holes=True),
    # BASELINE.json configs[1] = the benchmarked workload, full size (~10 min of CPU each; `--cases` selects)
    "c2_80x240x432_ellipse_it20": dict(T=80, H=240, W=432, mask="ellipse", raft_iter=20, sub=80, stride=16, frame_step=2,
                                       holes=True, hole_step=8),
    # configs[2] clip: 25 % border mask (video completion); the reference's CPU path is fp32 (inference_propainter.py:221-222)
    "c3_80x240x432_border_it20": dict(T=80, H=240, W=432, mask="border", raft_iter=20, sub=80, stride=16, frame_step=2,
                                      holes=True, hole_step=24),
}
DEFAULT_CASES = ["c1_8x128x128_square_it6", "chunk_23x128x128_ellipse_it2_sub10"]

if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--reference", required=True, help="checkout of sczhou/ProPainter whose modules produce the fixtures")
    ap.add_argument("--cases", nargs="*", default=DEFAULT_CASES, choices=list(CASES))
    ap.add_argument("--threads", type=int, default=0)
    a = ap.parse_args()
    if a.threads:
        torch.set_num_threads(a.threads)
    nets = build_reference(a.reference)
    out_dir = os.path.dirname(os.path.abspath(__file__))
    for name in a.cases:
        c = CASES[name]
        u8, fm, md = synth.make_clip(c["T"], c["H"], c["W"], mask=c["mask"], seed=0)
        comp, st = reference_pipeline(nets, u8, fm, md, raft_iter=c["raft_iter"], subvideo_length=c["sub"])
        summarize(name, comp, st, out_dir, u8, md=md if c.get("holes") else None, stride=c.get("stride", 4),
                  frame_step=c.get("frame_step", 1), hole_step=c.get("hole_step", 1))
        print(name, "done", comp.shape, os.path.getsize(os.path.join(out_dir, name + ".npz")) // 1024, "KiB")
