"""TEST HARNESS ONLY.  CPU stand-ins for ``propainter_b200.ops`` (built from tests/hostsim and plain torch)
that the CPU test-suite monkeypatches in, so the *host-side plumbing* of the drop-in modules -- weight
packing, channel orders of the concat buffers, scan bookkeeping, stage scheduling -- is checked against
the oracle without a GPU.  The product never imports this file and has no CPU path; the GPU tests run
the real kernels.
"""
import ctypes
import math

import torch
import torch.nn.functional as F

FP = ctypes.POINTER(ctypes.c_float)


def _fp(t):
    assert t.dtype == torch.float32 and t.is_contiguous() and not t.is_cuda
    return ctypes.cast(t.data_ptr(), FP)


def install(monkeypatch, hostsim):
    from propainter_b200 import ops

    def corr_build(fmap, idx1, idx2, levels, h, w):
        from oracle import ops_ref
        F_, N, D = fmap.shape
        fm = fmap.view(F_, h, w, D).permute(0, 3, 1, 2)
        pyr = ops_ref.corr_pyramid(fm[idx1.long()], fm[idx2.long()])
        wl = w
        for lv, p in zip(levels, pyr):
            lv[:, :, :wl] = p[:, 0]
            wl //= 2

    def corr_lookup(levels, coords, out=None):
        B, h, w, _ = coords.shape
        if out is None:
            out = torch.empty(B, h, w, 324)
        c = coords.contiguous()
        hostsim.hs_corr_lookup(_fp(levels[0]), _fp(levels[1]), _fp(levels[2]), _fp(levels[3]), _fp(c), _fp(out),
                               ctypes.c_long(B * h * w), h, w)
        return out

    def convex_upsample(mask_pm, flow_lr, mask_scale=0.25):
        n, h, w, _ = flow_lr.shape
        m, fl = mask_pm.contiguous(), flow_lr.contiguous()
        out = torch.empty(n, 2, 8 * h, 8 * w)
        hostsim.hs_convex_upsample(_fp(m), m.shape[-1], ctypes.c_float(mask_scale), _fp(fl), _fp(out), n, h, w)
        return out

    def img_prop_scan(frames, flows_f, flows_b, masks, nearest=True):
        t, _, H, W = frames.shape
        of, om = torch.empty_like(frames), torch.empty_like(masks)
        a, b, c, d = frames.contiguous(), flows_f.contiguous(), flows_b.contiguous(), masks.contiguous()
        hostsim.hs_img_prop_scan(_fp(a), _fp(b), _fp(c), _fp(d), _fp(of), _fp(om), t, H, W, int(bool(nearest)))
        return of, om

    def prop_cond(cur, prop, fprop, fcheck, mcur, cond, bb, first):
        h, w, C = cur.shape
        assert cur.stride(-1) == 1 and bb.stride(-1) == 1
        args = [_fp_view(cur), cur.stride(-2), _fp_view(prop) if prop is not None else None,
                prop.stride(-2) if prop is not None else C, _fp(fprop) if fprop is not None else None,
                _fp(fcheck) if fcheck is not None else None, _fp(mcur.contiguous()),
                _fp_view(cond) if cond is not None else None, cond.stride(-2) if cond is not None else 2 * C + 8,
                _fp_view(bb), bb.stride(-2), h, w, C, int(bool(first))]
        hostsim.hs_prop_cond(*args)

    def _fp_view(t):
        assert t.dtype == torch.float32 and t.stride(-1) == 1
        return ctypes.cast(t.data_ptr(), FP)

    def deform_align(x, o, flow, max_res, w_packed, bias, out, o_bias=None):
        if x.dim() == 4:                                  # batched entry: independent maps
            for i in range(x.shape[0]):
                deform_align(x[i], o[i], None if flow is None else flow[i], max_res, w_packed, bias, out[i], o_bias)
            return out
        H, W, Cin = x.shape
        if o_bias is not None:
            o = (o + o_bias).contiguous()
        cols = torch.empty(H * W, 9 * Cin)
        hostsim.hs_deform_cols(_fp_view(x), x.stride(-2), _fp_view(o), o.stride(-2), _fp(flow) if flow is not None else None,
                               ctypes.c_float(max_res), _fp(cols), H, W, Cin)
        out.copy_((cols @ w_packed + bias).view(H, W, -1))
        return out

    def gen_prep(flows_f, flows_b, masks_in, masks_upd, lt):
        ds = lambda z: (F.interpolate(z, scale_factor=0.25, mode="bilinear", align_corners=False) / 4.0).permute(0, 2, 3, 1).contiguous()
        nn_ = lambda z: F.interpolate(z[:lt], scale_factor=0.25, mode="nearest")[:, 0]
        pmask = torch.stack([nn_(masks_in), nn_(masks_upd)], -1).contiguous()
        if lt > 1:
            return ds(flows_f), ds(flows_b), pmask
        e = torch.zeros(0, pmask.shape[1], pmask.shape[2], 2)
        return e, e, pmask

    def window_mask(pmask, fh, fw, nwh, nww):
        lt = pmask.shape[0]
        mp = F.max_pool2d(pmask[..., 0][:, None], (7, 7), (3, 3), (3, 3))
        mp = F.pad(mp, (0, nww * 9 - fw, 0, nwh * 5 - fh))
        return (F.max_pool2d(mp, (5, 9), (5, 9)).view(lt, -1).sum(0) > 0).int()

    def sparse_window_attn(qkv, pool_kv, key_tok, flags, t, NT, kf_start, kf_step, out=None, WN=45, C=512):
        heads, ch = C // 128, 128
        out = torch.zeros(t, NT, C)
        q, k, v = qkv[..., :C], qkv[..., C:2 * C], qkv[..., 2 * C:]
        kf = list(range(kf_start, t, kf_step))
        scale = 1.0 / math.sqrt(ch)
        for wi in range(key_tok.shape[0]):
            own = key_tok[wi, :WN].long()
            for hd in range(heads):
                sl = slice(hd * ch, (hd + 1) * ch)
                if flags[wi] != 0:
                    allk = key_tok[wi].long()
                    K = torch.cat([torch.cat([k[f][allk][:, sl], pool_kv[f][:, :C][:, sl]], 0) for f in kf], 0)
                    V = torch.cat([torch.cat([v[f][allk][:, sl], pool_kv[f][:, C:][:, sl]], 0) for f in kf], 0)
                    for f in range(t):
                        a = torch.softmax((q[f][own][:, sl] @ K.t()) * scale, -1)
                        out[f, own, sl] = a @ V
                else:
                    for f in range(t):
                        a = torch.softmax((q[f][own][:, sl] @ k[f][own][:, sl].t()) * scale, -1)
                        out[f, own, sl] = a @ v[f][own][:, sl]
        return out

    def ffn_overlap_add(Y, frames, h, w, CH=40):
        Y = Y.contiguous()
        Z = torch.empty_like(Y)
        hostsim.hs_ffn_overlap_add(_fp(Y), Y.shape[-1], _fp(Z), Z.shape[-1], frames, h, w, CH)
        return Z

    def u8_to_frames(u8):
        T, H, W, _ = u8.shape
        u8 = u8.contiguous()
        out = torch.empty(T, 3, H, W)
        hostsim.hs_u8_to_frames(ctypes.c_void_p(u8.data_ptr()), _fp(out), T, H, W)
        return out

    def composite_blend(pred, masks, ori_u8, comp_u8, frame_ids, first_flags):
        n, _, H, W = pred.shape
        fr = (ctypes.c_int * n)(*[int(i) for i in frame_ids])
        fs = (ctypes.c_int * n)(*[int(bool(i)) for i in first_flags])
        p, m = pred.contiguous(), masks.contiguous()
        hostsim.hs_composite(_fp(p), _fp(m), ctypes.c_void_p(ori_u8.data_ptr()), ctypes.c_void_p(comp_u8.data_ptr()), n, fr,
                             fs, H, W)

    _act = {"none": lambda t: t, "relu": F.relu, "leaky": None, "sigmoid": torch.sigmoid, "tanh": torch.tanh}

    def bias_act(x_pm, bias=None, act="none", slope=0.0, res=None, post_relu=False, out=None, pre=None):
        t = x_pm if bias is None else x_pm + bias
        if pre is not None:
            t = t + pre
        t = F.leaky_relu(t, slope) if act == "leaky" else _act[act](t)
        if res is not None:
            t = t + res
        if post_relu:
            t = F.relu(t)
        out = x_pm if out is None else out
        out.copy_(t)
        return out

    def bias_act_(x_pm, bias, act="none", slope=0.0):
        return bias_act(x_pm, bias, act, slope)

    def pool_depthwise(x_pm, w_taps, bias, kh, kw):
        C = x_pm.shape[-1]
        w = w_taps.t().reshape(C, 1, kh, kw)
        return F.conv2d(x_pm.permute(0, 3, 1, 2), w, bias, stride=(kh, kw), groups=C).permute(0, 2, 3, 1).contiguous()

    def add_layernorm(x, delta, gamma, beta, eps=1e-5):
        xo = x if delta is None else x + delta
        return xo, F.layer_norm(xo, (x.shape[-1],), gamma, beta, eps)

    def instance_norm(x_pm, relu=False, res=None, post_relu=False, eps=1e-5, out=None):
        t = F.instance_norm(x_pm.permute(0, 3, 1, 2), eps=eps).permute(0, 2, 3, 1)
        if relu:
            t = F.relu(t)
        if res is not None:
            t = t + res
        if post_relu:
            t = F.relu(t)
        out = torch.empty_like(x_pm) if out is None else out
        out.copy_(t)
        return out

    def gru_gate(zr_pm, bias, net_view, z_out, rnet_view, pre=None):
        C = z_out.shape[-1]
        g = torch.sigmoid(zr_pm + (0 if bias is None else bias) + (0 if pre is None else pre))
        z_out.copy_(g[..., :C])
        rnet_view.copy_(g[..., C:] * net_view)

    def gru_update(q_pm, bias, z, net_view, net_copy=None, pre=None):
        net_view.copy_((1 - z) * net_view + z * torch.tanh(q_pm + (0 if bias is None else bias) + (0 if pre is None else pre)))
        if net_copy is not None:
            net_copy.copy_(net_view)

    def raft_pack_motion(mot_pm, flow_pm, d0_view, d1_view, bias=None):
        m = mot_pm if bias is None else F.relu(mot_pm + bias)
        v = torch.cat([m[..., :126], flow_pm], -1)
        d0_view.copy_(v)
        d1_view.copy_(v)

    def upsample2x(x_pm):
        n, h, w, C = x_pm.shape
        x_pm = x_pm.contiguous()
        out = torch.empty(n, 2 * h, 2 * w, C)
        hostsim.hs_upsample2x(_fp(x_pm), _fp(out), n, h, w, C)
        return out

    def tf32_round(w):
        return w                                           # plumbing is checked in exact fp32; the rounding itself is a GPU-test matter

    def conv_umma(segs, w_packed, KH, KW, Cout, bias=None, act="none", slope=0.0, pre=None, res=None, post_relu=False, out=None,
                  round_tf32=False, bn=0, tile_w=0, tile_m=0):
        """unpacks the [Cout][K] weight layout of pp_conv2d_umma (include/propainter_b200.h) back to [Cout,Cin,KH,KW]"""
        chans = [sg.shape[-1] for sg in segs]
        nblk = sum((c + 31) // 32 for c in chans)
        assert tuple(w_packed.shape) == (Cout, nblk * KH * KW * 32)
        wb = w_packed.view(Cout, nblk, KH, KW, 32)
        parts, b = [], 0
        for c in chans:
            for c0 in range(0, c, 32):
                cw = min(32, c - c0)
                assert wb[:, b, :, :, cw:].abs().max().item() == 0 if cw < 32 else True      # padded channels carry zero weights
                parts.append(wb[:, b, :, :, :cw].permute(0, 3, 1, 2))
                b += 1
        w = torch.cat(parts, 1)
        x = torch.cat(list(segs), -1).permute(0, 3, 1, 2)
        t = F.conv2d(x, w, bias, padding=(KH // 2, KW // 2)).permute(0, 2, 3, 1)
        if pre is not None:
            t = t + pre
        t = F.leaky_relu(t, slope) if act == "leaky" else _act[act](t)
        if res is not None:
            t = t + res
        if post_relu:
            t = F.relu(t)
        if out is None:
            return t.contiguous()
        out.copy_(t)
        return out

    def deform_gather(x, o, flow, max_res, cols=None, o_bias=None, x2=None):
        if x2 is not None:
            x = torch.cat([x, x2], -1)
        n, H, W, Cin = x.shape
        if o_bias is not None:
            o = o + o_bias
        if cols is None:
            cols = torch.empty(n, H, W, 9 * Cin)
        for i in range(n):
            xi, oi = x[i].contiguous(), o[i].contiguous()
            ci = torch.empty(H * W, 9 * Cin)
            hostsim.hs_deform_cols(_fp(xi), Cin, _fp(oi), oi.shape[-1], _fp(flow[i].contiguous()) if flow is not None else None,
                                   ctypes.c_float(max_res), _fp(ci), H, W, Cin)
            cols[i].copy_(ci.view(H, W, -1))
        return cols

    def flow_warp_fbcheck(feat, fprop, fcheck=None, warped=None, aux=None, want_warp=True, round_tf32=False):
        from oracle import ops_ref
        if want_warp:
            wv = ops_ref.flow_warp(feat.permute(0, 3, 1, 2), fprop, "bilinear").permute(0, 2, 3, 1)
            if warped is None:
                warped = wv.contiguous()
            else:
                warped.copy_(wv)
        if fcheck is not None:
            valid = ops_ref.fb_consistency(fprop.permute(0, 3, 1, 2), fcheck.permute(0, 3, 1, 2))
            if aux is None:
                aux = torch.zeros(*fprop.shape[:3], 4)
            aux[..., 0:2] = fprop
            aux[..., 2] = valid[:, 0]
        return warped, aux

    for name, fn in list(locals().items()):
        if callable(fn) and hasattr(ops, name) and not name.startswith("_"):
            monkeypatch.setattr(ops, name, fn)
    # plan choices are keyed by shape, not device: ones measured by GPU tests earlier in the session would replay
    # CUDA-only library plans (cuDNN's fused conv-bias-ReLU) on these CPU tensors
    from propainter_b200 import autotune
    monkeypatch.setattr(autotune, "_choice", {})
