"""ORACLE (test infrastructure): deterministic synthetic weight sets for the FuseTrack oracle
(SURVEY.md 8d).  There are no trained checkpoints offline; these exercise every code path.

  "A": the reference's init rules (kaiming / xavier / normal as cited in SURVEY A.13).  bn3.gamma = 0
       and score_thresh 0.6 mean residual branches vanish and nothing is detected -> plumbing only.
  "B": dense-random: every conv/linear kaiming-uniform-ish, BN gamma~U(.5,1.5), beta~N(0,.1), running
       stats random, non-zero DCN offsets, FlowNet2 xavier with small biases.
  "C": B + detection forcing: bbox_head.fc_cls scaled up / fc_reg scaled down so that >= a few dozen
       RoIs pass the 0.6 threshold and the mask / tracking / fusion stages see real instances.
"""
import torch

from vps_b200.synth import init_weights  # noqa: F401  (shared, model-agnostic parameter initialiser)


@torch.no_grad()
def calibrate(model, size=(128, 256), seed=123, scales=None):
    """Data-dependent rescaling (LSUV-style) so the synthetic network is numerically non-degenerate:
    O(1) pyramid features, sub-pixel..pixel flows, un-saturated class scores, O(1) mask logits and
    tracker scores.  Deterministic (fixed seed, CPU fp32).  Only linear output layers are rescaled.
    Returns the factors applied, in order.  The measured factors differ in their last bits between hosts (thread count,
    CPU kernels); `scales`, such a list from an earlier run, is applied instead of them: that run's weights, bit for bit."""
    import torch.nn.functional as F
    from . import model as M
    g = torch.Generator().manual_seed(seed)
    H, W = size
    img = torch.randn(1, 3, H, W, generator=g)
    ref = torch.roll(img, shifts=(1, 2), dims=(2, 3)) + 0.05 * torch.randn(1, 3, H, W, generator=g)

    applied = []

    def scale_(mod, s):
        if scales is not None:
            s = float(scales[len(applied)])
        applied.append(s)
        mod.weight.mul_(s)
        if getattr(mod, "bias", None) is not None:
            mod.bias.mul_(s)

    # FlowNet2: final flow ~ 1.5 px RMS
    taps = {}
    model.compute_flow(img.clone(), ref.clone(), 0.25, taps)
    rms = taps["flow_full"].pow(2).mean().sqrt().item()
    scale_(model.flownet2.flownetfusion.predict_flow0, 1.5 / max(rms, 1e-6))
    # pyramid features ~ unit RMS at every level
    c = model.backbone(img)
    for i, l in enumerate(model.neck.lateral_convs):
        rms = l(c[i]).pow(2).mean().sqrt().item()
        scale_(l.conv, 1.0 / max(rms, 1e-6))
    for _ in range(2):
        p = model.neck(c)
        for i in range(4):
            rms = p[i].pow(2).mean().sqrt().item()
            scale_(model.neck.fpn_convs[i].conv, 1.0 / max(rms, 1e-6))
    x = model.neck(c)
    rx = model.neck(model.backbone(ref))
    flow = torch.zeros(1, 2, H // 4, W // 4)
    en = model.extra_neck
    bsf, rbsf = en.gather(x), en.gather(rx)
    ff = en.liteflownet(bsf, M.O.flow_warp(rbsf, flow), flow)
    scale_(en.liteflownet.flow_estimator.convs[3], 0.7 / max(ff.pow(2).mean().sqrt().item(), 1e-6))
    taps = {}
    en(x, rx, flow, taps)
    scale_(en.tcea_fusion.tAtt_1, 0.25 / max(en.tcea_fusion.tAtt_1(bsf).pow(2).mean().sqrt().item(), 1e-6))
    scale_(en.tcea_fusion.tAtt_2, 0.25 / max(en.tcea_fusion.tAtt_2(bsf).pow(2).mean().sqrt().item(), 1e-6))
    taps = {}
    en(x, rx, flow, taps)
    scale_(en.tcea_fusion.sAtt_4, 1.0 / max(taps["fused"].pow(2).mean().sqrt().item(), 1e-6) ** 0.5)
    taps = {}
    en(x, rx, flow, taps)
    scale_(en.refine.conv, 0.7 / max(taps["refined"].pow(2).mean().sqrt().item(), 1e-6))
    xf = en(x, rx, flow)
    # semantic logits ~ 2 RMS
    _, fs = model.panopticFPN(xf[:4])
    scale_(model.panopticFPN.conv_pred.conv, 2.0 / max(fs.pow(2).mean().sqrt().item(), 1e-6))
    # RPN: logits ~1.5, deltas ~0.3
    cls, reg = model.rpn_head(xf)
    scale_(model.rpn_head.rpn_cls, 1.5 / max(cls[0].pow(2).mean().sqrt().item(), 1e-6))
    scale_(model.rpn_head.rpn_reg, 0.3 / max(reg[0].pow(2).mean().sqrt().item(), 1e-6))
    cls, reg = model.rpn_head(xf)
    props = model.rpn_head.get_bboxes(cls, reg, (H, W, 3), M.TEST_CFG_RPN)
    rois = torch.cat([props.new_zeros(props.size(0), 1), props[:, :4]], dim=-1)
    rf = M.roi_extract(xf[:4], rois, 7)
    bh = model.bbox_head
    h0 = F.relu(bh.shared_fcs[0](rf.view(rf.size(0), -1)))
    scale_(bh.shared_fcs[0], 1.0 / max(h0.pow(2).mean().sqrt().item(), 1e-6))
    h1 = F.relu(bh.shared_fcs[1](F.relu(bh.shared_fcs[0](rf.view(rf.size(0), -1)))))
    scale_(bh.shared_fcs[1], 1.0 / max(h1.pow(2).mean().sqrt().item(), 1e-6))
    cs, bp = bh(rf)
    scale_(bh.fc_cls, 4.0 / max(cs.pow(2).mean().sqrt().item(), 1e-6))
    scale_(bh.fc_reg, 0.5 / max(bp.pow(2).mean().sqrt().item(), 1e-6))
    th = model.track_head
    e0 = F.relu(th.fcs[0](rf.view(rf.size(0), -1)))
    scale_(th.fcs[0], 1.0 / max(e0.pow(2).mean().sqrt().item(), 1e-6))
    e1 = th.embed(rf)
    scale_(th.fcs[1], (3.0 / max((e1 @ e1.t()).pow(2).mean().sqrt().item(), 1e-6)) ** 0.5)
    mf = M.roi_extract(xf[:4], rois[:32], 14)
    ms = model.mask_head(mf)
    scale_(model.mask_head.conv_logits, 2.0 / max(ms.pow(2).mean().sqrt().item(), 1e-6))
    assert scales is None or len(scales) == len(applied)
    return applied


def make_model(kind="C", seed=0, calibrated=True, cache_dir="/tmp/vps_oracle_weights", scales=None):
    """Oracle model with synthetic weights; the calibrated state_dict is cached on disk.  `scales`: calibrate() replays
    these factors (no cache)."""
    import os
    from .model import PanopticFuseTrack
    m = PanopticFuseTrack()
    if scales is not None:
        init_weights(m, kind, seed)
        calibrate(m, scales=scales)
        return m
    path = os.path.join(cache_dir, "w_%s_%d_%d.pt" % (kind, seed, int(calibrated)))
    if os.path.exists(path):
        m.load_state_dict(torch.load(path))
        return m
    init_weights(m, kind, seed)
    if calibrated and kind != "A":
        calibrate(m)
    try:
        os.makedirs(cache_dir, exist_ok=True)
        torch.save(m.state_dict(), path)
    except OSError:
        pass
    return m
