"""Generate golden fixtures from the REAL reference (run in the build container only; needs /root/reference).

    YOLO_CONFIG_DIR=/tmp/ulcfg python tests/golden/make_golden.py

Writes (all committed, all small):
  yolo26-master-n.keys.json     reference state_dict key -> (shape, dtype)
  yolo26-master-n.bnstats.pt    BatchNorm running statistics calibrated on synthetic images (fp32)
  yolo26-master-n.golden.pt     reference outputs (fp32) for seeded inputs: per-layer activations, router decisions,
                                raw Detect head outputs and the final (B,300,6) detections
Weights are NOT stored: both sides regenerate them from state_dict key names with utils/synth.fill_state_dict_.
"""
import json
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, "/root/reference")
sys.path.insert(0, ROOT)
os.environ.setdefault("YOLO_CONFIG_DIR", "/tmp/ulcfg")

from ultralytics.nn.modules.moe.routers import EfficientSpatialRouter  # noqa: E402
from ultralytics.nn.tasks import DetectionModel  # noqa: E402

from yolo_master_b200.utils.synth import fill_state_dict_, load_norm_stats_, synth_images  # noqa: E402

OUT = os.path.dirname(os.path.abspath(__file__))
CFG = "/root/reference/ultralytics/cfg/models/26/yolo26-master-n.yaml"
NAME = "yolo26-master-n"
KEEP_LAYERS = [2, 4, 6, 8, 9, 10, 13, 16, 19, 22]


def calibrated_reference(seed=0, cfg=None):
    m = DetectionModel(cfg or CFG, verbose=False)
    sd = m.state_dict()
    fill_state_dict_(sd, seed)
    m.load_state_dict(sd)
    m.eval()
    bns = [mod for mod in m.modules() if isinstance(mod, torch.nn.BatchNorm2d)]
    for b in bns:
        b.train()
        b.momentum = None
        b.reset_running_stats()
    with torch.no_grad():
        m(synth_images(8, 320, 320, seed=7))
    for b in bns:
        b.eval()
        b.momentum = 0.03
    return m


def run(m, x):
    feats, routes = {}, {}
    hooks = [mod.register_forward_hook(lambda mod, i, o, k=k: feats.__setitem__(k, o)) for k, mod in enumerate(m.model)]
    for name, mod in m.named_modules():
        if isinstance(mod, EfficientSpatialRouter):
            hooks.append(mod.register_forward_hook(lambda mod, i, o, n=name: routes.__setitem__(n, (o[0].clone(), o[1].clone()))))
    with torch.no_grad():
        y, preds = m(x)
    for h in hooks:
        h.remove()
    return y, preds, feats, routes


def main():
    torch.manual_seed(0)
    m = calibrated_reference(0)
    sd = m.state_dict()
    json.dump({k: [list(v.shape), str(v.dtype)] for k, v in sd.items()}, open(f"{OUT}/{NAME}.keys.json", "w"))
    stats = {k: v.clone() for k, v in sd.items() if k.endswith("running_mean") or k.endswith("running_var")}
    torch.save(stats, f"{OUT}/{NAME}.bnstats.pt")

    # the fixture must be reproducible from key names + stats alone
    m2 = DetectionModel(CFG, verbose=False)
    sd2 = m2.state_dict()
    load_norm_stats_(fill_state_dict_(sd2, 0), stats)
    assert all(torch.equal(sd[k], sd2[k]) for k in sd if sd[k].is_floating_point())

    gold = {"cases": {}}
    for tag, (B, H, W, seed) in {"b2_160": (2, 160, 160, 1), "b1_64": (1, 64, 64, 2)}.items():
        x = synth_images(B, H, W, seed)
        y, preds, feats, routes = run(m, x)
        gold["cases"][tag] = {
            "B": B, "H": H, "W": W, "seed": seed,
            "final": y.clone(),
            "layers": {i: feats[i].clone() for i in KEEP_LAYERS},
            "routes": {n: (w.float(), i.int()) for n, (w, i) in routes.items()},
            "head_boxes": preds["one2one"]["boxes"].clone(),
            "head_scores": preds["one2one"]["scores"].clone(),
        }
        print(tag, "final", tuple(y.shape), "score range", float(y[..., 4].min()), float(y[..., 4].max()))
    torch.save(gold, f"{OUT}/{NAME}.golden.pt")
    for f in os.listdir(OUT):
        print(f, os.path.getsize(os.path.join(OUT, f)))


V0 = "/root/reference/ultralytics/cfg/models/master/v0/det/"
EXTRA_MODELS = {
    # name: (cfg, kept layers, {tag: (B, H, W, seed)})
    "yolo-master-n-v0": (V0 + "yolo-master-n.yaml", [3, 6, 8, 9, 11, 12, 18, 21, 24], {"b2_128": (2, 128, 128, 3), "b1_64": (1, 64, 64, 4)}),
    "yolo-master-l-v0": (V0 + "yolo-master-l.yaml", [8, 11, 12, 24], {"b1_64": (1, 64, 64, 5)}),
    # MoT + MoA neck (C2fMoT x3, C2fMoA x1), end2end head; "-s" = the same YAML with an injected s scale (SURVEY.md §8d, C3)
    "yolo26-master-moa-mot-n": ("/root/reference/ultralytics/cfg/models/26/yolo26-master-moa-mot-n.yaml", [6, 10, 13, 16, 19, 22],
                                {"b2_224": (2, 224, 224, 6), "b1_96": (1, 96, 96, 7)}),
    # gated MoE family (SURVEY.md §8f rank 1): oracle pinned ahead of the CUDA path
    "yolo-master-n-v0_10": ("/root/reference/ultralytics/cfg/models/master/v0_10/det/yolo-master-n.yaml", [5, 8, 11, 17, 20, 23],
                            {"b2_160": (2, 160, 160, 9), "b1_128": (1, 128, 128, 10)}),   # (B=1 with a 5..7-pixel P4/P5 map makes the
                            # reference itself raise: its router GroupNorm then sees one value per group, gated.py:113)
    # ModularRouterExpertMoE (= OptimizedMOEImproved) as a top-level layer that owns its residual: the v0_1 zoo
    "yolo-master-n-v0_1": ("/root/reference/ultralytics/cfg/models/master/v0_1/det/yolo-master-n.yaml", [5, 8, 11, 23],
                           {"b2_128": (2, 128, 128, 12)}),
    # Pose head (SURVEY.md 8(f) rank 4) on the v0_1 backbone: built with the reference's PoseModel
    "yolo-master-pose-n-v0_1": ("/root/reference/ultralytics/cfg/models/master/v0_1/pose/yolo-master-pose-n.yaml", [11, 23],
                                {"b2_128": (2, 128, 128, 14)}),
    # Segment head + Proto on the v0_1 backbone (reference model built from the seg YAML)
    "yolo-master-seg-n-v0_1": ("/root/reference/ultralytics/cfg/models/master/v0_1/seg/yolo-master-seg-n.yaml", [23],
                               {"b2_96": (2, 96, 96, 15)}),
    # OBB head on the v0_1 backbone (rotated boxes + angle row)
    "yolo-master-obb-n-v0_1": ("/root/reference/ultralytics/cfg/models/master/v0_1/obb/yolo-master-obb-n.yaml", [23],
                               {"b2_96": (2, 96, 96, 16)}),
    # LatentMixture (multi-input latent-routed mixture on every Detect input); residual_init 0.01 so that the experts contribute
    "yolo26-master-latent-n": ("/root/reference/ultralytics/cfg/models/26/yolo26-master-latent-n-resinit010.yaml", [22, 23, 24, 25],
                               {"b2_128": (2, 128, 128, 17)}),
    "yolo26-master-moa-mot-s": (("/root/reference/ultralytics/cfg/models/26/yolo26-master-moa-mot-n.yaml", "s", [0.50, 0.50, 1024]),
                                [13, 16, 19, 22], {"b1_160": (1, 160, 160, 8)}),
}


def _route_hooks(m, routes):
    """Capture MoT (dense weights, top-k indices) and MoA (soft weights) router outputs by module name."""
    from ultralytics.nn.modules.moa.router import _MoARouter
    from ultralytics.nn.modules.mot.router import _MoTRouter
    hooks = []
    for name, mod in m.named_modules():
        if isinstance(mod, _MoTRouter):
            hooks.append(mod.register_forward_hook(
                lambda mod, i, o, n=name: routes.__setitem__(n, (o[0].float().clone(), o[1].to(torch.int8).clone()))))
        elif isinstance(mod, _MoARouter):
            hooks.append(mod.register_forward_hook(
                lambda mod, i, o, n=name: routes.__setitem__(n, ((o[0] if isinstance(o, tuple) else o).float().clone(),))))
    return hooks


def extra_model_golden(name):
    """v0 family (ES_MOE x4, A2C2f area attention with/without layer-scale residual, DFL Detect, no end2end): per-layer
    activations, raw head outputs and the dense (B, 4+nc, A) prediction of the REAL reference."""
    cfg, keep, cases = EXTRA_MODELS[name]
    torch.manual_seed(0)
    if isinstance(cfg, tuple):      # (yaml, scale key, scale constants): inject a scale without editing the YAML file
        from ultralytics.nn.tasks import yaml_model_load
        d = yaml_model_load(cfg[0])
        d["scales"][cfg[1]] = cfg[2]
        d["scale"] = cfg[1]
        cfg = d
    m = calibrated_reference(0, cfg)
    sd = m.state_dict()
    json.dump({k: [list(v.shape), str(v.dtype)] for k, v in sd.items() if torch.is_tensor(v)}, open(f"{OUT}/{name}.keys.json", "w"))
    # calibrated BatchNorm statistics + the constants the key-seeded generator leaves alone (router temperature buffers,
    # the frozen DFL arange): everything a test needs besides key names to rebuild the exact state_dict
    stats = {k: v.clone() for k, v in sd.items() if torch.is_tensor(v) and (
             k.endswith(("running_mean", "running_var", ".temperature", "dfl.conv.weight"))
             or (v.is_floating_point() and v.dim() == 0))}       # scalar gates / scales keep their constructor values
    torch.save(stats, f"{OUT}/{name}.bnstats.pt")
    gold = {"cases": {}}
    for tag, (B, H, W, seed) in cases.items():
        x = synth_images(B, H, W, seed)
        routes = {}
        hooks = _route_hooks(m, routes)
        y, preds, feats, _ = run(m, x)
        for h in hooks:
            h.remove()
        proto = None
        if isinstance(y, tuple):            # Segment: (dense prediction + mask coefficients, prototypes)
            y, proto = y
        pr = preds["one2one"] if "one2one" in preds else preds
        gold["cases"][tag] = {"B": B, "H": H, "W": W, "seed": seed, "final": y.clone().half() if name.endswith("l-v0") else y.clone(),
                              "layers": {i: feats[i].clone() for i in keep},
                              "head_boxes": pr["boxes"].clone(), "head_scores": pr["scores"].clone(), "routes": routes}
        if proto is not None:
            gold["cases"][tag]["proto"] = proto.clone()
        print(name, tag, "final", tuple(y.shape), "max score", float(y[:, 4:].max()))
    torch.save(gold, f"{OUT}/{name}.golden.pt")
    for f in sorted(os.listdir(OUT)):
        if f.startswith(name):
            print(f, os.path.getsize(os.path.join(OUT, f)))


def dispatch_golden():
    """Reference BatchedExpertComputation (moe/utils.py:119-209) with 1x1-conv experts on small seeded cases."""
    from ultralytics.nn.modules.moe.utils import BatchedExpertComputation
    cases = []
    for seed, (B, C, H, W, E, k) in enumerate([(6, 32, 5, 7, 4, 2), (9, 16, 4, 4, 8, 2), (4, 24, 3, 3, 3, 1)]):
        g = torch.Generator().manual_seed(100 + seed)
        x = torch.randn((B, C, H, W), generator=g)
        Wt = torch.randn((E, C, C), generator=g) / C ** 0.5
        experts = torch.nn.ModuleList([torch.nn.Conv2d(C, C, 1, bias=False) for _ in range(E)]).eval()
        for e in range(E):
            experts[e].weight.data.copy_(Wt[e].view(C, C, 1, 1))
        idx = torch.stack([torch.randperm(E, generator=g)[:k] for _ in range(B)])
        w = torch.rand((B, k), generator=g)
        w = w / w.sum(1, keepdim=True)
        w[0, -1] = 0.004
        with torch.no_grad():
            out = BatchedExpertComputation.compute_sparse_experts_batched(x, experts, w, idx, k, E)
        cases.append({"x": x, "W": Wt, "w": w, "idx": idx, "out": out})
    torch.save({"cases": cases}, f"{OUT}/dispatch.golden.pt")


def synth_predictions(B, nc, A, seed, dense=True):
    """Seeded (B, 4+nc, A) predictions: xywh boxes in a 640x640 frame, clustered so that NMS has work to do."""
    g = torch.Generator().manual_seed(seed)
    ncl = max(A // 12, 1)
    centres = torch.rand((B, ncl, 2), generator=g) * 600 + 20
    sizes = torch.exp(torch.randn((B, ncl, 2), generator=g) * 0.5 + 3.6)
    which = torch.randint(0, ncl, (B, A), generator=g)
    cxy = torch.gather(centres, 1, which[..., None].expand(-1, -1, 2)) + torch.randn((B, A, 2), generator=g) * (4 if dense else 40)
    wh = torch.gather(sizes, 1, which[..., None].expand(-1, -1, 2)) * torch.exp(torch.randn((B, A, 2), generator=g) * 0.1)
    cls_of_cluster = torch.randint(0, nc, (B, ncl), generator=g)
    cl = torch.gather(cls_of_cluster, 1, which)
    scores = torch.rand((B, nc, A), generator=g) * 0.05
    peak = torch.rand((B, A), generator=g) ** 2
    scores.scatter_(1, cl[:, None, :], peak[:, None, :])
    return torch.cat([cxy.transpose(1, 2), wh.transpose(1, 2), scores], 1).contiguous()


def nms_golden():
    """Reference ultralytics.utils.nms.non_max_suppression (TorchNMS greedy kernel; torchvision not imported here)."""
    assert "torchvision" not in sys.modules
    from ultralytics.utils.nms import non_max_suppression
    cases = []
    for seed, (B, nc, A, conf, iou, max_det) in enumerate([(3, 80, 2100, 0.25, 0.7, 300), (2, 80, 8400, 0.25, 0.45, 300),
                                                           (2, 3, 500, 0.05, 0.5, 20), (1, 80, 1000, 0.99, 0.7, 300)]):
        pred = synth_predictions(B, nc, A, 500 + seed)
        out, keep = non_max_suppression(pred.clone(), conf, iou, max_det=max_det, return_idxs=True)
        cases.append({"B": B, "nc": nc, "A": A, "seed": 500 + seed, "conf": conf, "iou": iou, "max_det": max_det,
                      "out": [o.clone() for o in out], "keep": [k.clone().long().view(-1) for k in keep]})
        print("nms case", seed, [len(o) for o in out])
    torch.save({"cases": cases}, f"{OUT}/nms.golden.pt")


def synth_obb_predictions(B, nc, A, seed):
    """Seeded (B, 4+nc+1, A) OBB-head style predictions: clustered xywh boxes, class scores, angle in [-pi/4, 3pi/4)."""
    g = torch.Generator().manual_seed(seed)
    pred = synth_predictions(B, nc, A, seed)
    pred[:, 2:4] *= torch.exp(torch.randn((B, 2, A), generator=g) * 0.4)            # elongated boxes: the angle matters
    ncl = max(A // 12, 1)
    base = (torch.rand((B, ncl), generator=g) - 0.25) * torch.pi
    which = torch.randint(0, ncl, (B, A), generator=g)
    ang = torch.gather(base, 1, which) + torch.randn((B, A), generator=g) * 0.15
    return torch.cat([pred, ang[:, None, :]], 1).contiguous()


def postproc_golden():
    """Reference ops.process_mask (both branches) and non_max_suppression(rotated=True) on seeded inputs (inputs stored)."""
    from ultralytics.utils import ops
    from ultralytics.utils.nms import non_max_suppression
    masks = []
    for seed, (nm, mh, mw, n, shape) in enumerate([(32, 80, 80, 7, (320, 320)), (32, 24, 40, 5, (96, 160)), (8, 20, 12, 9, (77, 50)),
                                                    (32, 40, 40, 0, (160, 160)), (16, 28, 28, 17, (112, 112))]):
        g = torch.Generator().manual_seed(900 + seed)
        protos = (torch.randn((nm, mh, mw), generator=g) * 0.7).half().float()      # fp16-representable: the head emits fp16
        for _ in range(2):                                                          # smooth, so that the masks have structure
            protos = torch.nn.functional.avg_pool2d(protos[None], 3, 1, 1)[0]
        protos = protos.half().float()
        coef = torch.randn((n, nm), generator=g)
        cxy = torch.rand((n, 2), generator=g) * torch.tensor([shape[1], shape[0]])
        wh = torch.rand((n, 2), generator=g) * torch.tensor([shape[1], shape[0]]) * 0.6 + 2
        boxes = torch.cat([cxy - wh / 2, cxy + wh / 2], 1)
        if n:
            boxes[0] = torch.tensor([-5.0, -3.0, shape[1] + 4.0, shape[0] + 9.0])   # a box past every edge
        case = {"protos": protos, "coef": coef, "boxes": boxes, "shape": shape}
        for up in (True, False):
            m = ops.process_mask(protos.clone(), coef.clone(), boxes.clone(), shape, upsample=up)
            assert m.dtype == torch.uint8 and int(m.max()) <= 1 if m.numel() else True
            key = "up" if up else "native"                                          # 0 / 1 masks, stored as packed bits
            case[key + "_shape"], case[key + "_bits"] = tuple(m.shape), torch.from_numpy(np.packbits(m.numpy().reshape(-1)))
            print("mask case", seed, key, tuple(m.shape), int(m.sum()))
        masks.append(case)
    nms = []
    for seed, (B, nc, A, conf, iou, max_det, max_nms) in enumerate([(2, 15, 2100, 0.25, 0.45, 300, 30000), (2, 3, 600, 0.05, 0.3, 25, 30000),
                                                                     (1, 15, 1500, 0.01, 0.6, 300, 400), (1, 4, 300, 0.999, 0.45, 300, 30000)]):
        pred = synth_obb_predictions(B, nc, A, 950 + seed)
        out, keep = non_max_suppression(pred.clone(), conf, iou, nc=nc, max_det=max_det, max_nms=max_nms, rotated=True, return_idxs=True)
        nms.append({"pred": pred, "nc": nc, "conf": conf, "iou": iou, "max_det": max_det, "max_nms": max_nms,
                    "out": [o.clone() for o in out], "keep": [k.clone().long().view(-1) for k in keep]})
        print("rotated nms case", seed, [len(o) for o in out])
    torch.save({"masks": masks, "nms": nms}, f"{OUT}/postproc.golden.pt")


ESMOE_CASES = [(64, 4, 2, 20, 24, 6), (32, 4, 2, 9, 7, 5), (128, 4, 2, 10, 10, 4)]   # C, E, top_k, H, W, B


def esmoe_weights(sd, seed):
    """Key-seeded fill + wider router logits so that the 0.4 dynamic threshold is exercised both ways."""
    fill_state_dict_(sd, 40 + seed)
    for k in sd:
        if k.endswith("routing_network.2.weight"):
            sd[k] *= 6
    return sd


def esmoe_golden():
    """Reference ES_MOE (moe/modules.py:410-741) eval outputs; weights are regenerated from key names by the tests."""
    from ultralytics.nn.modules.moe.modules import ES_MOE
    from ultralytics.utils.torch_utils import initialize_weights
    cases = []
    for seed, (C, E, k, H, W, B) in enumerate(ESMOE_CASES):
        m = ES_MOE(C, C, num_experts=E, top_k=k)
        initialize_weights(m)
        m.load_state_dict(esmoe_weights(m.state_dict(), seed))
        m.eval()
        x = torch.randn((B, C, H, W), generator=torch.Generator().manual_seed(seed))
        with torch.no_grad():
            y = m(x)
        cases.append({"seed": seed, "keys": {kk: list(v.shape) for kk, v in m.state_dict().items()}, "y": y.clone()})
    torch.save({"cases": cases}, f"{OUT}/esmoe.golden.pt")


LETTERBOX_CASES = [(480, 640), (720, 1280), (1080, 1920), (1200, 1600), (427, 640), (640, 480), (333, 500), (100, 37), (64, 64)]


LETTERBOX_VARIANTS = [(300, 400, (640, 640), {"auto": True}), (500, 333, (640, 640), {"auto": True}),
                      (200, 300, (640, 640), {"scaleup": False}), (375, 500, (640, 640), {"scale_fill": True}),
                      (480, 640, (640, 640), {"center": False}), (1080, 1920, (384, 640), {}), (97, 211, (320, 416), {"auto": True})]
SCALE_BOX_CASES = [((640, 640), (480, 640)), ((640, 640), (1080, 1920)), ((384, 640), (720, 1280)), ((640, 640), (100, 37)),
                   ((640, 640), (333, 500, 3))]


def letterbox_golden():
    """Reference pre-processing of one seeded uint8 BGR frame per case: the REAL `LetterBox` (cv2.resize INTER_LINEAR +
    copyMakeBorder 114) followed by the predictor's BGR->RGB / HWC->CHW (engine/predictor.py:164-170).  Stores only a CRC and a
    coarse 16x16 block-mean thumbnail per case (the expected tensors are 1.2 MB each) plus the cv2 version."""
    import zlib

    import cv2
    import numpy as np
    from ultralytics.data.augment import LetterBox
    cases = []
    for seed, (h, w) in enumerate(LETTERBOX_CASES):
        img = np.random.default_rng(900 + seed).integers(0, 256, (h, w, 3), dtype=np.uint8)
        out = LetterBox((640, 640), auto=False, stride=32)(image=img)
        chw = np.ascontiguousarray(out[..., ::-1].transpose(2, 0, 1))
        cases.append({"h": h, "w": w, "seed": 900 + seed, "crc": zlib.crc32(chw.tobytes()), "shape": list(chw.shape),
                      "thumb": torch.from_numpy(chw.reshape(3, 40, 16, 40, 16).astype(np.float32).mean((2, 4)))})
        print("letterbox", (h, w), chw.shape, cases[-1]["crc"])
    # LetterBox option variants (HWC output of the transform itself) and `ops.scale_boxes` on seeded boxes
    from ultralytics.utils import ops
    variants = []
    for seed, (h, w, new_shape, kw) in enumerate(LETTERBOX_VARIANTS):
        img = np.random.default_rng(950 + seed).integers(0, 256, (h, w, 3), dtype=np.uint8)
        lb = LetterBox(new_shape, stride=32, **kw)
        out = lb(image=img)
        prm = lb.get_params({"img": img})
        variants.append({"h": h, "w": w, "seed": 950 + seed, "new_shape": new_shape, "kw": kw, "shape": list(out.shape),
                         "crc": zlib.crc32(np.ascontiguousarray(out).tobytes()),
                         "params": [list(prm["new_unpad"]), prm["top"], prm["bottom"], prm["left"], prm["right"]]})
        print("letterbox variant", (h, w), new_shape, kw, out.shape)
    boxes = []
    for seed, (img1, img0) in enumerate(SCALE_BOX_CASES):
        g = torch.Generator().manual_seed(970 + seed)
        b = torch.rand((64, 6), generator=g) * torch.tensor([img1[1], img1[0], img1[1], img1[0], 1, 80]) * 1.1 - 8.0
        for xywh in (False, True):
            boxes.append({"img1": img1, "img0": img0, "seed": 970 + seed, "xywh": xywh,
                          "out": ops.scale_boxes(img1, b[:, :4].clone(), img0, xywh=xywh)})
    torch.save({"cv2": cv2.__version__, "cases": cases, "variants": variants, "scale_boxes": boxes}, f"{OUT}/letterbox.golden.pt")


def scale_coords_golden():
    """The reference's `ops.scale_coords` (640x640 -> frame, with and without `normalize`) on seeded keypoints that straddle the
    frame: inputs and fp32 outputs."""
    from ultralytics.utils import ops
    g = torch.Generator().manual_seed(12)
    cases = []
    for shape0 in ((480, 640), (1080, 1920), (100, 37), (640, 640)):
        for norm in (False, True):
            k = torch.rand((7, 17, 3), generator=g) * 800 - 60
            cases.append({"shape0": shape0, "normalize": norm, "coords": k,
                          "out": ops.scale_coords((640, 640), k.clone(), shape0, normalize=norm)})
    torch.save({"cases": cases}, f"{OUT}/scale_coords.golden.pt")
    print("scale_coords", len(cases), os.path.getsize(f"{OUT}/scale_coords.golden.pt"))


def zoo_golden():
    """The reference's model zoo as tests/test_zoo_builds.py reads it: every detection YAML (`master/**/det`, `master/exp`, the
    `26/*master*` files) and the n file of every seg / pose / obb / cls family, parsed, keyed by the path below `cfg/models`, one
    file per line."""
    import glob

    import ultralytics
    import yaml
    ref = os.path.join(os.path.dirname(ultralytics.__file__), "cfg", "models")
    files = sorted(glob.glob(f"{ref}/master/**/*.yaml", recursive=True) + glob.glob(f"{ref}/26/*master*.yaml"))
    files = [f for f in files if "/det/" in f or "/26/" in f or "/exp/" in f
             or (any(f"/{t}/" in f for t in ("seg", "pose", "obb", "cls")) and f.endswith("-n.yaml"))]
    rows = [f"{json.dumps(os.path.relpath(f, ref))}: {json.dumps(yaml.safe_load(open(f)), separators=(',', ':'))}" for f in files]
    with open(f"{OUT}/zoo.golden.json", "w") as f:
        f.write("{\n" + ",\n".join(rows) + "\n}\n")
    print("zoo", len(rows), os.path.getsize(f"{OUT}/zoo.golden.json"))


def cls_golden():
    """Reference ClassificationModel (v0_1 cls n: ModularRouterExpertMoE backbone + Classify) on seeded 64x64 images: probabilities,
    logits and the layer-11 feature; key table + calibrated BatchNorm statistics like the other model fixtures."""
    from ultralytics.nn.tasks import ClassificationModel
    name = "yolo-master-cls-n-v0_1"
    m = ClassificationModel("/root/reference/ultralytics/cfg/models/master/v0_1/cls/yolo-master-cls-n.yaml", verbose=False)
    sd = m.state_dict()
    fill_state_dict_(sd, 0)
    m.load_state_dict(sd)
    m.eval()
    bns = [mod for mod in m.modules() if isinstance(mod, torch.nn.BatchNorm2d)]
    for b in bns:
        b.train()
        b.momentum = None
        b.reset_running_stats()
    with torch.no_grad():
        m(synth_images(8, 128, 128, seed=7))
    for b in bns:
        b.eval()
        b.momentum = 0.03
    sd = m.state_dict()
    json.dump({k: [list(v.shape), str(v.dtype)] for k, v in sd.items() if torch.is_tensor(v)}, open(f"{OUT}/{name}.keys.json", "w"))
    stats = {k: v.clone() for k, v in sd.items() if k.endswith(("running_mean", "running_var", "num_batches_tracked"))
             or (v.dim() == 0 and v.is_floating_point())}
    torch.save(stats, f"{OUT}/{name}.bnstats.pt")
    x = synth_images(3, 64, 64, 21)
    feats = {}
    h = m.model[11].register_forward_hook(lambda mod, i, o: feats.__setitem__(11, o.clone()))
    with torch.no_grad():
        y, logits = m(x)
    h.remove()
    torch.save({"cases": {"b3_64": {"B": 3, "H": 64, "W": 64, "seed": 21, "final": y.clone(), "logits": logits.clone(), "layers": feats}}},
               f"{OUT}/{name}.golden.pt")
    print(name, tuple(y.shape), float(y.max()), [os.path.getsize(f"{OUT}/{name}{e}") for e in (".golden.pt", ".bnstats.pt", ".keys.json")])


GATED_FAMILY = ["AdaptiveGateMoE", "FusedAdaptiveGateMoE", "HybridAdaptiveGateMoE", "LowRankHybridAdaptiveGateMoE",
                "RefinedLowRankHybridAdaptiveGateMoE", "DetailAwareLowRankHybridAdaptiveGateMoE",
                "ContextRefinedLowRankHybridAdaptiveGateMoE", "VisualEnhancedAdaptiveGateMoE"]


def gated_family_golden():
    """Module-level goldens of every class of the AdaptiveGateMoE line (v0_4 ... v0_10 model zoos): the REAL reference module
    (c1 = c2 = 64, top-2 of 4 and of 16 experts, key-seeded weights) on a seeded (2, 64, 12, 12) input -> output, router decisions
    before the complexity gate, and the state-dict key table."""
    from ultralytics.nn.modules.moe import gated as G
    path = f"{OUT}/gated_family.golden.pt"
    out = torch.load(path) if os.path.exists(path) and not os.environ.get("GATED_REGEN") else {}
    from ultralytics.nn.modules.moe import modules as MM
    for ci, name in enumerate(GATED_FAMILY + ["UltimateOptimizedMoE", "HybridAdaptiveGateMoEv2", "OptimalHybridGateMoE", "MultiHeadRouterMoE", "GatedFusionMoE", "UltraOptimizedMoE", "DiversifiedExpertMoE"]):
        for E in (4, 16):
            if f"{name}/E{E}" in out:                    # entries are deterministic; GATED_REGEN=1 recomputes them all
                continue
            torch.manual_seed(0)
            split = 0.375 if (E == 16 and name in ("HybridAdaptiveGateMoEv2", "OptimalHybridGateMoE", "MultiHeadRouterMoE", "GatedFusionMoE", "DiversifiedExpertMoE")) else 0.5   # the v0_11 / v0_12 P5 setting
            if name == "UltraOptimizedMoE":          # (in, out, num_experts, top_k): no channel split
                m = MM.UltraOptimizedMoE(64, 64, E, 2).eval()
            else:
                m = getattr(G if hasattr(G, name) and name != "UltimateOptimizedMoE" else MM, name)(64, 64, E, 2, split).eval()
            for mod in m.modules():                      # inside a model every BatchNorm2d runs with eps = 1e-3
                if isinstance(mod, torch.nn.BatchNorm2d):   # (initialize_weights, utils/torch_utils.py:552-562)
                    mod.eps = 1e-3
            sd = m.state_dict()
            fill_state_dict_(sd, 300 + ci)
            for k, v in sd.items():                      # 0-dim parameters keep their init values; a zero one (CrossPathGate's
                if v.dim() == 0 and v.is_floating_point() and float(v) == 0.0:   # gate_scale) would switch its branch off
                    v.fill_(0.7)
            if name == "GatedFusionMoE":                 # its last Linear is zero-initialised and the key-seeded fill keeps
                g = torch.Generator().manual_seed(77)    # "bias" tensors small: give the gate something to do
                sd["cross_gate.gate_net.4.bias"].copy_(torch.randn(sd["cross_gate.gate_net.4.bias"].shape, generator=g))
            m.load_state_dict(sd)
            hw = 24 if name == "UltraOptimizedMoE" else 12        # its router pools 8x8: 24x24 exercises the pooled branch
            x = torch.randn((2, 64, hw, hw), generator=torch.Generator().manual_seed(400 + ci))
            route = {}
            h = m.routing.register_forward_hook(lambda mod, i, o: route.update(w=o[0].flatten(1).clone(), idx=o[1].flatten(1).clone()))
            with torch.no_grad():
                y = m(x)
            h.remove()
            out[f"{name}/E{E}"] = {"seed": 300 + ci, "xseed": 400 + ci, "split": split, "y": y.clone(), "route_w": route["w"], "route_idx": route["idx"],
                                   "keys": {k: list(v.shape) for k, v in sd.items()},
                                   "scalars": {k: v.clone() for k, v in sd.items() if (v.dim() == 0 and v.is_floating_point()) or k == "cross_gate.gate_net.4.bias"},
                                   "backend": getattr(m, "expert_backend", "fused" if name == "UltimateOptimizedMoE" else "shared_inverted"), "hw": hw}
            print("gated", name, E, out[f"{name}/E{E}"]["backend"], float(y.abs().mean()))
    torch.save(out, f"{OUT}/gated_family.golden.pt")


if __name__ == "__main__":
    which = sys.argv[1:] or ["main", "dispatch", "nms", "postproc", "esmoe", "letterbox", "scale_coords", "zoo", "gated_family", "cls",
                             *EXTRA_MODELS]
    for w in which:
        if w in EXTRA_MODELS:
            extra_model_golden(w)
        else:
            {"main": main, "dispatch": dispatch_golden, "nms": nms_golden, "postproc": postproc_golden, "esmoe": esmoe_golden, "letterbox": letterbox_golden,
             "gated_family": gated_family_golden, "cls": cls_golden, "scale_coords": scale_coords_golden, "zoo": zoo_golden}[w]()
