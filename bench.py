#!/usr/bin/env python
"""Benchmark of the hot path: yolo26-master-n detection forward, synthetic 640x640 batches (BASELINE.json configs[1]).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

One "step" = one forward pass of a batch of 32 synthetic images per GPU (weak scaling: per-GPU batch fixed).
  value     images/s with the batch already resident in HBM (CUDA-graph replay of the whole forward, CUDA events,
            max over ranks)
  e2e       images/s through the host-buffer call: pinned host images -> H2D -> forward -> D2H of the (B,300,6) result
  roofline  dominant kernel (area attention at P3) timed live with CUDA events, vs MEASURED_PEAKS.json
  cpu_baseline  the unmodified reference (oracle/_ref/ultralytics, built by `make -C oracle`) on a bounded sample, host cores stated
  torch_eager_gpu  the same unmodified reference as torch-eager on this GPU (the north-star's same-box baseline)
`--impl reference` times the reference's own PyTorch-CPU forward (fp32, all useful host threads) on rank 0, same 32-image batch.
Prints ONE JSON line on rank 0.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import torch  # noqa: E402

METRIC = "images/sec @ 640x640 bs32"
UNIT = "images/s"
IMG = 640
FLOPS_PER_IMAGE = 30.23e9      # SURVEY.md §8d: conv 7.67 G + attention bmm 22.57 G (2*MAC)
BYTES_PER_IMAGE = 139e6        # SURVEY.md §8d algorithmic fp16 bytes (unfused layer I/O + attention streams)
# one ex2 per attention score: AAttn at P3 / P4 / P5 (two ABlockMoE each, 2 heads) + C2PSA's Attention at P5 (2 heads)
EXPS_PER_IMAGE = 2 * 2 * (6400.0 ** 2 + 1600.0 ** 2 + 400.0 ** 2) + 2 * 400.0 ** 2
SM_CLOCK_HZ = 1.965e9          # clocks.max.sm of the pool's B200s (the bench records the clock it saw under load)


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return {"hbm_gbs": d["hbm_gbs"], "tflops_burst": d["bf16_tflops"], "tflops_sustained": d["bf16_tflops_sustained"],
                "source": "MEASURED_PEAKS.json (of measured)"}
    return {"hbm_gbs": 6650.0, "tflops_burst": 1590.0, "tflops_sustained": 1400.0, "source": "B200_PROFILING.md fallback (of fallback)"}


def synthetic_weights():
    from _util import synth_sd_from_keys
    return synth_sd_from_keys(0)


class ClockSampler:
    """nvidia-smi clock / throttle sampling during the timed region (B200_PROFILING.md recipe)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.proc, self.path = index, None, f"/tmp/ym_clocks_{os.getpid()}.csv"

    def __enter__(self):
        try:
            self.f = open(self.path, "w")
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "20",
                                          "-i", str(self.index)], stdout=self.f, stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None
        return self

    def __exit__(self, *a):
        if self.proc is not None:
            time.sleep(0.15)
            self.proc.terminate()
            try:
                self.proc.wait(timeout=5)
            except Exception:
                self.proc.kill()
            self.f.close()

    def summary(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        try:
            rows = [r.strip().split(", ") for r in open(self.path) if r.strip()]
            sm = sorted(float(r[1]) for r in rows)
            if sm:
                out["sm_mhz"] = sm[len(sm) // 2]
                out["sm_max_mhz"] = float(rows[0][2])
                out["samples"] = len(sm)
                out["power_w_max"] = max(float(r[3]) for r in rows)
                names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
                for j, n in enumerate(names):
                    if any(r[5 + j].strip().lower().startswith("active") for r in rows):
                        out["reasons"].append(n)
            os.remove(self.path)
        except Exception as e:  # clocks are evidence, never a reason to lose the number
            out["error"] = str(e)
        return out


def dump_outputs(out_dir, arrays):
    """Writes each tensor as `out_dir/<name>.npy` (float32), so that the outputs of two builds on the same seeded inputs can be compared."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    for name, t in arrays.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), t.detach().float().cpu().numpy())


def pick_cpu_threads(forward_one):
    """The reference's PyTorch-CPU path does not scale to every core of a large host (N x N attention is memory bound):
    probe 8/16/32/64/all threads on one image and keep the fastest, so the CPU arm is shown at its best."""
    cores = os.cpu_count() or 1
    best_t, best = None, 1e30
    for t in sorted({min(c, cores) for c in (8, 16, 32, 64, cores)}):
        torch.set_num_threads(t)
        forward_one()
        t0 = time.perf_counter()
        forward_one()
        dt = time.perf_counter() - t0
        if dt < best:
            best, best_t = dt, t
        elif dt > 1.5 * best:
            break
    torch.set_num_threads(best_t)
    return best_t, cores


def bench_config(world, B):
    """ONE config dict for both arms (ours / --impl reference): same workload, same batch, same image size."""
    return {"workload": "yolo26-master-n forward, 640x640, bs32 per GPU (BASELINE.json configs[1]); random-init weights (key-seeded) "
                        "with calibrated BatchNorm statistics; ES-MoE top-2 of 4/8/16 experts",
            "global_batch": world * B, "batch_per_gpu": B, "imgsz": IMG,
            "parallelism": f"replicas x{world} (no data-path collective)",
            "l2": f"4 rotating input batches ({4 * B * 3 * IMG * IMG * 2 / 1e6:.0f} MB) and ~{BYTES_PER_IMAGE * B / 1e9:.1f} GB of per-step "
                  "activations exceed the 126 MB L2"}


def reference_model(device="cpu", half=False):
    """The UNMODIFIED reference (`oracle/_ref/ultralytics`, built by `make -C oracle`): its own DetectionModel, YAML and
    `_predict_once`, `.eval().fuse()`, with the same key-seeded synthetic weights as our arm.  Returns (callable, kind)."""
    from oracle import reference_runner as R
    if R.available():
        m = R.build_reference_model(synthetic_weights())
        if half:
            m = m.half()
        m = m.to(device)
        return (lambda x: m(x)[0]), "reference"
    # oracle/_ref absent (it is git-ignored: `make -C oracle` was not run where /root/reference exists): the oracle port
    from _util import yaml_n
    from oracle import yolo_master_oracle as O
    spec = O.parse_spec(yaml_n())
    sd = {k: (v.to(device).half() if (half and v.is_floating_point()) else v.to(device)) for k, v in synthetic_weights().items()}
    return (lambda x: O.forward(spec, sd, x, dtype=torch.float16 if half else torch.float32)), "port"


def run_reference(args):
    """Reference arm: the reference's own PyTorch-CPU forward (stock `ultralytics.nn.tasks.DetectionModel`, fp32 - the CPU path has
    no fp16), all useful host threads, on the SAME config as our arm: one step = one 32-image 640x640 batch."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from yolo_master_b200.utils.synth import synth_images

    B = args.batch
    fwd, kind = reference_model("cpu", False)
    xs = [synth_images(B, IMG, IMG, 100 + i) for i in range(2)]
    with torch.inference_mode():
        cores, host_cores = pick_cpu_threads(lambda: fwd(xs[0][:4]))
        for i in range(args.warmup):
            fwd(xs[i % 2])
        t0 = time.perf_counter()
        for i in range(args.steps):
            y = fwd(xs[i % 2])
        dt = time.perf_counter() - t0
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"detections": y})
    v = B * args.steps / dt
    src = ("unmodified reference: oracle/_ref/ultralytics DetectionModel('yolo26-master-n.yaml').eval().fuse()" if kind == "reference"
           else "oracle port of the reference forward (oracle/_ref missing)")
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": bench_config(args.gpus, B),
        "cpu_baseline": {"value": v, "unit": UNIT, "cores": cores, "kind": kind,
                         "sample": f"{args.steps} steps x {B} synthetic 640x640 images (the full batch of configs[1]), fp32 PyTorch-CPU, {src}; "
                                   f"{cores} threads (fastest of 8/16/32/64/{host_cores} on this {host_cores}-core host)"},
        "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


def time_attention_kernel(dev, batch, pk):
    """Dominant kernel, timed alone on the launching stream: AAttn at P3 (80x80 tokens, 2 heads x 32) for the full batch."""
    from yolo_master_b200 import ops
    N, heads, hd = (IMG // 8) ** 2, 2, 32
    qkv = torch.randn((batch, IMG // 8, IMG // 8, 3 * heads * hd), device=dev).half()
    out = ops.new_act(batch, IMG // 8, IMG // 8, heads * hd, dev)
    for _ in range(3):
        ops.attention(qkv, batch, N, heads, 3 * hd, 0, hd, 2 * hd, hd, hd, hd ** -0.5, out=out)
    reps = 10
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for _ in range(reps):
        ops.attention(qkv, batch, N, heads, 3 * hd, 0, hd, 2 * hd, hd, hd, hd ** -0.5, out=out)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / reps
    flops = 4.0 * N * N * hd * heads * batch
    algo_bytes = 4.0 * N * hd * heads * batch * 2
    tf = flops / (ms * 1e-3) / 1e12
    traffic = None
    try:   # DRAM bytes per launch of this kernel from the committed `ncu --set full` capture (profiles/, read - not measured - here)
        tj = json.load(open(os.path.join(ROOT, "profiles", "r02_traffic.json")))["tc_attention2_kernel<32>"]
        if batch == 32:
            traffic = tj["dram_bytes_read"] + tj["dram_bytes_write"]
    except Exception:
        pass
    exps = float(N) * N * heads * batch
    texp = exps / (ms * 1e-3) / 1e12
    exp_peak = 148 * 16 * SM_CLOCK_HZ / 1e12          # 16 ex2 per clock per SM on the MUFU (B300_MICROARCH.md), at the measured clock
    return {"kernel": "tc_attention2_kernel<32> (warp-specialised tcgen05: S = QK^T SS-mode, O += PV TS-mode with P in tensor memory, TMA K/V ring; "
                      "AAttn P3: N=6400, 2 heads x d32, whole batch)",
            "bound": "exp", "achieved": texp, "peak": exp_peak, "unit": "Texp/s", "frac": texp / exp_peak,
            "tensor": {"achieved": tf, "peak": pk["tflops_burst"], "unit": "TFLOP/s", "frac": tf / pk["tflops_burst"]},
            "traffic": traffic, "traffic_source": "profiles/r02_traffic.json (ncu --set full of the same launch; committed, not measured in this run)",
            "ms_per_launch": ms, "algorithmic_flops_per_launch": flops, "algorithmic_bytes_per_launch": algo_bytes,
            "exp_per_launch": exps,
            "note": "softmax attention at d=32 is bound by one ex2 per score on the MUFU (16 lanes/clk/SM -> 4.65 T scores/s at 1965 MHz), "
                    "not by the tensor pipe (128 FLOP per score -> 27 % of the bf16 peak AT that ceiling) nor by HBM (K/V are L2-resident); "
                    "`frac` is therefore achieved / MUFU ceiling and `tensor.frac` is reported beside it (SURVEY.md 8d); peaks " + pk["source"]}


def model_roofline(images_per_s_per_gpu, pk):
    """Whole-forward lower bounds per image (SURVEY.md 8d) and where the measured step sits against the binding one."""
    t_hbm = BYTES_PER_IMAGE / (pk["hbm_gbs"] * 1e9)
    t_tensor = FLOPS_PER_IMAGE / (pk["tflops_sustained"] * 1e12)
    t_exp = EXPS_PER_IMAGE / (148 * 16 * SM_CLOCK_HZ)
    bound = max((t_exp, "exp"), (t_hbm, "hbm"), (t_tensor, "tensor"))
    t_img = 1.0 / images_per_s_per_gpu
    return {"flops_per_image": FLOPS_PER_IMAGE, "bytes_per_image": BYTES_PER_IMAGE, "exps_per_image": EXPS_PER_IMAGE,
            "lower_bound_us_per_image": {"hbm": t_hbm * 1e6, "tensor": t_tensor * 1e6, "exp": t_exp * 1e6},
            "bound": bound[1], "achieved": bound[0] / t_img, "unit": "fraction of the binding lower bound (max of the three) per image",
            "us_per_image": t_img * 1e6,
            "tflops": FLOPS_PER_IMAGE * images_per_s_per_gpu / 1e12, "algorithmic_gbs": BYTES_PER_IMAGE * images_per_s_per_gpu / 1e9,
            "hbm_frac": t_hbm / t_img, "tensor_frac": t_tensor / t_img, "exp_frac": t_exp / t_img}


def time_dispatch(dev, pk, B=64, baseline=True):
    """ES-MoE dispatch microbench (BASELINE.json configs[4]): B*1024 tokens (65536 at B=64) x d=256, 8 experts, top-2, 1x1-conv
    experts (BatchedExpertComputation semantics).  Algorithmic bytes = (k+1)*d*2 = 1536 B/token (SURVEY.md §8d)."""
    from yolo_master_b200 import ops
    C, H, W, E, K = 256, 32, 32, 8, 2
    g = torch.Generator().manual_seed(0)
    nrot = max(6, min(64, int(200e6 / (2 * B * H * W * C * 2)) + 1))   # rotating in/out buffers exceed the 126 MB L2 (6 x 33.5 MB x 2 at B=64)
    xs = [torch.randn((B, H, W, C), generator=g).half().to(dev) for _ in range(nrot)]
    outs = [ops.new_act(B, H, W, C, dev) for _ in range(nrot)]
    Wt = (torch.randn((E, C, C), generator=g) / C ** 0.5).half().to(dev)
    idx = torch.stack([torch.randperm(E, generator=g)[:K] for _ in range(B)]).int().to(dev)
    w = torch.rand((B, K), generator=g)
    w = (w / w.sum(1, keepdim=True)).to(dev)
    for i in range(3):
        ops.moe_dispatch(xs[i % nrot], Wt, idx, w, out=outs[i % nrot])
    # one CUDA graph over the rotating buffers: the timed region is kernel time, not ctypes / tensor-map-encode host time
    side = torch.cuda.Stream(device=dev)
    side.wait_stream(torch.cuda.current_stream(dev))
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph, stream=side):
        for i in range(nrot):
            ops.moe_dispatch(xs[i], Wt, idx, w, out=outs[i])
    graph.replay()
    reps = 5
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for i in range(reps):
        graph.replay()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / (reps * nrot)
    tokens = B * H * W
    gbs = 1536.0 * tokens / (ms * 1e-3) / 1e9
    res = {"workload": f"{B * H * W} tokens x d=256, 8 experts top-2, 1x1-conv experts (configs[4])", "kernel": "tc_dispatch2_kernel<256> (2-CTA clusters, tcgen05.mma.cta_group::2 M=256 N=256, TMA loads/stores, TMEM slot ring)",
           "ms": ms, "tokens_per_s": tokens / (ms * 1e-3), "algorithmic_gbs": gbs, "hbm_frac": gbs / pk["hbm_gbs"],
           "tflops": 2.0 * K * C * C * tokens / (ms * 1e-3) / 1e12, "bytes_per_token": 1536}
    if not baseline:
        return res
    # the reference's torch path on the same GPU (restated dispatcher on CUDA tensors, fp16): a baseline, not the product
    try:
        from oracle.moe_dispatch_oracle import compute_sparse_experts_batched, conv1x1_experts

        xr = xs[0].permute(0, 3, 1, 2).contiguous()
        ex = conv1x1_experts(Wt)
        for _ in range(2):
            compute_sparse_experts_batched(xr, ex, w, idx.long(), C)
        torch.cuda.synchronize()
        e0.record()
        for _ in range(5):
            compute_sparse_experts_batched(xr, ex, w, idx.long(), C)
        e1.record()
        torch.cuda.synchronize()
        mr = e0.elapsed_time(e1) / 5
        res["torch_eager_gpu"] = {"ms": mr, "algorithmic_gbs": 1536.0 * tokens / (mr * 1e-3) / 1e9,
                                  "note": "reference dispatcher (Python loop over experts, gather, conv, index_add_) on this GPU"}
    except Exception as e:  # baseline only
        res["torch_eager_gpu"] = {"error": str(e)[:200]}
    return res


def time_torch_eager_gpu(dev, B):
    """The reference's own torch-eager path ON THIS GPU: the unmodified `ultralytics` DetectionModel (oracle/_ref),
    `.eval().fuse().half().cuda()`, same weights, same 32-image batch - the same-box GPU baseline BASELINE.json's north_star names
    (nn/tasks.py:182-218 with its host syncs, moe/modules.py:1128-1142 Python expert loop).  A baseline leg like cpu_baseline:
    never part of the product path, timed after the product numbers are taken."""
    from yolo_master_b200.utils.synth import synth_images
    out = {}
    for half in (True, False):
        tag = "fp16" if half else "fp32"
        try:
            fwd, kind = reference_model(dev, half)
            xs = [synth_images(B, IMG, IMG, 300 + i).to(dev) for i in range(2)]
            xs = [x.half() if half else x for x in xs]
            with torch.inference_mode():
                for i in range(3):
                    fwd(xs[i % 2])
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                torch.cuda.synchronize()
                reps = 6
                e0.record()
                for i in range(reps):
                    fwd(xs[i % 2])
                e1.record()
                torch.cuda.synchronize()
            ms = e0.elapsed_time(e1) / reps
            out[tag] = {"value": B / (ms * 1e-3), "unit": UNIT, "ms_per_step": ms, "kind": kind}
            del fwd, xs
        except Exception as e:  # baseline only
            out[tag] = {"error": f"{type(e).__name__}: {str(e)[:300]}"}
        torch.cuda.empty_cache()
    best = max((v for v in out.values() if "value" in v), key=lambda v: v["value"], default=None)
    if best is None:
        return {"error": out}
    return {"value": best["value"], "unit": UNIT, "ms_per_step": best["ms_per_step"], "kind": best["kind"], "by_dtype": out,
            "note": "unmodified reference DetectionModel (oracle/_ref), torch-eager on the same B200, device-resident input, CUDA events, "
                    "6 steps of the same 32-image batch; the faster of fp16 / fp32 is the headline baseline"}


class _GraphedDetector:
    """The graphed uint8 forward with the attributes DetectionPredictor reads from a model."""

    def __init__(self, model, graphed):
        self._model, self._g = model, graphed
        self.stride, self.end2end, self.names = model.stride, True, getattr(model, "names", None)
        self.model = model.model

    def parameters(self):
        return self._model.parameters()

    def __call__(self, im):
        return self._g(im)


def time_predictor(model, g8, B, dev, steps, warmup):
    """Second end-to-end figure, through the predictor API (engine/predictor.py:155-206 of the reference): B raw 1280x720 BGR uint8 frames
    (numpy, pageable host memory, as cv2 hands them over) -> DetectionPredictor: pinned staging + H2D, device letterbox to 640x640,
    the graphed forward, confidence filter, boxes back to frame coordinates, `Results` objects -> detections read back to the host.
    Every step is one synchronous call; nothing overlaps between steps."""
    import numpy as np
    from yolo_master_b200.engine.predictor import DetectionPredictor
    rng = np.random.default_rng(0)
    frames = [[rng.integers(0, 256, (720, 1280, 3), dtype=np.uint8) for _ in range(B)] for _ in range(2)]
    pred = DetectionPredictor(_GraphedDetector(model, g8), imgsz=IMG, conf=0.25, half=None, device=dev)

    def step(i):
        res = pred(frames[i % 2])
        rows = torch.cat([r.boxes.data for r in res]) if res else torch.zeros((0, 6))
        return rows.cpu()

    for i in range(max(1, warmup)):
        step(i)
    torch.cuda.synchronize(dev)
    t0 = time.perf_counter()
    for i in range(steps):
        out = step(i)
    torch.cuda.synchronize(dev)
    ms = (time.perf_counter() - t0) * 1e3
    return {"value": B * steps / (ms * 1e-3), "unit": UNIT, "ms_per_step": ms / steps, "h2d_bytes_per_step": B * 720 * 1280 * 3,
            "d2h_bytes_per_step": int(out.numel() * out.element_size()),
            "api": "DetectionPredictor(frames) -> list[Results], one synchronous call per batch",
            "input": f"{B} raw 1280x720 BGR uint8 numpy frames per step (pageable memory); letterbox on the device"}


def time_two_streams(model, dev_in, B, steps, warmup, dev):
    """EXPERIMENT, reported beside the headline, never as it: two CUDA-graph instances of the forward (own activation pools) replayed on
    two streams, alternate batches to alternate streams - the MUFU-bound attention of one batch can overlap the latency / HBM-bound
    convolutions of the other.  Same K steps of 32 images; time = first launch to last completion."""
    from yolo_master_b200.nn.tasks import GraphedForward
    try:
        gs = [GraphedForward(model, B, IMG, IMG, torch.float16) for _ in range(2)]
        streams = [torch.cuda.Stream(device=dev) for _ in range(2)]
        for j in range(2):
            gs[j].static_in.copy_(dev_in[j])
        cur = torch.cuda.current_stream(dev)

        def run(n):
            for s in streams:
                s.wait_stream(cur)
            for i in range(n):
                with torch.cuda.stream(streams[i & 1]):
                    gs[i & 1].graph.replay()
            for s in streams:
                cur.wait_stream(s)
        run(warmup)
        torch.cuda.synchronize(dev)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        run(steps)
        e1.record()
        torch.cuda.synchronize(dev)
        ms = e0.elapsed_time(e1)
        return {"value": B * steps / (ms * 1e-3), "unit": UNIT, "ms_per_step": ms / steps,
                "note": "two forward graphs on two streams, batches alternate; throughput experiment, not the headline"}
    except Exception as e:
        return {"error": f"{type(e).__name__}: {str(e)[:300]}"}


def run_ours(args):
    import torch.distributed as dist
    from yolo_master_b200 import ops
    from yolo_master_b200.nn.tasks import DetectionModel
    from yolo_master_b200.utils.synth import synth_images

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (the product path has no CPU fallback); use --impl reference for the CPU arm")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if args.kernel_priority:
        from yolo_master_b200 import _lib
        _lib.load().ym_set_kernel_priority(args.kernel_priority)     # read at launch (capture) time by every kernel but attention
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    pk = peaks()
    B = args.batch

    # ---- model: rank 0 owns the (synthetic) checkpoint, weights broadcast over NCCL/NVLink once at start-up
    model = DetectionModel("yolo26-master-n.yaml")
    if rank == 0:
        model.load_state_dict(synthetic_weights())
    model.to(dev).eval()
    from yolo_master_b200 import parallel
    parallel.broadcast_module_state(model, src=0)

    # ---- CPU baseline (rank 0, N==1): the unmodified reference (oracle/_ref) on a bounded sample of the same workload
    cpu_base = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        fwd, kind = reference_model("cpu", False)
        xs = synth_images(args.ref_images, IMG, IMG, 0)
        with torch.inference_mode():
            cores, host_cores = pick_cpu_threads(lambda: fwd(xs[:4]))
            t0 = time.perf_counter()
            reps = 0
            while reps < 1 or time.perf_counter() - t0 < 10.0:
                fwd(xs)
                reps += 1
            dt = time.perf_counter() - t0
        cpu_base = {"value": args.ref_images * reps / dt, "unit": UNIT, "cores": cores, "kind": kind,
                    "sample": f"{reps} x {args.ref_images} synthetic 640x640 images, fp32 PyTorch-CPU, "
                              + ("unmodified reference DetectionModel (oracle/_ref)" if kind == "reference" else "oracle port") +
                              f" ({dt:.1f} s), {cores} threads (fastest of 8/16/32/64/{host_cores} on this {host_cores}-core host)"}
        del fwd

    # ---- inputs: 4 rotating device batches (315 MB > 126 MB L2) + pinned host copies for the e2e leg
    nrot = 4
    dev_in = [synth_images(B, IMG, IMG, seed=100 + rank * 10 + i).half().to(dev) for i in range(nrot)]
    # e2e leg: uint8 RGB frames in pinned host memory, as the reference's predictor receives them (the /255 and the fp16
    # cast happen on the device, engine/predictor.py:164-176; here inside the stem kernel)
    host_in = [(synth_images(B, IMG, IMG, seed=200 + rank * 10 + i) * 255).round().to(torch.uint8).pin_memory() for i in range(3)]
    g = model.graphed(B, IMG, IMG, dtype=torch.float16)
    g8 = model.graphed(B, IMG, IMG, dtype=torch.uint8)
    kernels_per_step = g.kernels_per_replay

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    def timed(fn, steps, warmup):
        for i in range(warmup):
            fn(i)
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(steps):
            fn(i)
        e1.record()
        barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item())

    depth = max(1, args.streams)
    pipe = model.pipelined(B, IMG, IMG, dtype=torch.float16, depth=depth) if depth > 1 else None
    pipe8 = model.pipelined(B, IMG, IMG, dtype=torch.uint8, depth=depth) if depth > 1 else None

    def timed_pipe(steps, warmup):
        """K steps through PipelinedForward: `depth` graph instances on `depth` streams, batch i on instance i % depth; the events sit on
        the calling stream, which run_device joins to the instance streams on both sides."""
        pipe.run_device(dev_in[i % nrot] for i in range(warmup))
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        pipe.run_device(dev_in[i % nrot] for i in range(steps))
        e1.record()
        barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item())

    with ClockSampler(local) as clk:
        ms_single = timed(lambda i: g(dev_in[i % nrot]), args.steps, args.warmup)
        ms_dev = timed_pipe(args.steps, args.warmup) if depth > 1 else ms_single
    clocks = clk.summary()
    if args.dump_outputs and rank == 0:
        # the headline path's last step: batch steps - 1 ran on pipeline instance (steps - 1) % depth (or on the single graph)
        last = pipe.graphs[(args.steps - 1) % depth].static_out if depth > 1 else g.static_out
        dump_outputs(args.dump_outputs, {"detections": last})
    # e2e: K batches through the public pipelined host-buffer API; every step's H2D (uint8 frames) and D2H ((B,300,6) fp32)
    # are inside the timed region, on copy streams that overlap the neighbouring steps' compute
    def e2e_run(n):
        for out in (pipe8 if depth > 1 else g8).stream_host(host_in[i % 3] for i in range(n)):
            pass
    e2e_run(args.warmup)
    barrier()
    t0 = time.perf_counter()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    e2e_run(args.steps)
    e1.record()
    barrier()
    wall_ms = (time.perf_counter() - t0) * 1e3          # the last D2H lands on its own stream: wall clock covers it
    ms_e2e_t = torch.tensor([max(e0.elapsed_time(e1), wall_ms)], device=dev)
    if world > 1:
        dist.all_reduce(ms_e2e_t, op=dist.ReduceOp.MAX)
    ms_e2e = float(ms_e2e_t.item())
    ms_e2e_sync = timed(lambda i: g8.run_host(host_in[i % 3]), args.steps, args.warmup)   # unpipelined call, for reference

    value = world * B * args.steps / (ms_dev * 1e-3)
    pred_e2e = None
    if rank == 0 and world == 1:
        try:
            pred_e2e = time_predictor(model, g8, B, dev, args.steps, args.warmup)
        except Exception as e:      # a secondary figure must not take the contract line down
            pred_e2e = {"error": f"{type(e).__name__}: {str(e)[:200]}"}
    sweep = None
    if rank == 0 and world == 1 and args.depth_sweep:          # how throughput moves with the number of graph instances in flight
        sweep = {"1": world * B * args.steps / (ms_single * 1e-3), str(depth): value}
        for d3 in (2, 3, 4):
            if str(d3) in sweep:
                continue
            try:
                p3 = model.pipelined(B, IMG, IMG, dtype=torch.float16, depth=d3)
                p3.run_device(dev_in[i % nrot] for i in range(args.warmup))
                torch.cuda.synchronize(dev)
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                p3.run_device(dev_in[i % nrot] for i in range(args.steps))
                e1.record()
                torch.cuda.synchronize(dev)
                sweep[str(d3)] = B * args.steps / (e0.elapsed_time(e1) * 1e-3)
            except Exception as e:
                sweep[str(d3)] = f"{type(e).__name__}: {str(e)[:120]}"
    two = time_two_streams(model, dev_in, B, args.steps, args.warmup, dev) if (rank == 0 and args.two_stream) else None
    e2e = world * B * args.steps / (ms_e2e * 1e-3)
    roof = time_attention_kernel(dev, B, pk) if rank == 0 else None
    disp = time_dispatch(dev, pk) if rank == 0 else None
    if disp is not None:   # token sweep of the same microbench (SURVEY.md §8d: 4096 ... 262144 tokens): fixed launch / pipeline-fill cost vs size
        disp["sweep"] = []
        for nb in (4, 16, 64, 256):
            r = disp if nb == 64 else time_dispatch(dev, pk, B=nb, baseline=False)
            disp["sweep"].append({"tokens": nb * 1024, "ms": r["ms"], "algorithmic_gbs": r["algorithmic_gbs"], "hbm_frac": r["hbm_frac"]})
    eager = time_torch_eager_gpu(dev, B) if (rank == 0 and world == 1 and not args.no_cpu_baseline) else None

    if rank == 0:
        step_ms = ms_dev / args.steps
        out = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": step_ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f16",
            "data": "synthetic",
            "config": bench_config(world, B),
            "execution": (f"{depth} CUDA-graph instances of the whole bs{B} forward on {depth} streams, consecutive batches on consecutive "
                          "instances (PipelinedForward: same kernels and per-batch results as one graph; the exp-bound attention of one batch "
                          "overlaps the latency / HBM-bound layers of the other)") if depth > 1 else "CUDA graph of the whole forward",
            "single_stream": {"value": world * B * args.steps / (ms_single * 1e-3), "unit": UNIT, "ms_per_step": ms_single / args.steps,
                              "note": "one CUDA graph replayed back to back on one stream (the latency of one bs32 forward)"},
            "e2e": {"value": e2e, "unit": UNIT, "h2d_bytes_per_step": B * 3 * IMG * IMG, "d2h_bytes_per_step": B * 300 * 6 * 4,
                    "ms_per_step": ms_e2e / args.steps, "input": "uint8 RGB frames in pinned host memory (x/255 on the device)",
                    "api": ("PipelinedForward.stream_host" if depth > 1 else "GraphedForward.stream_host") + " (H2D / forward / D2H of neighbouring batches overlap)",
                    "unpipelined_ms_per_step": ms_e2e_sync / args.steps,
                    "unpipelined_value": world * B * args.steps / (ms_e2e_sync * 1e-3)},
            "e2e_predictor": pred_e2e,
            "gpu_launches": kernels_per_step * args.steps,
            "kernels_per_step": kernels_per_step,
            "clocks": clocks,
            "roofline": roof,
            "model_roofline": model_roofline(value / world, pk),
            "dispatch": disp,
            "two_stream": two,
            "depth_sweep_images_per_s": sweep,
            "torch_eager_gpu": eager,
            "cpu_baseline": cpu_base,
        }
        print(json.dumps(out))
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--batch", type=int, default=32)
    ap.add_argument("--ref-images", type=int, default=8, help="images per CPU-oracle step (bounded sample)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--two-stream", action="store_true", help="(legacy experiment leg) also time two raw graph replays on two streams")
    ap.add_argument("--kernel-priority", type=int, default=0,
                    help="launch priority (0 = off, -1 .. -8) of every kernel except the attention kernels (ym_set_kernel_priority)")
    ap.add_argument("--depth-sweep", action="store_true", help="also time PipelinedForward at depth 1 / 2 / 3 / 4")
    ap.add_argument("--streams", type=int, default=4, help="graph instances / streams of PipelinedForward (1 = a single graph)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the (B, 300, 6) detections of the last timed step to DIR/detections.npy (float32)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3)
    # stdout carries exactly ONE JSON line: libraries that print to the C-level stdout (NCCL prints "NCCL version ..." there on
    # init) are redirected to stderr for the duration of the run; the JSON goes to the saved descriptor.
    sys.stdout.flush()
    real_stdout = os.dup(1)
    os.dup2(2, 1)
    sys.stdout = os.fdopen(real_stdout, "w")
    try:
        if args.impl == "reference":
            run_reference(args)
        else:
            run_ours(args)
    finally:
        sys.stdout.flush()


if __name__ == "__main__":
    main()
