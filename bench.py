#!/usr/bin/env python
"""Headline benchmark: images/sec of DeepLabv3+ / Xception65 bf16 inference at 1025x2049, batch 8 per GPU
(BASELINE.json configs[1]) through the segb200 CUDA engine.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference]

One JSON line on stdout (rank 0).  Keys follow the driver contract; see DESIGN.md "Measurement".
  value        whole-job images/s with the input batch already resident in HBM (CUDA-graph replay);
  e2e          same metric through the public engine call with pinned HOST input (fp32 NCHW batch copied
               host->device inside the timed region) and the per-step result (uint8 argmax class maps,
               the tensor the reference's eval loop moves to the CPU, utils/score.py:108-110) read back;
  roofline     the dominant kernel (tcgen05 implicit-GEMM conv): algorithmic FLOPs of all its launches in
               one step / their CUDA-event time, against the measured sustained bf16 peak;
  cpu_baseline the oracle port (plain PyTorch fp32 restatement of the reference forward) on the host cores,
               one image of the same workload.
`--impl reference` times that CPU path alone (rank 0 only), one image per step.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOAD = "deeplabv3plus_xception65_bf16_infer_1025x2049_b8"
MODEL = "deeplabv3plus_xception65"
H, W, B, NCLASS = 1025, 2049, 8, 19
METRIC = "images/sec"


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm=d.get("hbm_gbs", 6650.0), tc=d.get("bf16_tflops_sustained", d.get("bf16_tflops", 1400.0)),
                    tc_burst=d.get("bf16_tflops", 1590.0), src="measured (MEASURED_PEAKS.json)")
    return dict(hbm=6650.0, tc=1400.0, tc_burst=1590.0, src="fallback (B200_PROFILING.md)")


class ClockSampler:
    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index=0):
        self.p = None
        try:
            self.p = subprocess.Popen(["nvidia-smi", "-i", str(index), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                       "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.p = None

    def stop(self):
        if self.p is None:
            return None
        self.p.terminate()
        try:
            out, _ = self.p.communicate(timeout=5)
        except Exception:
            self.p.kill()
            return None
        sm, mx, reasons = [], [], set()
        for line in out.strip().splitlines():
            f = [t.strip() for t in line.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1]))
            except ValueError:
                continue
            for name, v in zip(["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"], f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return None
        return dict(sm_mhz=statistics.median(sm), sm_max_mhz=max(mx), reasons=sorted(reasons), samples=len(sm))


def _cpu_reference_forward():
    """-> (forward(x) -> logits, kind, params): the reference's CPU implementation of the path.  The unmodified reference package
    staged under baseline/_ref when present ("reference"), else the oracle port ("port"); same weights either way."""
    import torch
    from oracle import segref as R
    P = R.build_params(MODEL, 0)
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    try:
        import ref_harness as H
        if H.available():
            model = H.build_model("cityscapes_deeplabv3_plus.yaml")
            model.load_state_dict(P.state_dict(), strict=True)

            def fwd(x):
                with torch.no_grad():
                    return model(x)[0]
            return fwd, "reference", P
    except Exception as e:                                   # noqa: BLE001
        print(f"[bench] staged reference unusable on the CPU ({type(e).__name__}: {e}); using the oracle port", file=sys.stderr)

    def fwd_port(x):
        with torch.no_grad():
            return R.forward(MODEL, P, x)
    return fwd_port, "port", P


def _time_cpu(fwd, x):
    t = time.perf_counter()
    fwd(x)
    return time.perf_counter() - t


def _pick_threads_fn(fwd, x):
    import torch
    ncpu = os.cpu_count() or 1
    cands = sorted({c for c in (ncpu, ncpu // 2, 32, 16) if 1 <= c <= ncpu})
    probe = x[:, :, :257, :513]
    best, best_t = cands[-1], None
    for c in cands:
        torch.set_num_threads(c)
        _time_cpu(fwd, probe)
        t = min(_time_cpu(fwd, probe) for _ in range(2))
        if best_t is None or t < best_t:
            best, best_t = c, t
    torch.set_num_threads(best)
    return best


def run_reference(args):
    """--impl reference: the reference's own CPU implementation of the path on the box's host cores, rank 0 only: the unmodified
    reference package (baseline/_ref, `get_segmentation_model()`) when it is staged, else the oracle port."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import torch
    fwd, kind, _ = _cpu_reference_forward()
    x = torch.randn(1, 3, H, W, generator=torch.Generator().manual_seed(1024))
    cores = _pick_threads_fn(fwd, x)
    for _ in range(args.warmup):
        _time_cpu(fwd, x)
    t = 0.0
    for _ in range(args.steps):
        t += _time_cpu(fwd, x)
    val = args.steps / t
    what = "the reference package (baseline/_ref)" if kind == "reference" else "the CPU oracle port of the reference forward"
    sample = f"1 image (1x3x{H}x{W} fp32) per step, {args.steps} steps, torch CPU {torch.get_num_threads()} threads, {what}"
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": val, "unit": "images/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * t / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": WORKLOAD, "note": f"{what} on the host cores; one image per step"},
        "cpu_baseline": {"value": val, "unit": "images/s", "cores": cores, "kind": kind, "sample": sample},
        "e2e": {"value": val, "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }), flush=True)


def _time_forward(fn, iters=5, warm=3):
    import torch
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters


def cudnn_reference(P, x_dev, eng, bsz):
    """The north-star denominator, measured in the same process on the same GPU: the reference's OWN model
    (`get_segmentation_model()` from the unmodified copy under baseline/_ref, segmentron/models/model_zoo.py:17-24) with the same
    weights, `.to(bf16)`, eval, cudnn.benchmark on (utils/default_setup.py:18), NCHW and channels_last -- the faster layout counts.
    Falls back to the oracle port (the same torch ops) only when baseline/_ref is absent.  Also reports the parity the north-star
    states: this engine's bf16 logits vs the reference's own cuDNN bf16 logits, both against the reference's fp32 forward."""
    import torch
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    import ref_harness as H
    torch.backends.cudnn.benchmark = True
    res, kind, parity = {}, "port", None
    with torch.no_grad():
        if H.available():
            kind = "reference"
            model = H.build_model("cityscapes_deeplabv3_plus.yaml")
            model.load_state_dict(P.state_dict(), strict=True)
            m32 = model.cuda()
            x1 = x_dev[:1]
            tf = (torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32)
            torch.backends.cudnn.allow_tf32 = torch.backends.cuda.matmul.allow_tf32 = False
            y32 = m32(x1)[0].float()                                      # the reference's fp32 forward of image 0 (TF32 off)
            torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = tf
            mb = m32.to(torch.bfloat16)
            xb = x_dev.to(torch.bfloat16)
            yb = mb(xb[:1])[0].float()
            yo = eng(x1).float()                                          # this engine, bf16, same image (batch-invariant)

            def rel(a, b):
                return float((a - b).norm() / b.norm())
            am32 = y32.argmax(1)
            parity = {"image": "image 0 of the bench batch, 1x3x%dx%d" % tuple(x1.shape[2:]),
                      "ours_bf16_vs_ref_fp32_rel_l2": rel(yo, y32), "ref_cudnn_bf16_vs_ref_fp32_rel_l2": rel(yb, y32),
                      "ours_bf16_vs_ref_cudnn_bf16_rel_l2": rel(yo, yb),
                      "argmax_mismatch_ours_vs_ref_fp32": int((yo.argmax(1) != am32).sum()),
                      "argmax_mismatch_refbf16_vs_ref_fp32": int((yb.argmax(1) != am32).sum()),
                      "argmax_mismatch_ours_vs_refbf16": int((yo.argmax(1) != yb.argmax(1)).sum()), "pixels": int(am32.numel())}
            del y32, yb, yo
            res["nchw"] = bsz / (_time_forward(lambda: mb(xb)) * 1e-3)
            mcl = mb.to(memory_format=torch.channels_last)
            xcl = xb.contiguous(memory_format=torch.channels_last)
            res["channels_last"] = bsz / (_time_forward(lambda: mcl(xcl)) * 1e-3)
            del model, m32, mb, mcl, xb, xcl
        else:
            from oracle import segref as R
            for fmt in ("nchw", "channels_last"):
                Pg = P.to("cuda", torch.bfloat16)
                xb = x_dev.to(torch.bfloat16)
                if fmt == "channels_last":
                    xb = xb.contiguous(memory_format=torch.channels_last)
                    for k, v in Pg.t.items():
                        if v.dim() == 4:
                            Pg.t[k] = v.contiguous(memory_format=torch.channels_last)
                res[fmt] = bsz / (_time_forward(lambda: R.forward(MODEL, Pg, xb)) * 1e-3)
                del Pg, xb
    torch.cuda.empty_cache()
    return {"value": max(res.values()), "unit": "images/s", "by_layout": res, "kind": kind, "parity": parity,
            "what": ("the reference's own model (baseline/_ref, get_segmentation_model) " if kind == "reference" else
                     "oracle port (same torch ops as the reference) ") + "on this GPU, bf16 eager, cudnn.benchmark on; faster layout"}


def train_subrecord(args, rank, world, parallel):
    """BASELINE.json configs[2], the one path with a data-path collective: DeepLabv3+/ResNet101 bf16 training at 1025x2049,
    per-GPU batch 4 (weak scaling), SyncBatchNorm + bucketed NCCL gradient all-reduce overlapped with backward.  A step =
    trainer.step(images, targets) = forward + CrossEntropy(ignore -1) + backward + SGD; CUDA events, barrier on both sides, max over
    ranks.  Every rank must call this."""
    import torch
    from oracle import segref as R
    from segmentron_b200.train import DeepLabV3PlusTrainerB200
    model = "deeplabv3plus_resnet101"
    P = R.build_params(model, 0)
    shape = (4, 3, H, W)
    g = torch.Generator().manual_seed(2048 + rank)
    x = torch.randn(*shape, generator=g).cuda()
    target = torch.randint(-1, 19, (shape[0], shape[2], shape[3]), generator=g).cuda()
    tr = DeepLabV3PlusTrainerB200(P.state_dict(), backbone="resnet101", dtype=torch.bfloat16, lr=0.02, sync_bn=True)
    losses = [float(tr.step(x, target)) for _ in range(3)]
    parallel.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.train_steps):
        tr.step(x, target)
    e1.record()
    torch.cuda.synchronize()
    ms = parallel.max_over_ranks(e0.elapsed_time(e1)) / args.train_steps
    parallel.barrier()
    st = tr.plan_for(shape)
    rec = {"workload": "deeplabv3plus_resnet101_bf16_train_1025x2049_b4_per_gpu", "metric": "images/sec", "n_gpus": world,
           "value": world * shape[0] / (ms * 1e-3), "ms_per_step": ms, "steps": args.train_steps, "scaling": "weak",
           "sync_bn": world > 1, "allreduce_buckets": len(st["buckets"]) if world > 1 else 0,
           "collectives_per_step": tr.collectives_per_step(shape) if hasattr(tr, "collectives_per_step") else None,
           "launches_per_step": tr.n_launches(shape), "loss_first_steps": [round(v, 4) for v in losses],
           "grad_dtype": str(getattr(tr, "grad_comm_dtype", torch.float32)).replace("torch.", "")}
    del tr, x, target
    torch.cuda.empty_cache()
    return rec


DUMP_PIXELS = 1 << 19          # 19 float32 logits + 1 class per pixel: 42 MB


def dump_outputs(out_dir, logits, amax):
    """The forward's outputs at the same DUMP_PIXELS pixels of every run with the same batch shape (torch.randperm seeded with 0,
    in flat (image, row, column) order): logits.npy [DUMP_PIXELS, nclass] and argmax.npy [DUMP_PIXELS], both float32."""
    import numpy as np
    import torch
    n, c, h, w = logits.shape
    idx = torch.randperm(n * h * w, generator=torch.Generator().manual_seed(0))[:DUMP_PIXELS].sort().values.to(logits.device)
    img, pix = idx // (h * w), idx % (h * w)
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "logits.npy"), logits.view(n, c, h * w)[img, :, pix].float().cpu().numpy())
    np.save(os.path.join(out_dir, "argmax.npy"), amax.view(n, h * w)[img, pix].float().cpu().numpy())


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="segb200", choices=["segb200", "reference"])
    ap.add_argument("--batch", type=int, default=B)
    ap.add_argument("--height", type=int, default=H)
    ap.add_argument("--width", type=int, default=W)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--cudnn-ref", action="store_true", help="(default on; kept for compatibility)")
    ap.add_argument("--no-cudnn-ref", action="store_true", help="skip timing the reference's own cuDNN bf16 forward on this GPU")
    ap.add_argument("--no-train", action="store_true", help="skip the config-3 training sub-record (the path with a collective)")
    ap.add_argument("--train-steps", type=int, default=8)
    ap.add_argument("--dump-kernels", default=None, help="write the per-launch timing table to this file")
    ap.add_argument("--no-graph", action="store_true", help="replay the launch list directly instead of one CUDA graph (for profilers)")
    ap.add_argument("--dump-outputs", default=None, metavar="DIR",
                    help="write what the last timed step returned to DIR/*.npy (float32): the logits and the argmax class of a fixed, "
                         "seeded sample of pixels")
    args = ap.parse_args()
    args.warmup = max(args.warmup, 3)
    if args.impl == "reference":
        return run_reference(args)

    import torch
    import __graft_entry__ as ge
    ge.build()
    from segmentron_b200.engine import DeepLabV3PlusB200

    from segmentron_b200 import parallel
    if not torch.cuda.is_available():
        raise RuntimeError("bench.py needs a CUDA device (the engine has no CPU fallback)")
    torch.cuda.set_device(int(os.environ.get("LOCAL_RANK", "0")))
    rank, world, local = parallel.init_from_env("nccl")
    dist = None
    if world > 1:
        import torch.distributed as dist
    bsz, hh, ww = args.batch, args.height, args.width

    # ---- synthetic weights (reference architecture, seeded; BN stats randomised) and inputs --------------
    # The parameter dict uses the reference's state_dict names; generating it needs only torch (seeded CPU RNG).
    from oracle import segref as R      # parameter generator + cpu_baseline only; never on the timed GPU path
    P = R.build_params(MODEL, 0)
    eng = DeepLabV3PlusB200(P.state_dict(), backbone="xception65", nclass=NCLASS, eps_encoder=1e-3, dtype=torch.bfloat16,
                            cuda_graph=not args.no_graph, want_argmax=True)
    g = torch.Generator().manual_seed(1024 + rank)
    x_host = torch.randn(bsz, 3, hh, ww, generator=g).pin_memory()
    x_dev = x_host.cuda(non_blocking=True)
    st = eng.plan_for(x_dev)
    plan = st["plan"]
    st["holder"]["x"].copy_(x_dev)
    amax_host = torch.empty(bsz, hh, ww, dtype=torch.uint8).pin_memory()
    torch.cuda.synchronize()

    barrier = parallel.barrier

    def timed(step_fn, k, finish=None):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(k):
            step_fn(i)
        if finish is not None:
            finish()
        e1.record()
        torch.cuda.synchronize()
        ms = parallel.max_over_ranks(e0.elapsed_time(e1))
        barrier()
        return ms

    # ---- kernel-only throughput: input resident in HBM, one CUDA-graph replay per step -------------------
    graph = st["graph"]
    if graph is None:                                   # --no-graph: same launch list, launched one by one
        class _Direct:
            def replay(self_):
                plan.run()
        graph = _Direct()
    for _ in range(args.warmup):
        graph.replay()
    sampler = ClockSampler(local) if rank == 0 else None
    ms = timed(lambda i: graph.replay(), args.steps)
    clocks = sampler.stop() if sampler else None
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, st["out"], st["amax"])
    value = world * bsz * args.steps / (ms * 1e-3)

    # ---- end to end: pinned host batch -> H2D -> engine -> argmax class maps -> D2H, every step -----------------
    # Public call path with HOST buffers.  Every step copies ITS OWN input batch host->device and reads ITS result back
    # inside the timed region; the H2D of step i+1 runs on a copy stream while step i computes (double-buffered staging),
    # the D2H of step i on a third stream -- a user-side pipeline, no work is skipped.
    cur = torch.cuda.current_stream()
    s_in, s_out = torch.cuda.Stream(), torch.cuda.Stream()
    stage = [torch.empty_like(st["holder"]["x"]) for _ in range(2)]
    ev_in = [torch.cuda.Event() for _ in range(2)]
    ev_free = [torch.cuda.Event() for _ in range(2)]
    ev_done, ev_read = torch.cuda.Event(), torch.cuda.Event()
    amax_dev = torch.empty_like(st["amax"])

    def h2d(i):
        with torch.cuda.stream(s_in):
            s_in.wait_event(ev_free[i & 1])              # the engine has consumed what was staged here two steps ago
            stage[i & 1].copy_(x_host, non_blocking=True)
            ev_in[i & 1].record(s_in)

    def e2e_step(i):
        if i == 0:
            h2d(0)
        if i + 1 < e2e_total["k"]:
            h2d(i + 1)                                   # prefetch the next step's batch while this one computes
        cur.wait_event(ev_in[i & 1])
        st["holder"]["x"].copy_(stage[i & 1], non_blocking=True)
        ev_free[i & 1].record(cur)
        graph.replay()
        cur.wait_event(ev_read)                          # previous result has left amax_dev (its D2H overlapped this step's compute)
        amax_dev.copy_(st["amax"], non_blocking=True)
        ev_done.record(cur)
        with torch.cuda.stream(s_out):
            s_out.wait_event(ev_done)
            amax_host.copy_(amax_dev, non_blocking=True)
            ev_read.record(s_out)

    def e2e_finish():
        cur.wait_stream(s_out)
        cur.wait_stream(s_in)

    e2e_total = {"k": 2}
    for i in range(2):
        ev_free[i].record(cur)
    ev_read.record(cur)
    for i in range(2):
        e2e_step(i)
    e2e_finish()
    torch.cuda.synchronize()
    for i in range(2):
        ev_free[i].record(cur)
    e2e_total["k"] = args.steps
    ms_e2e = timed(e2e_step, args.steps, e2e_finish)
    e2e_val = world * bsz * args.steps / (ms_e2e * 1e-3)

    # ---- the same pipeline returning what forward()[0] returns: the bf16 logits [B,19,H,W] (0.64 GB per step over PCIe) ----
    logits_host = torch.empty(st["out"].shape, dtype=st["out"].dtype).pin_memory()
    logits_dev = torch.empty_like(st["out"])

    def e2e_logits_step(i):
        if i == 0:
            h2d(0)
        if i + 1 < e2e_total["k"]:
            h2d(i + 1)
        cur.wait_event(ev_in[i & 1])
        st["holder"]["x"].copy_(stage[i & 1], non_blocking=True)
        ev_free[i & 1].record(cur)
        graph.replay()
        cur.wait_event(ev_read)                          # the previous step's logits have left logits_dev: their 0.64 GB D2H ran under this step
        logits_dev.copy_(st["out"], non_blocking=True)
        ev_done.record(cur)
        with torch.cuda.stream(s_out):
            s_out.wait_event(ev_done)
            logits_host.copy_(logits_dev, non_blocking=True)
            ev_read.record(s_out)

    k_log = max(3, args.steps // 2)
    e2e_total["k"] = k_log
    for i in range(2):
        ev_free[i].record(cur)
    ev_read.record(cur)
    ms_e2e_logits = timed(e2e_logits_step, k_log, e2e_finish)
    e2e_logits_val = world * bsz * k_log / (ms_e2e_logits * 1e-3)
    d2h_logits = logits_host.numel() * logits_host.element_size()
    del logits_host, logits_dev

    train = None
    if not args.no_train and (bsz, hh, ww) == (B, H, W):
        train = train_subrecord(args, rank, world, parallel)

    out = None
    if rank == 0:
        pk = peaks()
        # ---- per-kernel timing (direct launches, CUDA events on the launching stream) -------------------
        plan.run_timed()
        rows = plan.run_timed()
        agg = {}
        for m, t in rows:
            a = agg.setdefault(m["kind"], dict(ms=0.0, flops=0.0, bytes=0.0, n=0))
            a["ms"] += t; a["flops"] += m["flops"]; a["bytes"] += m["bytes"]; a["n"] += 1
        tot_ms = sum(a["ms"] for a in agg.values())
        cg = agg["conv_gemm"]
        # dominant kernel = conv_gemm; dominant SHAPE = the layer shape with the largest summed time (50 of the 79
        # launches are the middle-flow 728->728 GEMM).  `traffic` comes from the committed ncu capture of that shape.
        shapes = {}
        for m, t in rows:
            if m["kind"] == "conv_gemm":
                s_ = shapes.setdefault(m["desc"], dict(ms=0.0, flops=0.0, bytes=0.0, n=0))
                s_["ms"] += t; s_["flops"] += m["flops"]; s_["bytes"] += m["bytes"]; s_["n"] += 1
        top_desc, top = max(shapes.items(), key=lambda kv: kv[1]["ms"])
        ach = top["flops"] / (top["ms"] * 1e-3) / 1e12
        traffic = None
        tj = os.path.join(ROOT, "profiles", "traffic.json")
        if os.path.exists(tj):
            traffic = json.load(open(tj)).get(top_desc)
            if isinstance(traffic, dict):
                traffic = traffic.get("dram_bytes_per_launch")
        roofline = {"kernel": "conv_gemm_kernel<bf16> (tcgen05 implicit GEMM)", "shape": top_desc, "bound": "tensor",
                    "achieved": ach, "peak": pk["tc"], "unit": "TFLOP/s", "frac": ach / pk["tc"], "traffic": traffic,
                    "algorithmic_flop_per_launch": top["flops"] / top["n"], "algorithmic_bytes_per_launch": top["bytes"] / top["n"],
                    "avg_launch_ms": top["ms"] / top["n"], "launches_per_step": top["n"], "share_of_step": top["ms"] / tot_ms,
                    "peak_source": pk["src"] + ", sustained bf16"}
        ach_all = cg["flops"] / (cg["ms"] * 1e-3) / 1e12
        roofline_all = {"kernel": "conv_gemm_kernel<bf16>, all 79 launches of a step", "bound": "tensor", "achieved": ach_all,
                        "peak": pk["tc"], "unit": "TFLOP/s", "frac": ach_all / pk["tc"], "launches_per_step": cg["n"],
                        "share_of_step": cg["ms"] / tot_ms}
        dw = agg.get("dwconv3x3")
        roofline_dw = None
        if dw:
            a2 = dw["bytes"] / (dw["ms"] * 1e-3) / 1e9
            roofline_dw = {"kernel": "dwconv3x3_kernel<bf16>", "bound": "hbm", "achieved": a2, "peak": pk["hbm"], "unit": "GB/s",
                           "frac": a2 / pk["hbm"], "traffic": None, "launches_per_step": dw["n"], "share_of_step": dw["ms"] / tot_ms}
        if args.dump_kernels:
            with open(args.dump_kernels, "w") as f:
                f.write("kind\tms\tGFLOP\tMB\tTFLOP/s\tGB/s\tdesc\n")
                for m, t in rows:
                    f.write(f"{m['kind']}\t{t:.4f}\t{m['flops'] / 1e9:.2f}\t{m['bytes'] / 1e6:.1f}\t"
                            f"{m['flops'] / max(t, 1e-6) / 1e9:.1f}\t{m['bytes'] / max(t, 1e-6) / 1e6:.0f}\t{m['desc']}\n")
                f.write("\n# per kind: " + json.dumps({k: dict(ms=round(v["ms"], 3), n=v["n"]) for k, v in agg.items()}) + "\n")
        # ---- CPU baseline: oracle port, one image of the same workload ----------------------------------
        cpu = None
        if not args.no_cpu_baseline:
            xc = x_host[:1].clone()
            cfwd, ckind, _ = _cpu_reference_forward()
            cores = _pick_threads_fn(cfwd, xc)
            t = _time_cpu(cfwd, xc)
            cpu = {"value": 1.0 / t, "unit": "images/s", "cores": cores, "kind": ckind,
                   "sample": f"1 image 1x3x{hh}x{ww} fp32, 1 forward of "
                             f"{'the reference package (baseline/_ref)' if ckind == 'reference' else 'the oracle port'}, {torch.get_num_threads()} threads"}
        cudnn = None
        if not args.no_cudnn_ref:
            cudnn = cudnn_reference(P, x_dev, eng, bsz)
        h2d = x_host.numel() * x_host.element_size()
        d2h = amax_host.numel()
        out = {
            "metric": METRIC, "value": value, "unit": "images/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16",
            "data": "synthetic",
            "config": {"workload": WORKLOAD if (bsz, hh, ww) == (B, H, W) else f"deeplabv3plus_xception65_bf16_infer_{hh}x{ww}_b{bsz}",
                       "per_gpu_batch": bsz, "global_batch": bsz * world, "parallelism": f"replicas x{world} (no data-path collective)",
                       "l2": "activations ~15 GB/step >> 126 MB L2 (inputs larger than L2, no flush needed)",
                       "weights": "reference architecture, seeded random init, BN stats randomised"},
            "e2e": {"value": e2e_val, "unit": "images/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "ms_per_step": ms_e2e / args.steps, "input": "pinned fp32 NCHW batch, H2D of step i+1 overlapped with step i",
                    "result": "uint8 argmax class maps"},
            "e2e_logits": {"value": e2e_logits_val, "unit": "images/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h_logits,
                           "ms_per_step": ms_e2e_logits / k_log, "steps": k_log,
                           "result": "bf16 logits [B,19,H,W], what forward()[0] returns (0.64 GB per step over PCIe, overlapped with the next step's compute)"},
            "gpu_launches": plan.n_launch * args.steps, "launches_per_step": plan.n_launch,
            "roofline": roofline, "roofline_all_gemm": roofline_all, "roofline_dw": roofline_dw, "cpu_baseline": cpu, "clocks": clocks,
            "per_kind_ms": {k: round(v["ms"], 3) for k, v in agg.items()},
        }
        if cudnn:
            out["cudnn_ref"] = cudnn
            out["vs_cudnn_ref"] = {"device_resident": value / world / cudnn["value"], "e2e": e2e_val / world / cudnn["value"],
                                   "note": "per-GPU images/s of this engine / the reference's cuDNN bf16 forward on the same GPU"}
        if train:
            out["train"] = train
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()
    if out is not None:
        print(json.dumps(out), flush=True)


if __name__ == "__main__":
    main()
