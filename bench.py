#!/usr/bin/env python
"""Benchmark of the FlowNet2 forward hot path (BASELINE.json metric: frame-pairs/s, FlowNet2 forward
@1024x436; correlation-layer HBM GB/s).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

ours:       one process per GPU; full FlowNet2 (CSS + SD + fusion) deploy net through the Caffe-surface
            engine (fn2_net_* C-ABI), B pairs per GPU (weak scaling: config 4 = 32 pairs over 8 GPUs).
            Weights are filled on rank 0 and sent with ONE NCCL broadcast of the parameter arena; every step
            ends with a gather of the flow fields to rank 0.  `value` times K steps with inputs resident in
            HBM; `e2e` times the same K steps with pinned-host inputs (H2D inside) and the flows read back
            to the host (D2H inside).  --dump-outputs DIR: rank 0 writes the flow fields of the last timed step as
            DIR/predict_flow_final.npy; weights and inputs are seeded, so two builds can be compared output for output.
reference:  the reference's own CPU forward on all host cores, ONE WHOLE 1024x436 pair per step (fixed workload, no
            scaling): oracle/_ref (the reference's layer sources compiled unmodified) runs conv/deconv (im2col +
            OpenBLAS sgemm), ReLU, Eltwise, Concat, FlowWarp, ChannelNorm; Correlation / Resample / DataAugmentation
            have no CPU implementation in the reference (NOT_IMPLEMENTED / LOG(FATAL)) and run the oracle port.
            Without oracle/_ref/libref_caffe.so the oracle port runs everything on a FIXED 256x128 tile.
Prints exactly one JSON line on rank 0.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

METRIC = "frame-pairs/sec FlowNet2 forward @1024x436"
UNIT = "frame-pairs/s"


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--model", default="FlowNet2")
    ap.add_argument("--width", type=int, default=1024)
    ap.add_argument("--height", type=int, default=436)
    ap.add_argument("--batch", type=int, default=4, help="frame pairs per GPU")
    ap.add_argument("--cpu-seconds", type=float, default=20.0, help="budget of the cpu_baseline sample")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extra", action="store_true", help="skip the config 2 / config 3 / 448x320 / config 5 side measurements")
    ap.add_argument("--config5-only", action="store_true", help="print only the config 5 (FlowNet2-C training step) measurement")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step computed as DIR/<name>.npy (float32)")
    a = ap.parse_args()
    if a.dump_outputs and (a.impl != "ours" or a.config5_only):
        ap.error("--dump-outputs writes the outputs of the forward path of --impl ours only")
    return a


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return {"hbm_gbs": d["hbm_gbs"], "bf16_tflops": d["bf16_tflops"], "bf16_tflops_sustained": d.get("bf16_tflops_sustained"),
                "source": "measured (MEASURED_PEAKS.json)"}
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "source": "fallback (B200_PROFILING.md)"}


DUMP_BYTES = 64 * 10 ** 6


def write_outputs(d, arrays):
    """--dump-outputs: every array as d/<name>.npy, float32, DUMP_BYTES in all.  An array larger than its share is replaced by a
    fixed, seeded sample of its flattened elements (in index order), the same sample for the same shape on every run."""
    os.makedirs(d, exist_ok=True)
    share = DUMP_BYTES // len(arrays) - 4096                  # room for the .npy header
    for name, a in arrays.items():
        a = np.ascontiguousarray(a, np.float32)
        if a.nbytes > share:
            a = a.reshape(-1)[np.sort(np.random.default_rng(0).choice(a.size, share // 4, replace=False))]
        np.save(os.path.join(d, name + ".npy"), a)


def config(args, n_gpus):
    return {"workload": "%s deploy forward, %dx%d synthetic pairs (adapted to /64), fp32" % (args.model, args.width, args.height),
            "model": args.model, "width": args.width, "height": args.height, "pairs_per_gpu": args.batch,
            "global_batch": args.batch * n_gpus, "parallelism": "frame-batch sharding x%d (1 NCCL weight broadcast, flow gather)" % n_gpus,
            "l2": "working set (weights ~650 MB + activations) exceeds the 126 MB L2; no explicit flush",
            "cpu_arm": cpu_arm_description(args)}


# ----------------------------------------------------------------------------------------------------------
# CPU arm: used for cpu_baseline (N=1, rank 0) and for --impl reference.  The workload is FIXED (never picked from a
# calibration run): one whole pair of the bench size through the reference's CPU layers, or -- only when oracle/_ref is
# not built -- one 256x128 tile through the oracle port, scaled by the pixel ratio.
# ----------------------------------------------------------------------------------------------------------
FALLBACK_TILE = (256, 128)


def cpu_arm_description(args):
    """The fixed workload of the CPU legs (--impl reference, cpu_baseline); part of `config` on both arms."""
    from oracle import ref as R
    if R.available():
        return ("one whole %dx%d pair per step, all host cores: reference CPU layers (oracle/_ref: im2col + OpenBLAS sgemm conv/deconv, "
                "ReLU, Eltwise, Concat, FlowWarp, ChannelNorm) + oracle port for Correlation/Resample/DataAugmentation "
                "(no CPU implementation in the reference)" % (args.width, args.height))
    return "one fixed %dx%d tile of a %dx%d pair per step (oracle port, OpenMP), scaled by the pixel ratio" % (
        FALLBACK_TILE + (args.width, args.height))


class CpuArm(object):
    def __init__(self, args):
        import flownet2_b200 as F
        from oracle import ref as R
        self.args = args
        r = np.random.default_rng(3)
        if R.available():
            self.kind, self.w, self.h, self.scale = "reference", args.width, args.height, 1.0
            proto = F.fill_template(F.model_template(args.model), self.w, self.h)
            self.net = R.RefCpuNet(proto, None, batch=1, synth_seed=1701)
            self.cores = os.cpu_count()
            self.sample = cpu_arm_description(args)
        else:
            from oracle.net import OracleNet
            self.kind, (self.w, self.h) = "port", FALLBACK_TILE
            self.scale = (self.w * self.h) / float(args.width * args.height)
            proto = F.fill_template(F.model_template(args.model), self.w, self.h)
            self.net = OracleNet(proto, None, batch=1, synth_seed=1701)
            self.cores = os.cpu_count()
            self.sample = cpu_arm_description(args)
        self.a = np.round(r.uniform(0, 255, (1, 3, self.h, self.w))).astype(np.float32)
        self.b = np.clip(self.a + np.round(r.normal(0, 3, self.a.shape)), 0, 255).astype(np.float32)

    def step(self):
        t0 = time.perf_counter()
        self.net.forward(img0=self.a, img1=self.b)
        return time.perf_counter() - t0

    def run(self, steps, warmup):
        for _ in range(warmup):
            self.step()
        times = [self.step() for _ in range(steps)]
        mean = float(np.mean(times))
        return self.scale / mean, mean


def reference_gpu_arm(args, batch, steps=5, warmup=2):
    """The reference's OWN GPU path (its unmodified layer classes from oracle/_ref: im2col + cuBLAS convolutions, its correlation /
    warp / resample kernels) on the same workload and the same B200 (tools/ref_forward_time.py).  A reported baseline like
    cpu_baseline, N = 1 only; None when oracle/_ref is not built.  Runs as a subprocess: a CHECK failure inside the reference aborts
    its process and must never take the bench line down."""
    try:
        from oracle import ref as R
        if not R.available():
            return None
        pr = subprocess.run([sys.executable, os.path.join(ROOT, "tools", "ref_forward_time.py"), args.model, str(args.width), str(args.height),
                             str(batch), str(steps), str(warmup)], capture_output=True, text=True, timeout=600)
        last = [l for l in pr.stdout.strip().splitlines() if l.startswith("{")]
        return json.loads(last[-1]) if last else {"unavailable": "exit %d: %s" % (pr.returncode, pr.stderr.strip()[-300:])}
    except Exception as e:
        return {"unavailable": "%s: %s" % (type(e).__name__, e)}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    arm = CpuArm(args)
    value, mean = arm.run(args.steps, args.warmup)
    cfg = config(args, args.gpus)
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": mean * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic", "config": cfg,
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": arm.cores, "kind": arm.kind, "sample": arm.sample},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


def profile_traffic(pattern):
    """dram__bytes_read.sum + dram__bytes_write.sum (bytes) of the single launch in the newest committed
    profiles/*<pattern>*_raw.csv (`ncu --set full --csv --page raw`; row 1 = units, row 2 = values), or (None, None)."""
    import csv
    import glob
    files = sorted(glob.glob(os.path.join(ROOT, "profiles", "r[0-9][0-9]_%s_raw.csv" % pattern)))
    if not files:
        return None, None
    path = files[-1]
    try:
        rows = list(csv.reader(open(path)))
        head, units, vals = rows[0], rows[1], rows[2]
        mult = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}
        total = 0.0
        for name in ("dram__bytes_read.sum", "dram__bytes_write.sum"):
            i = head.index(name)
            total += float(vals[i]) * mult[units[i]]
        return total, os.path.relpath(path, ROOT)
    except Exception:
        return None, os.path.relpath(path, ROOT)


def profile_metric(pattern, metric):
    """Value of `metric` for the (first) launch in the newest committed profiles/rNN_<pattern>.csv written by
    `ncu --metrics ... --csv` (one row per launch and metric), or (None, None)."""
    import csv
    import glob
    files = sorted(glob.glob(os.path.join(ROOT, "profiles", "r[0-9][0-9]_%s.csv" % pattern)))
    if not files:
        return None, None
    try:
        for r in csv.reader(open(files[-1])):
            if len(r) > 3 and r[-3] == metric:
                return float(r[-1].replace(",", "")), os.path.relpath(files[-1], ROOT)
    except Exception:
        pass
    return None, os.path.relpath(files[-1], ROOT)


# ----------------------------------------------------------------------------------------------------------
# GPU arm
# ----------------------------------------------------------------------------------------------------------
def clocks_sampler_start(dev_index):
    q = "timestamp,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
    try:
        return subprocess.Popen(["nvidia-smi", "-i", str(dev_index), "--query-gpu=" + q, "--format=csv,noheader,nounits", "-lms", "20"],
                                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
    except Exception:
        return None


def clocks_sampler_stop(p, t0=None, t1=None):
    """Samples are taken every 20 ms from before the warm-up on (nvidia-smi needs ~0.1 s to start); only those whose
    timestamp lies inside the timed region [t0, t1] (host clock) are used."""
    if p is None:
        return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
    p.terminate()
    try:
        out, _ = p.communicate(timeout=5)
    except Exception:
        p.kill()
        out = ""
    import datetime
    rows = []
    names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
    for line in out.strip().splitlines():
        f = [x.strip() for x in line.split(",")]
        if len(f) < 8:
            continue
        try:
            ts = datetime.datetime.strptime(f[0], "%Y/%m/%d %H:%M:%S.%f").timestamp()
            rows.append((ts, float(f[1]), float(f[2]), [nm for nm, v in zip(names, f[4:8]) if v.lower().startswith("active")]))
        except ValueError:
            continue
    inside = [r for r in rows if t0 is not None and t0 - 0.01 <= r[0] <= t1 + 0.01]
    use = inside if inside else rows[-3:]
    sm = [r[1] for r in use]; mx = [r[2] for r in use]
    reasons = set(x for r in use for x in r[3])
    if not sm:
        return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
    # median over the samples taken under load (upper half)
    sm_sorted = sorted(sm)
    load = sm_sorted[len(sm_sorted) // 2:]
    return {"sm_mhz": float(np.median(load)), "sm_max_mhz": float(max(mx)), "reasons": sorted(reasons), "samples": len(sm),
            "samples_in_timed_region": len(inside)}


def measure_tf32_peak(torch):
    """Dense TF32 tensor-core peak of this GPU: cuBLAS GEMM 8192^3 with TF32 allowed, best of 10 (a roofline denominator,
    measured outside every timed region)."""
    try:
        old = torch.backends.cuda.matmul.allow_tf32
        torch.backends.cuda.matmul.allow_tf32 = True
        a = torch.randn(8192, 8192, device="cuda")
        b = torch.randn(8192, 8192, device="cuda")
        best = 1e9
        for _ in range(3):
            torch.matmul(a, b)
        for _ in range(10):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            torch.matmul(a, b)
            e1.record()
            torch.cuda.synchronize()
            best = min(best, e0.elapsed_time(e1))
        torch.backends.cuda.matmul.allow_tf32 = old
        return 2.0 * 8192 ** 3 / (best * 1e-3) / 1e12
    except Exception:
        return None


def side_config(torch, F, model, w, h, batch, steps=10, warmup=3):
    """Device-resident throughput of another BASELINE.json configuration (same engine, same step definition), N=1."""
    proto = F.fill_template(F.model_template(model), w, h)
    net = F.Net(proto, None, F.TEST, batch=batch)
    net.fill_params(1701)
    r = np.random.default_rng(7)
    img0 = np.round(r.uniform(0, 255, (batch, 3, h, w))).astype(np.float32)
    img1 = np.clip(img0 + np.round(r.normal(0, 4, img0.shape)), 0, 255).astype(np.float32)
    d0, d1 = torch.from_numpy(img0).cuda(), torch.from_numpy(img1).cuda()
    out = torch.empty((batch, 2, h, w), device="cuda")
    stream = torch.cuda.ExternalStream(net.stream)
    with torch.cuda.stream(stream):
        def step():
            net.set_input_device("img0", d0.data_ptr())
            net.set_input_device("img1", d1.data_ptr())
            net.forward_async()
            net.get_blob_device("predict_flow_final", out.data_ptr())
        for _ in range(warmup):
            step()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            step()
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / steps
    res = {"workload": "%s deploy forward, %dx%d, %d pairs per step" % (model, w, h, batch), "value": batch / (ms * 1e-3), "unit": UNIT,
           "ms_per_step": ms, "steps": steps, "warmup": warmup, "output_finite": bool(torch.isfinite(out).all().item())}
    del net
    torch.cuda.empty_cache()
    return res


def train_config(torch, F, batch=8, crop=(448, 320), data=(512, 384), steps=10, warmup=3, dist=None):
    """BASELINE.json config 5: one FlowNet2-C training step (random augmentation of both frames and of the ground truth, forward,
    multi-scale EPE losses, backward down to every parameter gradient) on FlyingChairs-shaped synthetic data, batch 8, N=1.
    `value`: inputs resident in HBM; `e2e`: the same step fed from pinned host buffers, the five loss values read back."""
    cw, ch = crop
    dw, dh = data
    proto = F.fill_train_template(F.train_template("FlowNet2-C"), cw, ch, dw, dh, batch)
    net = F.Net(proto, None, F.TRAIN)
    net.fill_params(1701)
    r = np.random.default_rng(7)
    img0 = np.round(r.uniform(0, 255, (batch, 3, dh, dw))).astype(np.float32)
    img1 = np.clip(img0 + np.round(r.normal(0, 4, img0.shape)), 0, 255).astype(np.float32)
    gt = (4 * r.standard_normal((batch, 2, dh, dw))).astype(np.float32)
    dev = [torch.from_numpy(a).cuda() for a in (img0, img1, gt)]
    pin = [torch.from_numpy(a).pin_memory() for a in (img0, img1, gt)]
    names = ("img0", "img1", "flow_gt")
    losses = ["flow_loss%d" % l for l in (6, 5, 4, 3, 2)]
    host_loss = torch.empty(8, dtype=torch.float32).pin_memory()
    stream = torch.cuda.ExternalStream(net.stream)
    res = {}
    world = dist.get_world_size() if dist is not None else 1
    grads = None
    if world > 1:
        # data parallel: the same weights everywhere (one broadcast of the arena), every rank its own `batch` pairs, one all-reduce
        # of the contiguous gradient arena per step
        from flownet2_b200 import parallel as P
        with torch.cuda.stream(stream):
            P.broadcast_arena(P.arena_tensor(net), src=0)
            net.params_changed()
            grads = P.grad_arena_tensor(net)
    with torch.cuda.stream(stream):
        def step():
            for n, d in zip(names, dev):
                net.set_input_device(n, d.data_ptr())
            net.clear_param_diffs()
            net.forward_async()
            net.backward_async()
            if grads is not None:
                P.allreduce_gradients(grads)

        def step_host():
            for n, h in zip(names, pin):
                net.set_input_ptr(n, h.data_ptr())
            net.clear_param_diffs()
            net.forward_async()
            net.backward_async()
            if grads is not None:
                P.allreduce_gradients(grads)
            for i, l in enumerate(losses):
                net.get_blob_ptr(l, host_loss.data_ptr() + 4 * i)       # synchronous D2H of the scalar

        for fn, key in ((step, "device"), (step_host, "host")):
            for _ in range(warmup):
                fn()
            torch.cuda.synchronize()
            if world > 1:
                dist.barrier()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(steps):
                fn()
            e1.record()
            torch.cuda.synchronize()
            res[key] = e0.elapsed_time(e1) / steps
            if world > 1:                                   # max over the ranks
                t = torch.tensor([res[key]], device="cuda")
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
                res[key] = float(t.item())
        lt = net.time_layers()
    loss_vals = [float(net.blobs[l].data.reshape(-1)[0]) for l in losses]
    gw = net.param("conv3_1", 0, diff=True)
    out = {"workload": "FlowNet2-C training step (augmentation + forward + EPE losses + backward), crop %dx%d from %dx%d, batch %d" % (cw, ch, dw, dh, batch),
           "value": world * batch / (res["device"] * 1e-3), "unit": UNIT, "ms_per_step": res["device"], "steps": steps, "warmup": warmup,
           "n_gpus": world, "parallelism": "data parallel, one all-reduce of the %.0f MB gradient arena per step" % (net.param_diff_arena()[1] / 1e6) if world > 1 else "single GPU",
           "e2e": {"value": world * batch / (res["host"] * 1e-3), "unit": UNIT, "ms_per_step": res["host"],
                   "h2d_bytes_per_step": int(sum(a.nbytes for a in (img0, img1, gt))), "d2h_bytes_per_step": 4 * len(losses)},
           "launches_per_step": int(net.launches_per_forward + net.launches_per_backward),
           "forward_ms_layer_sum": float(sum(t for _, _, t in lt)),
           "losses": loss_vals, "losses_finite": bool(np.isfinite(loss_vals).all()),
           "grad_finite": bool(np.isfinite(gw).all() and np.abs(gw).max() > 0)}
    del net
    torch.cuda.empty_cache()
    if world > 1:
        return out
    # the reference's own GPU training step on the same graph (subprocess: a CHECK failure inside the reference aborts)
    try:
        import subprocess
        pr = subprocess.run([sys.executable, os.path.join(ROOT, "tools", "ref_train_time.py"), str(batch), "5"], capture_output=True,
                            text=True, timeout=600)
        last = [l for l in pr.stdout.strip().splitlines() if l.startswith("{")]
        out["reference_gpu"] = json.loads(last[-1]) if last else {"unavailable": "exit %d: %s" % (pr.returncode, pr.stderr.strip()[-300:])}
    except Exception as e:
        out["reference_gpu"] = {"unavailable": "%s: %s" % (type(e).__name__, e)}
    return out


def run_ours(args):
    import torch
    import torch.distributed as dist
    import flownet2_b200 as F

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        if world == 1 and args.gpus > 1:
            raise SystemExit("--gpus %d needs torchrun (WORLD_SIZE=%d)" % (args.gpus, world))
    assert torch.cuda.is_available(), "bench.py needs a GPU; there is no CPU fallback for the product path"
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    B, H, W = args.batch, args.height, args.width
    proto = F.fill_template(F.model_template(args.model), W, H)
    net = F.Net(proto, None, F.TEST, batch=B)
    stream = torch.cuda.ExternalStream(net.stream)

    # ---- weights: rank 0 fills, one NCCL broadcast of the contiguous parameter arena -------------------------
    from flownet2_b200 import parallel as P
    if rank == 0:
        net.fill_params(1701)
    if world > 1:
        arena = P.arena_tensor(net)          # zero-copy view of the contiguous parameter arena
        torch.cuda.synchronize()
        P.broadcast_arena(arena, src=0)
        torch.cuda.synchronize()
        net.params_changed()

    # ---- synthetic inputs (uint8-valued BGR floats as scripts/run-flownet.py:30-35 feeds them) ---------------
    r = np.random.default_rng(1000 + rank)
    img0 = np.round(r.uniform(0, 255, (B, 3, H, W))).astype(np.float32)
    img1 = np.clip(img0 + np.round(r.normal(0, 4, img0.shape)), 0, 255).astype(np.float32)
    pin0, pin1 = torch.from_numpy(img0).pin_memory(), torch.from_numpy(img1).pin_memory()
    dev0, dev1 = pin0.cuda(), pin1.cuda()
    # flow fields: double-buffered per rank; at N > 1 they are gathered to rank 0 ONLY (grouped ncclSend/ncclRecv, 1/N of an
    # all-gather's traffic) on a side stream, so the transfer of step i overlaps the forward of step i+1
    flow_out = [torch.empty((B, 2, H, W), device="cuda", dtype=torch.float32) for _ in range(2)]
    flow_dev = flow_out[0]
    flow_root = [torch.empty((world * B, 2, H, W), device="cuda", dtype=torch.float32) if (world > 1 and rank == 0) else None
                 for _ in range(2)]
    flow_host = torch.empty((world * B, 2, H, W), dtype=torch.float32).pin_memory() if rank == 0 else None
    gather_stream = torch.cuda.Stream() if world > 1 else None
    ev_ready = [torch.cuda.Event() for _ in range(2)]     # flow_out[k] holds this step's flow
    ev_sent = [torch.cuda.Event() for _ in range(2)]      # flow_out[k] has been gathered (buffer reusable)
    dev_state = {"i": 0}

    def gather_async(k):
        with torch.cuda.stream(gather_stream):
            gather_stream.wait_event(ev_ready[k])
            P.gather_flows_to_root(flow_out[k], flow_root[k], dst=0)
            ev_sent[k].record(gather_stream)

    def step_device():
        k = dev_state["i"] & 1
        dev_state["i"] += 1
        cur = torch.cuda.current_stream()
        net.set_input_device("img0", dev0.data_ptr())
        net.set_input_device("img1", dev1.data_ptr())
        net.forward_async()
        if world > 1:
            cur.wait_event(ev_sent[k])                    # the gather of two steps ago has released flow_out[k]
        net.get_blob_device("predict_flow_final", flow_out[k].data_ptr())
        if world > 1:
            ev_ready[k].record(cur)
            gather_async(k)

    def device_finish():
        if world > 1:
            cur = torch.cuda.current_stream()
            for e in ev_sent:
                cur.wait_event(e)

    # End-to-end loop = what a serving caller does with the public API: every step copies its inputs from pinned host
    # memory and reads its flow back to the host.  The copies run on their own streams with double buffers, so the H2D of
    # step i+1 and the D2H of step i-1 overlap the forward of step i; all of them lie inside the timed region.
    h2d_stream, d2h_stream = torch.cuda.Stream(), torch.cuda.Stream()
    stage0 = [torch.empty_like(dev0) for _ in range(2)]
    stage1 = [torch.empty_like(dev1) for _ in range(2)]
    flow_buf = flow_root if world > 1 else flow_out       # what rank 0 reads back to the host
    ev_h2d = [torch.cuda.Event() for _ in range(2)]
    ev_used = [torch.cuda.Event() for _ in range(2)]      # forward has consumed staging buffer k
    ev_flow = [torch.cuda.Event() for _ in range(2)]      # flow of the step is in flow_buf[k]
    ev_d2h = [torch.cuda.Event() for _ in range(2)]       # flow_buf[k] has been read back
    e2e_state = {"i": 0, "K": 1 << 30}

    def e2e_prefetch(k):
        with torch.cuda.stream(h2d_stream):
            h2d_stream.wait_event(ev_used[k])
            stage0[k].copy_(pin0, non_blocking=True)
            stage1[k].copy_(pin1, non_blocking=True)
            ev_h2d[k].record(h2d_stream)

    def step_e2e():
        i = e2e_state["i"]
        k = i & 1
        if i == 0:
            e2e_prefetch(0)
        if i + 1 < e2e_state["K"]:
            e2e_prefetch(k ^ 1)                           # inputs of the next step
        cur = torch.cuda.current_stream()
        cur.wait_event(ev_h2d[k])
        net.set_input_device("img0", stage0[k].data_ptr())
        net.set_input_device("img1", stage1[k].data_ptr())
        ev_used[k].record(cur)
        net.forward_async()
        cur.wait_event(ev_d2h[k])                         # flow buffers k of two steps ago have left for the host
        if world > 1:
            cur.wait_event(ev_sent[k])
        net.get_blob_device("predict_flow_final", flow_out[k].data_ptr())
        if world > 1:
            ev_ready[k].record(cur)
            gather_async(k)
            ev_flow[k] = ev_sent[k]
        else:
            ev_flow[k].record(cur)
        if rank == 0:
            with torch.cuda.stream(d2h_stream):
                d2h_stream.wait_event(ev_flow[k])
                flow_host.copy_(flow_buf[k], non_blocking=True)   # D2H of every pair's flow field
                ev_d2h[k].record(d2h_stream)
        e2e_state["i"] = i + 1

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def e2e_finish():
        cur = torch.cuda.current_stream()                 # the timed region ends when the last flow has reached the host
        for e in ev_d2h + ev_h2d + (ev_sent if world > 1 else []):
            cur.wait_event(e)

    def timed(step, K, finish=None):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(K):
            step()
        if finish:
            finish()
        e1.record()
        torch.cuda.synchronize()
        ms = torch.tensor([e0.elapsed_time(e1)], device="cuda")
        barrier()
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item())

    with torch.cuda.stream(stream):
        sampler = clocks_sampler_start(local) if rank == 0 else None       # started early: nvidia-smi takes ~0.1 s to come up
        for _ in range(max(args.warmup, 3)):
            step_device()
        barrier()
        launches0 = F.launch_count()
        t_begin = time.time()
        ms = timed(step_device, args.steps, device_finish)
        t_end = time.time()
        # the flow fields a caller of the timed path receives from its last step (on rank 0: every rank's, gathered)
        last_flow = (flow_root if world > 1 else flow_out)[(dev_state["i"] - 1) & 1]
        dumped = last_flow.cpu().numpy() if args.dump_outputs and rank == 0 else None
        clocks = clocks_sampler_stop(sampler, t_begin, t_end) if rank == 0 else None
        # graph replays do not go through the launch counter: count = kernels per forward + layout copies
        per_step_launches = net.launches_per_forward + 3
        for _ in range(2):
            step_e2e()
        torch.cuda.synchronize()
        e2e_state["i"], e2e_state["K"] = 0, args.steps
        for e in ev_used + ev_d2h + ev_sent:
            e.record(torch.cuda.current_stream())
        torch.cuda.synchronize()
        ms_e2e = timed(step_e2e, args.steps, e2e_finish)
        finite = bool(torch.isfinite(flow_out[0]).all().item() and torch.isfinite(flow_out[1]).all().item())
        # The library's own host API, no torch staging: fn2_net_set_input (pinned host NCHW -> device, layout conversion on
        # the net's stream), fn2_net_forward, fn2_net_get_blob (device -> pinned host, synchronises).  Serial, per rank.
        host_flow = torch.empty((B, 2, H, W), dtype=torch.float32).pin_memory()

        def step_host_api():
            net.set_input_ptr("img0", pin0.data_ptr())
            net.set_input_ptr("img1", pin1.data_ptr())
            net.forward_async()
            net.get_blob_ptr("predict_flow_final", host_flow.data_ptr())

        step_host_api()
        ms_host = timed(step_host_api, args.steps)

    pairs = world * B * args.steps
    value = pairs / (ms * 1e-3)
    e2e_value = pairs / (ms_e2e * 1e-3)
    line = None
    if rank == 0:
        pk = peaks()
        # per-layer device times (CUDA events on the net's stream, eager pass) -> roofline of the kernels
        with torch.cuda.stream(stream):
            net.time_layers()
            lt = net.time_layers()
        work = net.layer_work()
        conv_ms = sum(t for (_, ty, t) in lt if ty in ("Convolution", "Deconvolution"))
        conv_fl = sum(f for (_, ty, f, _) in work if ty in ("Convolution", "Deconvolution"))
        corr = [(t, w) for (n, ty, t), w in zip(lt, work) if ty == "Correlation"]
        total_ms = sum(t for (_, _, t) in lt)
        conv_tf = conv_fl / (conv_ms * 1e-3) / 1e12 if conv_ms > 0 else 0.0
        peak_bf16 = pk["bf16_tflops_sustained"] or pk["bf16_tflops"]
        tf32_peak = measure_tf32_peak(torch) if world == 1 else None
        # traffic: dram__bytes_read.sum + dram__bytes_write.sum of the profiled conv_tc_kernel<128> launch (conv3_1 of FlowNetC,
        # 473->256 3x3 at 56x128x4), read from the committed ncu capture; its algorithmic bytes are 4*(in + out + weights) = 62.8 MB
        tc_traffic, tc_traffic_file = profile_traffic("prof_tc128")
        corr_traffic, corr_traffic_file = profile_traffic("prof_corr")
        # tensor-pipe counter of the same conv3_1 launch (ncu --metrics pass, tools/gpu_profile_r02.sh)
        tp_pct, tp_file = profile_metric("tensor_pipe_tc128", "sm__pipe_tensor_cycles_active.avg.pct_of_peak_sustained_elapsed")
        roofline = {"kernel": "conv/deconv stack: conv_tc_kernel<NT> (tcgen05 3xTF32 implicit GEMM, fused bias+ReLU), summed over the layers",
                    "bound": "tensor", "achieved": conv_tf, "peak": peak_bf16, "unit": "TFLOP/s", "frac": conv_tf / peak_bf16,
                    "traffic": tc_traffic, "traffic_of": "conv3_1 launch (algorithmic 62.8e6 B), %s" % tc_traffic_file,
                    "tf32_dense_peak_measured": tf32_peak,
                    "tensor_pipe_active_pct_of_elapsed": tp_pct,
                    "tensor_pipe_counter": "sm__pipe_tensor_cycles_active.avg.pct_of_peak_sustained_elapsed of the conv3_1 launch, %s" % tp_file,
                    "peak_source": pk["source"] + ", sustained bf16 dense (kernel timed inside a long step)",
                    "share_of_step": conv_ms / total_ms if total_ms else None,
                    "algorithmic_gflop_per_step": conv_fl / 1e9,
                    # FP32 parity needs 3 TF32 MMAs per multiply-add; the TF32 pipe peaks at half the bf16 rate
                    "executed_tf32_tflops": 3.0 * conv_tf, "tf32_peak": tf32_peak or peak_bf16 / 2.0,
                    "tf32_peak_source": "cuBLAS TF32 GEMM 8192^3 measured in this run" if tf32_peak else "assumed bf16/2",
                    "frac_executed": 3.0 * conv_tf / (tf32_peak or peak_bf16 / 2.0)}
        rc = None
        if corr:
            t_ms = sum(t for t, _ in corr)
            by = sum(w[3] for _, w in corr)
            fl = sum(w[2] for _, w in corr)
            gbs = by / (t_ms * 1e-3) / 1e9
            rc = {"kernel": "Correlation d=21 k=1 s2=2 C=256: conv_tc_kernel<128> in correlation mode (3xTF32 tile x halo-block GEMMs) + hi/lo split", "bound": "hbm", "achieved": gbs, "peak": pk["hbm_gbs"], "unit": "GB/s",
                  "frac": gbs / pk["hbm_gbs"], "traffic": corr_traffic, "traffic_of": "%s (4x256x56x128 launch; algorithmic 109.3e6 B)" % corr_traffic_file, "peak_source": pk["source"],
                  "algorithmic_bytes_per_launch": by / len(corr), "ms_per_launch": t_ms / len(corr),
                  "fp32_tflops": fl / (t_ms * 1e-3) / 1e12, "share_of_step": t_ms / total_ms if total_ms else None,
                  # SURVEY 8(d): both fractions, and which one binds
                  "tensor_pipe_active_pct_of_elapsed": profile_metric("tensor_pipe_corr", "sm__pipe_tensor_cycles_active.avg.pct_of_peak_sustained_elapsed")[0],
                  "executed_tf32_tflops": 3.0 * (1008.0 / 441.0) * fl / (t_ms * 1e-3) / 1e12,
                  "binding": "tensor pipe / tensor-memory port (3xTF32 products of all 1008 halo pixels per tile, 441 kept); DRAM traffic equals the "
                             "algorithmic bytes, so HBM does not bind: frac is low because exact FP32 products cost 3 TF32 MMAs each"}
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
                "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
                "data": "synthetic", "config": config(args, world), "clocks": clocks,
                "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": int(world * 2 * B * 3 * H * W * 4),
                        "d2h_bytes_per_step": int(world * B * 2 * H * W * 4), "ms_per_step": ms_e2e / args.steps,
                        "pipelined": "H2D of step i+1 and D2H of step i-1 overlap the forward of step i (copy streams, double buffers)"},
                "e2e_host_api": {"value": world * B * args.steps / (ms_host * 1e-3), "unit": UNIT, "ms_per_step": ms_host / args.steps,
                                 "path": "fn2_net_set_input (pinned host) -> fn2_net_forward -> fn2_net_get_blob (pinned host, synchronous); no overlap",
                                 "h2d_bytes_per_step": int(world * 2 * B * 3 * H * W * 4), "d2h_bytes_per_step": int(world * B * 2 * H * W * 4)},
                "gpu_launches": int(per_step_launches * args.steps), "launches_per_step": int(per_step_launches),
                "output_finite": finite, "roofline": roofline, "roofline_correlation": rc,
                "layer_ms": {"total": total_ms, "conv_deconv": conv_ms, "correlation": sum(t for t, _ in corr) if corr else 0.0}}
        if world == 1 and not args.no_extra:
            del net
            torch.cuda.empty_cache()
            line["extra"] = {"config2": side_config(torch, F, "FlowNet2-C", 448, 320, 8, steps=args.steps),
                             "config3": side_config(torch, F, "FlowNet2-CSS", 768, 384, 4, steps=args.steps),
                             "flownet2_448x320": side_config(torch, F, "FlowNet2", 448, 320, 4, steps=args.steps),
                             "config5": train_config(torch, F, steps=args.steps)}
            rg = reference_gpu_arm(args, B)
            if rg is not None:
                line["extra"]["reference_gpu"] = rg
        if world == 1 and not args.no_cpu_baseline:
            arm = CpuArm(args)
            v, mean = arm.run(2, 1)
            line["cpu_baseline"] = {"value": v, "unit": UNIT, "cores": arm.cores, "kind": arm.kind,
                                    "sample": arm.sample + "; 1 warm-up + 2 timed steps, %.1f s per step" % mean}
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    if dumped is not None:
        write_outputs(args.dump_outputs, {"predict_flow_final": dumped})
    if line is not None:
        print(json.dumps(line), flush=True)


if __name__ == "__main__":
    a = parse_args()
    if a.config5_only:
        import torch
        import flownet2_b200 as F
        world, rank, local = int(os.environ.get("WORLD_SIZE", "1")), int(os.environ.get("RANK", "0")), int(os.environ.get("LOCAL_RANK", "0"))
        torch.cuda.set_device(local)
        dist = None
        if world > 1:
            import torch.distributed as dist
            dist.init_process_group("nccl", device_id=torch.device("cuda", local))
        line = train_config(torch, F, steps=a.steps, warmup=max(a.warmup, 3), dist=dist)
        if world > 1:
            dist.barrier()
            dist.destroy_process_group()
        if rank == 0:
            print(json.dumps(line), flush=True)
    elif a.impl == "reference":
        run_reference(a)
    else:
        run_ours(a)
