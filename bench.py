"""bench.py -- images/s of the YOLOv5 hot path on B200 (BASELINE.json metric: images/sec @640 at 1/2/4/8 GPUs + NMS us/img +
conv tensor-pipe fraction).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload config3|yolov5s|...] [--dump-outputs DIR]

Default workload = BASELINE.json configs[2] ("config3", the configuration the >= 2x / >= 70 % targets are quoted on):
yolov5l, 64 images of 640x640, bf16, forward + non_max_suppression through the public API of yolov5_b200.
  * N = 1: the whole batch of 64 on one GPU.  N > 1 (torchrun, one rank per GPU): the SAME 64 images sharded 64/N per GPU
    ("scaling": "strong", as configs[2] states it: "bs=64 on 1/2/4/8 x B200 (data-parallel shard)"); the path shards over
    independent images, so there is NO data-path collective; value = 64 * steps / max-over-ranks time.  The sub-record
    `weak_scaling` runs 64 images PER GPU for N > 1.
  * value : inputs resident in HBM, CUDA-event timed, barrier + synchronize on both sides.
  * e2e   : same metric with pinned HOST uint8 batches: every step uploads its batch (H2D) and downloads its detections
            (D2H) inside the timed region (upload of batch i+1 overlapped with compute of batch i).
  * roofline : every conv_gemm launch of one forward (Conv / C3 / SPPF / Detect head), timed per launch with CUDA events on
            the launching stream behind a queued blocker so host launch latency is not in the numbers; bound "tensor" against
            the measured sustained cuBLAS bf16 rate for l/x, "hbm" against the measured copy bandwidth for n/s/m (SURVEY 8d).
  * sub-records in the same JSON line: `config2` (yolov5s bs 32 fp16, BASELINE configs[1]), `train_ddp` (yolov5m, 16 images /
    GPU, AMP + GradScaler + fused SGD / clip / EMA; DDP's gradient all-reduce for N > 1, with the all-reduce time per step
    and the exposed part of it: BASELINE configs[3]), `sustained` (>= 2 s loop of the main step with clocks and power),
    `torch_cuda_reference` (the reference's expressions on torch-cuda: as shipped -- NCHW eager -- and tuned --
    channels_last + cudnn.benchmark + CUDA graph), `cpu_baseline`.
  * --impl reference : the reference's own CPU path.  The reference is pure Python and does not exist on the GPU box, so
    this is the oracle port (oracle/model_ref.py + oracle/nms_ref.py: the same torch-CPU fp32 expressions, pinned to the
    reference by tests/golden) on the host threads, on a bounded sample of the same workload.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

WORKLOADS = {  # name -> (model, images, image size, dtype, batch rule: "total" = sharded over the ranks, "per_gpu" = fixed per rank)
    "config3": ("yolov5l", 64, 640, "bf16", "total"),      # BASELINE.json configs[2]: the headline
    "yolov5l": ("yolov5l", 64, 640, "bf16", "per_gpu"),
    "yolov5s": ("yolov5s", 32, 640, "fp16", "per_gpu"),    # BASELINE.json configs[1]
    "yolov5n": ("yolov5n", 32, 640, "fp16", "per_gpu"),
    "yolov5m": ("yolov5m", 32, 640, "fp16", "per_gpu"),
    "yolov5x": ("yolov5x", 16, 640, "fp16", "per_gpu"),
    "yolov5x-seg-1280": ("yolov5x-seg", 2, 1280, "fp16", "per_gpu"),  # BASELINE.json configs[4]: 16 images total = 2 per GPU at 8 GPUs
    # training step (BASELINE.json configs[3]: yolov5m, 128 images total = 16 per GPU at 8 GPUs, AMP)
    "yolov5m-train": ("yolov5m", 16, 640, "fp16", "per_gpu"),
    "yolov5s-train": ("yolov5s", 16, 640, "fp16", "per_gpu"),
}
NMS_KW = dict(conf_thres=0.25, iou_thres=0.45, max_det=300)  # detect.py regime (reference detect.py:228 defaults)
TDT = {"fp16": torch.float16, "bf16": torch.bfloat16}
_OUT = None


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm=d["hbm_gbs"], tf_burst=d["bf16_tflops"], tf_sust=d["bf16_tflops_sustained"], src="measured")
    return dict(hbm=6650.0, tf_burst=1590.0, tf_sust=1400.0, src="fallback")


def synth_images_u8(bs, size, seed):
    """Blocky synthetic images (32-pixel random colour blocks + noise): unlike pure white noise they give the random
    network spatially varying activations, so objectness has a spread and NMS sees distinct candidates."""
    rs = np.random.RandomState(seed)
    base = rs.uniform(0, 1, (bs, 3, size // 32, size // 32)).astype(np.float32)
    img = np.repeat(np.repeat(base, 32, 2), 32, 3) * 0.8 + rs.uniform(0, 0.2, (bs, 3, size, size)).astype(np.float32)
    return (img * 255).astype(np.uint8)


def bench_state_dict(cfg, seed=0, frac=0.02):
    """Seeded synthetic weights shared by both arms.  Random-init heads emit no NMS candidates (objectness prior
    ~ sigmoid(-5)), so the Detect biases are calibrated once on the CPU (oracle forward of one seeded image): the
    objectness logits are rescaled/shifted so ~`frac` of the anchors have obj > 0.3 and the class logits are raised (+7) so obj*cls
    survives too -- synthetic weights only decide how much work NMS sees (~500 candidates / image, SURVEY.md section 6)."""
    from oracle import model_ref

    sd = model_ref.synth_state_dict(cfg, seed=seed, head_bias="init")
    x = torch.from_numpy(synth_images_u8(1, 640, seed + 77)).float() / 255
    threads = torch.get_num_threads()
    torch.set_num_threads(min(32, os.cpu_count() or 1))
    with torch.no_grad():
        raws = model_ref.forward(cfg, sd, x, fused=True)[-1]
    torch.set_num_threads(threads)
    nc = cfg["nc"]
    head = max(int(k.split(".")[1]) for k in sd if k.startswith("model."))
    for lvl, raw in enumerate(raws):
        na, no = raw.shape[1], raw.shape[-1]
        w = sd[f"model.{head}.m.{lvl}.weight"].view(na, no, -1)
        b = sd[f"model.{head}.m.{lvl}.bias"].view(na, no)
        for a in range(na):  # per anchor: each has its own random bias / weight row
            obj = raw[:, a, :, :, 4].flatten()
            gain = 2.0 / max(float(obj.std()), 1e-6)  # random nets give almost constant objectness: spread it to std 2
            w[a, 4] *= gain
            b[a, 4] *= gain
            q = torch.quantile(obj * gain, 1.0 - frac)
            b[a, 4] += float(-0.8473 - q.item())  # the (1-frac) quantile of the objectness logits lands on logit(0.3)
        b[:, 5 : 5 + nc] += 7.0                 # class scores ~0.9
    return sd


class StdoutGuard:
    """Keeps stdout to the single JSON line: while active, fd 1 is pointed at stderr (NCCL prints its version banner to
    stdout from native code, torchrun children inherit the fd); emit() writes to the real stdout."""

    def __init__(self):
        sys.stdout.flush()
        self.real = os.dup(1)
        os.dup2(2, 1)

    def emit(self, text: str):
        sys.stdout.flush()
        os.write(self.real, (text + "\n").encode())


class ClockSampler:
    """nvidia-smi clocks / power / throttle reasons sampled DURING the timed region (B200_PROFILING.md recipe)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int, period_ms: int = 100):
        self.idx, self.proc, self.lines, self.period = gpu_index, None, [], period_ms

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", str(self.period),
                                          "-i", str(self.idx)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, pw, reasons = [], [], [], set()
        for ln in self.lines:
            f = [t.strip() for t in ln.split(",")]
            if len(f) < 8:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2])); pw.append(float(f[3]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm), "power_w_max": max(pw) if pw else None,
                "power_w_median": statistics.median(pw) if pw else None}


# ---------------------------------------------------------------------------------------------------------------------
# CPU arm: the reference's expressions (oracle port), bounded sample
# ---------------------------------------------------------------------------------------------------------------------
def cpu_path_once(cfg, sd, x_cpu, nms_kw):
    from oracle import model_ref, nms_ref

    with torch.no_grad():
        z = model_ref.forward(cfg, sd, x_cpu, fused=True)[0]
    return nms_ref.non_max_suppression(z.numpy(), dtype="fp32", **nms_kw)


def cpu_baseline(model_name, size, sample_bs, seed, budget_s=15.0, steps=None, warmup=1):
    from yolov5_b200.cfg import model_cfg

    cores = os.cpu_count() or 1
    cfg = model_cfg(model_name)
    sd = bench_state_dict(cfg, seed)
    nms_kw = dict(NMS_KW, nm=32) if model_name.endswith("-seg") else dict(NMS_KW)
    x = torch.from_numpy(synth_images_u8(sample_bs, size, 1000)).float() / 255  # same generator as rank 0's GPU batches
    # "all the host threads it can use": torch's CPU convs get SLOWER past a point on many-core hosts (128 threads on
    # these layer sizes thrash), so probe a few pool sizes on one image and keep the fastest
    best_t, best_n = None, cores
    for n in sorted({c for c in (8, 16, 32, 64, cores) if c <= cores}):
        torch.set_num_threads(n)
        cpu_path_once(cfg, sd, x[:1], nms_kw)
        t0 = time.perf_counter()
        cpu_path_once(cfg, sd, x[:1], nms_kw)
        dt_ = time.perf_counter() - t0
        if best_t is None or dt_ < best_t:
            best_t, best_n = dt_, n
    torch.set_num_threads(best_n)
    for _ in range(warmup):
        cpu_path_once(cfg, sd, x, nms_kw)
    times = []
    t_end = time.perf_counter() + budget_s
    while (steps is None and time.perf_counter() < t_end and len(times) < 50) or (steps is not None and len(times) < steps):
        t0 = time.perf_counter()
        cpu_path_once(cfg, sd, x, nms_kw)
        times.append(time.perf_counter() - t0)
        if steps is None and len(times) >= 3 and sum(times) > budget_s:
            break
    ms = 1e3 * sum(times) / len(times)
    return {"value": sample_bs / (ms / 1e3), "unit": "images/s", "cores": torch.get_num_threads(), "kind": "port",
            "sample": f"{len(times)} x (forward + NMS) of {sample_bs} images {size}x{size} fp32 of {model_name}, oracle port of the reference's "
                      f"torch-CPU path (reference itself is Python and absent on this box)", "ms_per_step": ms}


# ---------------------------------------------------------------------------------------------------------------------
# distributed helpers
# ---------------------------------------------------------------------------------------------------------------------
class Dist:
    def __init__(self):
        self.rank = int(os.environ.get("RANK", 0))
        self.world = int(os.environ.get("WORLD_SIZE", 1))
        self.local = int(os.environ.get("LOCAL_RANK", 0))
        self.dev = None

    def init(self):
        import torch.distributed as dist

        assert torch.cuda.is_available(), "bench.py (ours) needs a CUDA device"
        torch.cuda.set_device(self.local)
        self.dev = torch.device("cuda", self.local)
        if self.world > 1 and not dist.is_initialized():
            os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
            dist.init_process_group("nccl", device_id=self.dev)

    def barrier(self):
        import torch.distributed as dist

        if self.world > 1:
            dist.barrier(device_ids=[self.local])
        torch.cuda.synchronize(self.dev)

    def done(self):
        import torch.distributed as dist

        if self.world > 1 and dist.is_initialized():
            dist.destroy_process_group()


def timed(D: Dist, fn, steps, sampler=None):
    """barrier + synchronize, CUDA events around `steps` calls of fn(i), barrier + synchronize.  Returns this rank's ms."""
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    D.barrier()
    if sampler is not None:
        sampler.start()
    e0.record()
    for i in range(steps):
        fn(i)
    e1.record()
    D.barrier()
    return e0.elapsed_time(e1)


DUMP_ELEMS = 2 << 20  # elements kept of a large output (8 MB of float32 + 16 MB of float64 positions)


def dump_outputs(out_dir, arrays):
    """Writes each array as out_dir/<name>.npy (float32, or float64 for integer data).  Large tensors are reduced to
    DUMP_ELEMS elements at seeded positions, stored beside them as <name>_index.npy, so two builds of the project can be
    compared element for element on the same inputs."""
    os.makedirs(out_dir, exist_ok=True)
    for name, t in arrays.items():
        t = t.detach()
        if t.numel() > DUMP_ELEMS:
            flat = t.reshape(-1)
            pos = np.sort(np.random.RandomState(0).choice(flat.numel(), DUMP_ELEMS, replace=False))
            t = flat[torch.from_numpy(pos).to(flat.device)]
            np.save(os.path.join(out_dir, f"{name}_index.npy"), pos.astype(np.float64))
        t = t.cpu()
        np.save(os.path.join(out_dir, f"{name}.npy"), (t.double() if not t.is_floating_point() else t.float()).numpy())


# ---------------------------------------------------------------------------------------------------------------------
# inference leg
# ---------------------------------------------------------------------------------------------------------------------
def infer_leg(D: Dist, model_name, bs, size, dt, steps, warmup, extras=True, cpu_base=True, sustain_s=0.0, tag="", dump_dir=None):
    """forward + NMS on `bs` images per rank.  Returns the record dict on rank 0 (None elsewhere).  With `dump_dir`, rank 0
    writes what the last timed step returned (see dump_outputs)."""
    from yolov5_b200 import _lib
    from yolov5_b200.cfg import model_cfg
    from yolov5_b200.models.yolo import DetectionModel, SegmentationModel
    from yolov5_b200.parallel import aggregate_throughput
    from yolov5_b200.utils.general import nms_device

    dev, rank, world = D.dev, D.rank, D.world
    seg = model_name.endswith("-seg")
    nms_kw = dict(NMS_KW, nm=32) if seg else dict(NMS_KW)
    cfg = model_cfg(model_name)
    sd = bench_state_dict(cfg, seed=0)
    model = (SegmentationModel if seg else DetectionModel)(model_name)
    model.load_state_dict(sd)
    model = model.to(TDT[dt]).to(dev).eval()
    n_rot = 3  # rotating inputs (> L2 together at these sizes); every step also streams GBs of activations
    host_u8 = [torch.from_numpy(synth_images_u8(bs, size, 1000 + 10 * rank + i)).pin_memory() for i in range(n_rot)]
    dev_in = [(h.to(dev).to(TDT[dt]) / 255) for h in host_u8]

    def step(i, keep=None):
        z = model(dev_in[i % n_rot])[0]
        out = nms_device(z, **nms_kw)  # device-side result (rows, idx, count): no host sync inside `value`
        if keep is not None:
            keep.update(z=z, nms=out)
        return out

    for i in range(warmup):
        out = step(i)
    torch.cuda.synchronize(dev)
    cand = int(out[2].sum().item())

    # ---------------- value: device-resident inputs ----------------
    sampler = ClockSampler(D.local) if rank == 0 else None
    l0 = _lib.launch_count()
    last = {}
    ms_total = timed(D, lambda i: step(i, last if i == steps - 1 else None), steps, sampler)
    clocks = sampler.stop() if sampler is not None else None
    eager_launches = _lib.launch_count() - l0
    if dump_dir and rank == 0:  # the last timed batch: model(x)[0] and what non_max_suppression returns for it, images concatenated
        rows, idx, cnt = last["nms"]
        dump_outputs(dump_dir, {"predictions": last["z"], "detections_per_image": cnt,
                                "detections": torch.cat([rows[b, :c] for b, c in enumerate(cnt.tolist())]),
                                "detection_indices": torch.cat([idx[b, :c] for b, c in enumerate(cnt.tolist())])})
    prog = model._program(dev_in[0])
    graph_launches = len(prog.ops) * steps if prog.graph is not None else 0
    images, worst_ms = aggregate_throughput(bs * steps, ms_total, dev)
    value = images / (worst_ms / 1e3)

    # ---------------- e2e: pinned host uint8 in, detections out, per step, copy/compute overlapped ----------------
    copy_s = torch.cuda.Stream(dev)
    main_s = torch.cuda.current_stream(dev)
    host_out = torch.empty(bs, NMS_KW["max_det"], 6 + (32 if seg else 0), dtype=torch.float32).pin_memory()
    host_cnt = torch.empty(bs, dtype=torch.int32).pin_memory()
    stage = [torch.empty(bs, 3, size, size, dtype=torch.uint8, device=dev) for _ in range(2)]
    ready = [torch.cuda.Event() for _ in range(2)]
    freed = [torch.cuda.Event() for _ in range(2)]

    def e2e_run(k):
        for i in range(k + 1):
            if i < k:  # upload batch i on the copy stream (uint8: the model scales by 1/255 on the device)
                with torch.cuda.stream(copy_s):
                    if i >= 2:
                        copy_s.wait_event(freed[i % 2])
                    stage[i % 2].copy_(host_u8[i % n_rot], non_blocking=True)
                    ready[i % 2].record(copy_s)
            if i >= 1:  # compute batch i-1
                j = (i - 1) % 2
                main_s.wait_event(ready[j])
                z = model(stage[j])[0]
                freed[j].record(main_s)
                rows, _, cnt = nms_device(z, **nms_kw)
                host_out.copy_(rows, non_blocking=True)
                host_cnt.copy_(cnt, non_blocking=True)

    e2e_run(2)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    D.barrier()
    e0.record()
    e2e_run(steps)
    e1.record()
    D.barrier()
    e2e_images, e2e_ms = aggregate_throughput(bs * steps, e0.elapsed_time(e1), dev)
    h2d = bs * 3 * size * size
    d2h = host_out.numel() * 4 + host_cnt.numel() * 4

    # ---------------- sustained: >= sustain_s seconds of the same step, clocks + power sampled ----------------
    sustained = None
    if sustain_s > 0:
        per_step = worst_ms / steps / 1e3
        n_long = max(steps, int(sustain_s / max(per_step, 1e-4)) + 1)
        s2 = ClockSampler(D.local, 200) if rank == 0 else None
        ms_long = timed(D, step, n_long, s2)
        ck = s2.stop() if s2 is not None else None
        li, lms = aggregate_throughput(bs * n_long, ms_long, dev)
        sustained = {"value": li / (lms / 1e3), "unit": "images/s", "steps": n_long, "seconds": lms / 1e3, "clocks": ck}

    rec = None
    if rank == 0:
        pk = peaks()
        st = _lib.stream_ptr(dev)
        # ---------------- roofline of the dominant kernel (conv_gemm incl. the Detect-head GEMMs), per launch ----------------
        import ctypes as C

        no = prog.det_shapes[0][-1]
        zbuf = torch.empty(prog.B, prog.z_rows, no, dtype=prog.dtype, device=dev)
        raws = [torch.empty(s, dtype=prog.dtype, device=dev) for s in prog.det_shapes]
        items = [(op.name, op.fn is prog.lib.y5_conv_plan_run, (lambda op=op: op.run(st))) for op in prog.ops]
        for plan, raw in zip(prog.head_ops, raws):
            items.append(("detect", True, (lambda plan=plan, raw=raw: _lib.check(
                prog.lib.y5_detect_plan_run_to(plan, raw.data_ptr(), zbuf.data_ptr(), C.c_void_p(st)), "detect"))))
        evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in items]
        reps, conv_ms, all_ms = 3, 0.0, 0.0
        for _ in range(reps):
            torch.cuda._sleep(30_000_000)  # ~15 ms of GPU time: the host enqueues everything before the GPU gets to it
            for (_, _, run), (s, e) in zip(items, evs):
                s.record(); run(); e.record()
            torch.cuda.synchronize(dev)
            for (_, is_conv, _), (s, e) in zip(items, evs):
                t = s.elapsed_time(e)
                all_ms += t
                if is_conv:
                    conv_ms += t
        conv_ms /= reps; all_ms /= reps
        conv_bytes = prog.act_bytes + prog.weight_bytes
        n_conv = sum(1 for _, c, _ in items if c)
        gbs = conv_bytes / (conv_ms / 1e3) / 1e9
        tfs = prog.flops / (conv_ms / 1e3) / 1e12
        traffic = None
        tp = os.path.join(ROOT, "profiles", "traffic.json")
        if os.path.exists(tp):
            traffic = json.load(open(tp)).get(model_name)
        hbm_bound = model_name in ("yolov5n", "yolov5s", "yolov5m")  # SURVEY.md section 8d: AI below machine balance
        roof = {"kernel": "conv_gemm_kernel (tcgen05 implicit GEMM: every Conv / C3 / SPPF / Detect-head launch of one forward)",
                "bound": "hbm" if hbm_bound else "tensor",
                "achieved": gbs if hbm_bound else tfs, "peak": pk["hbm"] if hbm_bound else pk["tf_sust"],
                "unit": "GB/s" if hbm_bound else "TFLOP/s", "frac": (gbs / pk["hbm"]) if hbm_bound else (tfs / pk["tf_sust"]),
                "traffic": traffic, "peak_source": pk["src"] + (" (sustained cuBLAS bf16: kernels timed inside a long step)" if not hbm_bound else " (copy)"),
                "launches": n_conv, "avg_launch_us": 1e3 * conv_ms / max(n_conv, 1),
                "algorithmic_bytes_per_launch": conv_bytes / max(n_conv, 1), "flops_per_launch": prog.flops / max(n_conv, 1),
                "hbm_gbs": gbs, "tensor_tflops": tfs, "tensor_frac_of_sustained": tfs / pk["tf_sust"], "tensor_frac_of_burst": tfs / pk["tf_burst"],
                "hbm_frac": gbs / pk["hbm"], "conv_ms_per_forward": conv_ms, "all_ops_ms_per_forward": all_ms}

        # ---------------- NMS us/img (second half of the metric) ----------------
        z = model(dev_in[0])[0]
        torch.cuda.synchronize(dev)
        e0.record()
        for _ in range(10):
            nms_device(z, **nms_kw)
        e1.record()
        torch.cuda.synchronize(dev)
        nms_us = 1e3 * e0.elapsed_time(e1) / 10 / bs

        fwd_only = tc_ref = cb = None
        torch.cuda.synchronize(dev)
        e0.record()
        for i in range(steps):
            model(dev_in[i % n_rot])
        e1.record()
        torch.cuda.synchronize(dev)
        fwd_only = bs * steps / (e0.elapsed_time(e1) / 1e3)
        if extras:
            tc_ref = torch_cuda_reference(cfg, sd, dev_in, dt, steps, dev)
        if cpu_base:
            cb = cpu_baseline(model_name, size, 2 if model_name in ("yolov5l", "yolov5x", "yolov5x-seg") else 4, seed=0, budget_s=15.0)
            cb = {k: cb[k] for k in ("value", "unit", "cores", "kind", "sample")}
        rec = {"value": value, "unit": "images/s", "ms_per_step": worst_ms / steps, "clocks": clocks,
               "e2e": {"value": e2e_images / (e2e_ms / 1e3), "unit": "images/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h},
               "gpu_launches": int(eager_launches + graph_launches), "roofline": roof, "cpu_baseline": cb,
               "forward_only": {"value": fwd_only, "unit": "images/s"}, "torch_cuda_reference": tc_ref, "sustained": sustained,
               "detail": {"model": model_name, "per_gpu_batch": bs, "nms_detections_per_batch": cand, "nms_us_per_img": nms_us,
                          "launches_per_forward": prog.launches_per_forward(), "gflop_per_img": prog.flops / bs / 1e9,
                          "nms_includes_host_sync": False}}
    del model
    torch.cuda.empty_cache()
    return rec


def torch_cuda_reference(cfg, sd, dev_in, dt, steps, dev):
    """The reference's own torch ops (oracle functional forward == models/common.py + models/yolo.py expressions) on torch-cuda,
    forward only, same weights / inputs: (a) as the reference ships it -- NCHW eager, cudnn.benchmark off; (b) tuned --
    channels_last + cudnn.benchmark + the whole forward replayed from a CUDA graph."""
    out = {}
    try:
        from oracle import model_ref

        bs = dev_in[0].shape[0]
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        sd_dev = {k: (v.to(dev, TDT[dt]) if v.is_floating_point() else v.to(dev)) for k, v in sd.items()}
        with torch.no_grad():
            for _ in range(3):
                model_ref.forward(cfg, sd_dev, dev_in[0], fused=True)
            torch.cuda.synchronize(dev)
            e0.record()
            for i in range(steps):
                model_ref.forward(cfg, sd_dev, dev_in[i % len(dev_in)], fused=True)
            e1.record()
            torch.cuda.synchronize(dev)
        out["as_shipped"] = {"value": bs * steps / (e0.elapsed_time(e1) / 1e3), "unit": "images/s",
                             "what": f"reference expressions (F.conv2d / silu / max_pool2d / cat ...) on torch-cuda {dt} NCHW eager, "
                                     f"cuDNN {torch.backends.cudnn.version()}, forward only"}
        try:
            old = torch.backends.cudnn.benchmark
            torch.backends.cudnn.benchmark = True
            sd_cl = {k: (v.contiguous(memory_format=torch.channels_last) if v.dim() == 4 else v) for k, v in sd_dev.items()}
            xs = [x.contiguous(memory_format=torch.channels_last) for x in dev_in]
            static_x = xs[0].clone()
            with torch.no_grad():
                side = torch.cuda.Stream(dev)
                side.wait_stream(torch.cuda.current_stream(dev))
                with torch.cuda.stream(side):
                    for _ in range(3):
                        model_ref.forward(cfg, sd_cl, static_x, fused=True)
                torch.cuda.current_stream(dev).wait_stream(side)
                torch.cuda.synchronize(dev)
                g = torch.cuda.CUDAGraph()
                with torch.cuda.graph(g):
                    static_out = model_ref.forward(cfg, sd_cl, static_x, fused=True)
                for i in range(3):
                    static_x.copy_(xs[i % len(xs)]); g.replay()
                torch.cuda.synchronize(dev)
                e0.record()
                for i in range(steps):
                    static_x.copy_(xs[i % len(xs)])
                    g.replay()
                e1.record()
                torch.cuda.synchronize(dev)
            out["tuned"] = {"value": bs * steps / (e0.elapsed_time(e1) / 1e3), "unit": "images/s",
                            "what": "same expressions, channels_last weights / activations + cudnn.benchmark + whole forward replayed from a CUDA graph"}
            del g, static_out
            torch.backends.cudnn.benchmark = old
        except Exception as ex:  # noqa: BLE001
            out["tuned"] = {"unavailable": repr(ex)[:200]}
        del sd_dev
    except Exception as ex:  # noqa: BLE001
        out["as_shipped"] = {"unavailable": repr(ex)[:200]}
    return out


# ---------------------------------------------------------------------------------------------------------------------
# training leg (BASELINE configs[3])
# ---------------------------------------------------------------------------------------------------------------------
def train_leg(D: Dist, model_name, bs, size, dt, steps, warmup, extras=True, dump_dir=None):
    """images/s of one optimisation step through the public API: model.train() under autocast, ComputeLoss, GradScaler-scaled
    backward, fused un-scale + clip + SGD-Nesterov (3 groups) + zero_grad (+ ModelEMA on rank 0, as train.py:251 does); per-GPU
    batch fixed, gradients averaged over ranks for N > 1 by FusedSGD.data_parallel -- one NCCL all-reduce of the packed arena -- with the
    smart_DDP wrapper timed beside it (reference train.py:401-421, utils/torch_utils.py:61-70)."""
    import torch.distributed as dist

    from oracle import loss_ref, model_ref  # synthetic labels / weights, and the torch reference arm
    from yolov5_b200 import _lib
    from yolov5_b200.cfg import HYP_SCRATCH_LOW, model_cfg
    from yolov5_b200.models.yolo import DetectionModel
    from yolov5_b200.parallel import aggregate_throughput
    from yolov5_b200.utils.loss import ComputeLoss
    from yolov5_b200.utils.torch_utils import GraphedTrainStep, ModelEMA, smart_DDP, smart_optimizer

    dev, rank, world = D.dev, D.rank, D.world
    tdt = TDT[dt]
    cfg = model_cfg(model_name)
    sd = model_ref.synth_state_dict(cfg, seed=0)
    hyp = dict(HYP_SCRATCH_LOW)

    def build():
        m = DetectionModel(model_name)
        m.load_state_dict(sd)
        m = m.to(dev).train()
        m.hyp = dict(hyp)
        return m

    model = build()
    loss_fn = ComputeLoss(model)
    net = model
    opt = smart_optimizer(model, "SGD", lr=1e-3, momentum=hyp["momentum"], decay=hyp["weight_decay"])
    if world > 1:  # the path's collective: gradients packed into one arena, ONE NCCL all-reduce per step, update from the arena
        opt.data_parallel(model)
    scaler = torch.amp.GradScaler("cuda", enabled=tdt == torch.float16)
    ema = ModelEMA(model) if rank == 0 else None
    n_rot = 3
    host_img = [torch.from_numpy(synth_images_u8(bs, size, 2000 + 10 * rank + i)).pin_memory() for i in range(n_rot)]
    host_tgt = [torch.from_numpy(loss_ref.synth_targets(bs, seed=3000 + 10 * rank + i)).float().pin_memory() for i in range(n_rot)]
    dev_img = [h.to(dev) for h in host_img]
    dev_tgt = [h.to(dev) for h in host_tgt]

    def step(img, tgt, net=net, opt=opt, loss_fn=loss_fn, scaler=scaler, ema=ema, model=model, sync=True):
        import contextlib

        ctx = net.no_sync() if (net is not model and not sync) else contextlib.nullcontext()
        with ctx:
            with torch.autocast("cuda", dtype=tdt):
                p = net(img)
            loss, items = loss_fn(p, tgt)
            if world > 1:
                loss = loss * world  # train.py:405: gradients are averaged over ranks, the reference rescales
            scaler.scale(loss).backward()
        opt.fused_step(scaler=scaler, max_norm=10.0, ema=ema, model=model)  # train.py:413-421
        opt.zero_grad()
        return items

    for i in range(max(warmup, 3)):
        step(dev_img[i % n_rot], dev_tgt[i % n_rot])
    sampler = ClockSampler(D.local) if rank == 0 else None
    l0 = _lib.launch_count()
    last = {}

    def timed_step(i):
        items = step(dev_img[i % n_rot], dev_tgt[i % n_rot])
        if i == steps - 1:
            last["items"] = items

    ms = timed(D, timed_step, steps, sampler)
    clocks = sampler.stop() if sampler is not None else None
    launches = _lib.launch_count() - l0
    if dump_dir and rank == 0:  # the last timed step's loss items and the parameters it left
        dump_outputs(dump_dir, {"loss_items": last["items"],
                                "parameters": torch.cat([q.detach().float().reshape(-1) for q in model.parameters()])})
    images, worst_ms = aggregate_throughput(bs * steps, ms, dev)
    value = images / (worst_ms / 1e3)

    # the collective: DDP's all-reduce of the fp32 gradients -- in isolation, and how much of it the step exposes
    comm = None
    n_params = sum(p.numel() for p in model.parameters())
    if world > 1:
        flat = torch.zeros(n_params, dtype=torch.float32, device=dev)
        for _ in range(3):
            dist.all_reduce(flat)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        D.barrier()
        e0.record()
        for _ in range(10):
            dist.all_reduce(flat)
        e1.record()
        D.barrier()
        _, ar_ms = aggregate_throughput(0, e0.elapsed_time(e1) / 10, dev)
        # the same step with the all-reduce skipped (pack + update from the arena still run): what the collective exposes
        dp = opt._dp
        opt._dp = (dp[0], 1)
        step(dev_img[0], dev_tgt[0])
        ms_local = timed(D, lambda i: step(dev_img[i % n_rot], dev_tgt[i % n_rot]), steps)
        opt._dp = dp
        _, local_ms = aggregate_throughput(0, ms_local, dev)
        # and the reference's arrangement for comparison: the module wrapped by smart_DDP (torch DistributedDataParallel:
        # autograd hooks, 25 MB buckets, per-step buffer broadcast), same kernels and optimizer otherwise
        ddp_ms = None
        try:
            m2 = build()
            net2 = smart_DDP(m2)
            opt2 = smart_optimizer(m2, "SGD", lr=1e-3, momentum=hyp["momentum"], decay=hyp["weight_decay"])
            sc2 = torch.amp.GradScaler("cuda", enabled=tdt == torch.float16)
            kw = dict(net=net2, opt=opt2, loss_fn=ComputeLoss(m2), scaler=sc2, ema=None, model=m2)
            for i in range(3):
                step(dev_img[i % n_rot], dev_tgt[i % n_rot], **kw)
            ms_ddp = timed(D, lambda i: step(dev_img[i % n_rot], dev_tgt[i % n_rot], **kw), steps)
            _, ddp_worst = aggregate_throughput(0, ms_ddp, dev)
            ddp_ms = ddp_worst / steps
            del m2, net2, opt2, kw
        except Exception as ex:  # noqa: BLE001
            ddp_ms = repr(ex)[:200]
        nbytes = 4 * n_params
        comm = {"collective": "ONE NCCL all-reduce (average) per step over the packed fp32 gradient arena (FusedSGD.data_parallel: y5_grad_pack -> "
                              "all_reduce -> y5_opt_step reading the arena); no autograd hooks / buckets / copy-backs",
                "bytes_per_step": nbytes, "allreduce_ms_in_isolation": ar_ms,
                "bus_gbs_in_isolation": 2 * (world - 1) / world * nbytes / (ar_ms / 1e3) / 1e9,
                "step_ms_with_allreduce": worst_ms / steps, "step_ms_without_allreduce": local_ms / steps,
                "exposed_ms_per_step": max(worst_ms - local_ms, 0.0) / steps,
                "step_ms_torch_DDP_wrapper (smart_DDP, same kernels)": ddp_ms,
                "what_limits": "per-GPU step time (kernels + Python launch issue); the all-reduce is not overlapped -- it is one "
                               "call of ~allreduce_ms_in_isolation after backward"}
        del flat

    # e2e: pinned host uint8 images + labels uploaded every step, loss items read back every step
    host_items = torch.empty(3, dtype=torch.float32).pin_memory()

    def e2e_step(i):
        img = host_img[i % n_rot].to(dev, non_blocking=True)
        tgt = host_tgt[i % n_rot].to(dev, non_blocking=True)
        host_items.copy_(step(img, tgt), non_blocking=True)

    e2e_step(0)
    e2e_ms = timed(D, e2e_step, steps)
    e2e_images, e2e_worst = aggregate_throughput(bs * steps, e2e_ms, dev)

    rec = None
    graphed = tc_ref = None
    graph_dp = world > 1 and os.environ.get("Y5_BENCH_GRAPH_DP", "0") != "0"
    if (world == 1 and rank == 0 and extras) or graph_dp:
        # whole step replayed from one CUDA graph through the public helper: what the kernels cost without Python.  N > 1: every
        # rank captures its step including the ONE all-reduce of the gradient arena (FusedSGD.data_parallel) and replays in lock-step.
        try:
            gm = build()
            gopt = smart_optimizer(gm, "SGD", lr=1e-3, momentum=hyp["momentum"], decay=hyp["weight_decay"])
            if world > 1:
                gopt.data_parallel(gm)
            gstep = GraphedTrainStep(gm, ComputeLoss(gm), gopt, batch=bs, size=size, amp_dtype=tdt, max_norm=10.0,
                                     ema=ModelEMA(gm) if rank == 0 else None)

            def g_run(i):
                host_items.copy_(gstep(host_img[i % n_rot], host_tgt[i % n_rot]), non_blocking=True)

            for i in range(2):
                g_run(i)
            g_ms = timed(D, g_run, steps)
            g_images, g_worst = aggregate_throughput(bs * steps, g_ms, dev)
            graphed = {"value": g_images / (g_worst / 1e3), "unit": "images/s", "ms_per_step": g_worst / steps,
                       "what": "yolov5_b200.utils.torch_utils.GraphedTrainStep: the same step (dynamic loss scale, clip, fused SGD, EMA"
                               + (", the gradient all-reduce" if world > 1 else "") + ") captured once in a CUDA graph per rank, replayed per batch "
                               "with pinned-host uint8 images + labels uploaded and loss items downloaded"}
            del gstep, gm, gopt
        except Exception as ex:  # noqa: BLE001
            graphed = {"unavailable": repr(ex)[:300]}
    if rank == 0 and extras:
        try:  # the reference's torch-cuda build: its expressions through autocast + its loss as torch ops + torch SGD/clip/GradScaler/EMA math
            params = {k: (torch.nn.Parameter(v.to(dev)) if v.is_floating_point() and "running" not in k and "anchors" not in k
                          else v.to(dev)) for k, v in sd.items()}
            plist = [q for q in params.values() if isinstance(q, torch.nn.Parameter)]
            anchors = params[[k for k in params if k.endswith(".anchors")][0]]
            opt_r = torch.optim.SGD(plist, lr=1e-3, momentum=hyp["momentum"], nesterov=True, weight_decay=0.0, foreach=True)
            sc_r = torch.amp.GradScaler("cuda", enabled=tdt == torch.float16)
            ema_r = [q.detach().clone() for q in plist]

            def step_ref(img, tgt):
                x = img.to(tdt) / 255
                with torch.autocast("cuda", dtype=tdt):
                    p = model_ref.forward(cfg, params, x, training=True, bn_batch_stats=True)
                    loss, _ = loss_ref.compute_loss_torch([q.float() for q in p], tgt, anchors, hyp)
                opt_r.zero_grad(set_to_none=True)
                sc_r.scale(loss).backward()
                sc_r.unscale_(opt_r)
                torch.nn.utils.clip_grad_norm_(plist, max_norm=10.0)
                sc_r.step(opt_r)
                sc_r.update()
                torch._foreach_mul_(ema_r, 0.999)
                torch._foreach_add_(ema_r, [q.detach() for q in plist], alpha=0.001)

            for i in range(3):
                step_ref(dev_img[i % n_rot], dev_tgt[i % n_rot])
            torch.cuda.synchronize(dev)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for i in range(steps):
                step_ref(dev_img[i % n_rot], dev_tgt[i % n_rot])
            e1.record()
            torch.cuda.synchronize(dev)
            tc_ref = {"value": bs * steps / (e0.elapsed_time(e1) / 1e3), "unit": "images/s",
                      "what": f"reference expressions under torch.autocast({dt}) on one GPU (no DDP): F.conv2d / batch_norm(training) / silu / max_pool2d / "
                              f"cat (cuDNN {torch.backends.cudnn.version()}), the reference's loss as torch ops (oracle.loss_ref.compute_loss_torch), GradScaler, "
                              "clip_grad_norm_, torch.optim.SGD(foreach), foreach EMA -- none of this repo's kernels"}
            del params, plist, opt_r, ema_r
        except Exception as ex:  # noqa: BLE001
            tc_ref = {"unavailable": repr(ex)[:300]}
    if rank == 0:
        pk = peaks()
        # algorithmic bytes of a training step (SURVEY.md 8d convention, layer-fused ideal, 2 B/element): forward reads each
        # conv input and writes its output once (A); backward reads dy + x for the weight gradient and dy for the data
        # gradient and writes dx (~2.5 A)
        roof = None
        try:
            em = DetectionModel(model_name)
            em.load_state_dict(sd)
            em = em.to(tdt).to(dev).eval()
            prog = em._program(torch.empty(bs, 3, size, size, dtype=tdt, device=dev))
            prog_bytes = 3.5 * prog.act_bytes + 3 * prog.weight_bytes
            flops = 3 * prog.flops
            ms_step = worst_ms / steps
            gbs = prog_bytes / (ms_step / 1e3) / 1e9
            roof = {"kernel": "whole training step (conv_gemm fwd+dgrad, conv_wgrad, BN/SiLU passes, fused optimizer)", "bound": "hbm", "achieved": gbs,
                    "peak": pk["hbm"], "unit": "GB/s", "frac": gbs / pk["hbm"], "traffic": None, "peak_source": pk["src"],
                    "algorithmic_bytes_per_step": prog_bytes, "flops_per_step": flops, "tensor_tflops": flops / (ms_step / 1e3) / 1e12}
            if isinstance(graphed, dict) and graphed.get("ms_per_step"):  # the same step without Python between the launches
                g_gbs = prog_bytes / (graphed["ms_per_step"] / 1e3) / 1e9
                roof["graph_replayed"] = {"achieved": g_gbs, "frac": g_gbs / pk["hbm"], "tensor_tflops": flops / (graphed["ms_per_step"] / 1e3) / 1e12}
            del em, prog
        except Exception:  # noqa: BLE001
            pass
        rec = {"value": value, "unit": "images/s", "ms_per_step": worst_ms / steps, "clocks": clocks,
               "e2e": {"value": e2e_images / (e2e_worst / 1e3), "unit": "images/s", "h2d_bytes_per_step": bs * 3 * size * size + int(host_tgt[0].numel()) * 4,
                       "d2h_bytes_per_step": 12},
               "gpu_launches": int(launches), "launches_per_step": int(launches) // max(steps, 1), "roofline": roof, "collective": comm,
               "cuda_graph_step": graphed, "torch_cuda_reference_train": tc_ref,
               "detail": {"model": model_name, "per_gpu_batch": bs, "global_batch": bs * world, "params": n_params,
                          "recipe": f"autocast {dt}, GradScaler, fp32 master weights, fused un-scale/clip/SGD-Nesterov(3 groups)/zero_grad, ModelEMA on rank 0",
                          "parallelism": f"dp{world} (one NCCL all-reduce of the packed gradient arena per step)" if world > 1 else "single GPU",
                          "labels": "COCO128-shaped synthetic targets (oracle.loss_ref.synth_targets), ~7.3 per image"}}
    del model, net, opt
    torch.cuda.empty_cache()
    return rec


# ---------------------------------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default=os.environ.get("Y5_BENCH_WORKLOAD", "config3"), choices=list(WORKLOADS))
    ap.add_argument("--batch", type=int, default=0, help="override the per-GPU batch")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-subrecords", action="store_true", help="main workload only (profiling runs)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the main workload's outputs of its last timed step to DIR/<name>.npy")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.dump_outputs and a.impl != "ours":
        ap.error("--dump-outputs records the outputs of --impl ours")
    a.warmup = max(a.warmup, 3)
    global _OUT
    _OUT = StdoutGuard()
    D = Dist()
    model_name, images, size, dt, rule = WORKLOADS[a.workload]
    world = D.world
    if rule == "total":
        if images % world:
            raise SystemExit(f"bench.py: {images} images do not shard over {world} ranks")
        bs = images // world
    else:
        bs = images
    if a.batch:
        bs = a.batch
    train = a.workload.endswith("-train")
    scaling = "strong" if rule == "total" and not a.batch else "weak"
    what = "training step" if train else "forward + NMS"
    cfg_desc = {"workload": f"{model_name} {what}, {bs * world} images of {size}x{size} per step ({bs}/GPU x {world}), {dt}"
                            + (" -- BASELINE.json configs[2]" if a.workload == "config3" else ""),
                "per_gpu_batch": bs, "global_batch": bs * world,
                "parallelism": (f"dp{world} DDP all-reduce" if train else f"replicas x{world} (image shards, no collective)"),
                "nms": None if train else "conf 0.25 iou 0.45 max_det 300 (detect regime)"}

    if a.impl == "reference":
        if D.rank != 0:
            return 0
        if train:
            _OUT.emit(json.dumps({"impl": "reference", "unavailable": "the CPU reference arm covers the inference metric only; the "
                                  "training workload reports torch_cuda_reference_train instead"}))
            return 0
        sample_bs = 2 if model_name in ("yolov5l", "yolov5x", "yolov5x-seg") else 4
        cb = cpu_baseline(model_name, size, sample_bs, seed=0, steps=a.steps, warmup=min(a.warmup, 2))
        cfg_desc["reference_sample"] = cb["sample"]
        line = {"impl": "reference", "metric": "images/sec @640 (forward + NMS)", "value": cb["value"], "unit": "images/s",
                "n_gpus": a.gpus, "steps": a.steps, "warmup": a.warmup, "ms_per_step": cb["ms_per_step"], "higher_is_better": True,
                "scaling": scaling, "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": cfg_desc,
                "cpu_baseline": {k: cb[k] for k in ("value", "unit", "cores", "kind", "sample")},
                "e2e": {"value": cb["value"], "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                "gpu_launches": 0}
        _OUT.emit(json.dumps(line))
        return 0

    D.init()
    subs = not a.no_subrecords and a.workload == "config3"
    if train:
        rec = train_leg(D, model_name, bs, size, dt, a.steps, a.warmup, dump_dir=a.dump_outputs)
        metric = "images/sec @640 (training step: forward + loss + backward + optimizer)"
    else:
        rec = infer_leg(D, model_name, bs, size, dt, a.steps, a.warmup, extras=True, cpu_base=not a.no_cpu_baseline,
                        sustain_s=2.5 if subs else 0.0, dump_dir=a.dump_outputs)
        metric = "images/sec @640 (forward + NMS)"
    sub = {}
    if subs:
        def leg(name, fn):
            """A sub-record never takes the headline down with it: an exception (raised symmetrically on every rank: the legs run
            the same code) is recorded in its place."""
            try:
                return fn()
            except Exception as ex:  # noqa: BLE001
                torch.cuda.empty_cache()
                return {"unavailable": f"{type(ex).__name__}: {str(ex)[:300]}"} if D.rank == 0 else None

        r2 = leg("config2", lambda: infer_leg(D, "yolov5s", 32, 640, "fp16", a.steps, a.warmup, extras=D.world == 1, cpu_base=False))
        if r2 is not None:
            r2["config"] = "BASELINE.json configs[1]: yolov5s forward + NMS, 32 images/GPU, 640x640, fp16 (per-GPU batch fixed)"
            sub["config2"] = r2
        if D.world > 1:
            rw = leg("weak", lambda: infer_leg(D, model_name, images, size, dt, max(a.steps // 2, 5), 3, extras=False, cpu_base=False))
            if rw is not None:
                rw["config"] = f"weak scaling of the main workload: {images} images PER GPU ({images * D.world} per step)"
                sub["weak_scaling"] = {k: rw[k] for k in ("value", "unit", "ms_per_step", "e2e", "config", "unavailable") if k in rw}
        rt = leg("train", lambda: train_leg(D, "yolov5m", 16, 640, "fp16", max(a.steps // 2, 8), 3, extras=D.world == 1))
        if rt is not None:
            rt["config"] = (f"BASELINE.json configs[3]: yolov5m training step, 16 images/GPU x {D.world} = {16 * D.world} per step, 640x640, AMP fp16"
                            + (", DDP gradient all-reduce" if D.world > 1 else ""))
            sub["train_ddp"] = rt
    if D.rank == 0:
        cfg_desc.update({"model": model_name, "l2": "3 rotating input batches and GBs of activations streamed per step (>> 126 MB L2)",
                         "weights": "seeded synthetic (oracle.model_ref.synth_state_dict), head bias calibrated to ~2% anchors > 0.25"})
        cfg_desc.update(rec.pop("detail"))
        sustained = rec.pop("sustained", None)
        line = {"metric": metric, "value": rec.pop("value"), "unit": rec.pop("unit"), "n_gpus": D.world, "steps": a.steps,
                "warmup": a.warmup, "ms_per_step": rec.pop("ms_per_step"), "higher_is_better": True, "scaling": scaling,
                "vs_baseline": None, "dtype": "f16" if dt == "fp16" else "bf16", "data": "synthetic", "config": cfg_desc}
        line.update(rec)
        if sustained is not None:
            line["sustained"] = sustained
        line.update(sub)
        _OUT.emit(json.dumps(line))
    D.done()
    return 0


if __name__ == "__main__":
    sys.exit(main())
