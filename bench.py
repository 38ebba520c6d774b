#!/usr/bin/env python
"""bench.py -- faces/sec of the RetinaFace mnet25 detect path on B200 (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--workload NAME] [--dump-outputs DIR]

One "step" = one pass of the hot path (u8 images -> conv0..SSH -> fused heads+decode -> NMS)
over one batch of synthetic S-real input (SURVEY.md 8d: the golden photo letter-boxed to the
network size, element i rolled by 8*i pixels so every image has faces but distinct content).

Printed JSON (rank 0, one line):
  value      faces/s, device-timed: inputs already resident in HBM (a ring of batches larger than
             2x L2 so that no step finds its input in L2), CUDA events on the library's stream,
             max over ranks, whole job (all GPUs).
  e2e        the same metric through the public C ABI with HOST (pinned) images: every step copies its own
             images H2D and reads its own faces back D2H inside the timed region -- rf_submit_batch /
             rf_collect_batch with several batches in flight (throughput mode); `e2e.blocking` is the same
             with one blocking rf_detect_batch per step (latency mode).
  roofline   dominant kernel: algorithmic bytes (layer-granular, SURVEY.md 8d) / CUDA-event time of
             that kernel launched K times on the library's stream, vs MEASURED_PEAKS.json.
  configs    the other BASELINE.json configurations measured in the same run (device-timed + end to end): batch 1 / 32,
             configs[2] INT8 batch 32, configs[3] 1280x896; at --gpus 8: configs[4] INT8 batch 32 per GPU + all-gather.
Timing: every number times exactly K steps, after W untimed warm-up steps of the same kind.  The default K = 4000 makes
the headline window about 0.3 s (77 us per step on a B200 at its 1000 W limit) and every other window at least as long,
except batch 1 (about 0.1 s); a much smaller K times a window of a few ms, which measures the clock and the scheduler as
much as the kernels.  At N > 1 every step -- device-timed and end to
end -- includes the exchange of the detection records (rf_detect_batch_device_allgather / rf_submit_batch_allgather:
fused into the NMS kernel, comm.cu).
  cpu_baseline  the oracle (cv2.dnn FP32 forward of the same caffemodel through a generated prototxt +
             oracle/postproc.c) timed on the host cores on a bounded sample (rank 0, N=1 only).

--impl reference runs only that CPU arm (the reference's own CPU path cannot be built here:
BVLC Caffe / OpenCV C++ / TensorRT are absent -- DESIGN.md), on the same config/metric/unit.

--dump-outputs DIR writes, after the timed steps of --workload, what its last device-timed step returned (rank 0; at N > 1
the gathered records of every rank): DIR/faces.npy (float32 [images][max_faces][15], FaceDetectInfo rows), DIR/anchor_index.npy
and DIR/counts.npy (float64 [images][max_faces] and [images]); entries past an image's count are 0 (-1 for the anchor index).
The inputs depend only on the arguments, so two builds can be compared output for output.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
GOLD = os.path.join(ROOT, "tests", "golden")

WORKLOADS = {
    # BASELINE.json configs[1]: the configuration the metric is quoted on
    "mnet25_fp16_b8_448": dict(model="mnet25", precision="fp16", batch=8, h=448, w=448),
    "mnet25_fp32_b8_448": dict(model="mnet25", precision="fp32", batch=8, h=448, w=448),
    "mnet25_fp16_b1_448": dict(model="mnet25", precision="fp16", batch=1, h=448, w=448),
    "mnet25_fp16_b32_448": dict(model="mnet25", precision="fp16", batch=32, h=448, w=448),
    # configs[2]: INT8 with the reference's TensorRT calibration table
    "mnet0517_int8_b32_448": dict(model="mnet-deconv-0517", precision="int8", batch=32, h=448, w=448),
    "mnet0517_int8_b8_448": dict(model="mnet-deconv-0517", precision="int8", batch=8, h=448, w=448),
    "mnet0517_fp16_b32_448": dict(model="mnet-deconv-0517", precision="fp16", batch=32, h=448, w=448),
    # configs[3]: large input / many-anchor NMS stress
    "mnet25_fp16_b8_1280x896": dict(model="mnet25", precision="fp16", batch=8, h=896, w=1280),
    # configs[4] per GPU (B=256 over 8 GPUs): the reference ships no mnet25 table -> mnet-deconv-0517 + its TensorRT table
    "mnet0517_int8_b32_448_per_gpu": dict(model="mnet-deconv-0517", precision="int8", batch=32, h=448, w=448),
}
EXTRA_1GPU = ["mnet25_fp16_b1_448", "mnet25_fp16_b32_448", "mnet0517_int8_b32_448", "mnet25_fp16_b8_1280x896"]
EXTRA_NGPU = ["mnet0517_int8_b32_448_per_gpu"]
DEFAULT_WORKLOAD = "mnet25_fp16_b8_448"
SCORE_THR, NMS_THR = 0.9, 0.4  # main.cpp:43, RetinaFace.h:66


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm_gbs=d["hbm_gbs"], bf16_tflops=d["bf16_tflops"], src="measured")
    return dict(hbm_gbs=6650.0, bf16_tflops=1590.0, src="fallback")


def make_batches(wl, count, rank):
    """`count` distinct S-real batches (u8 [count][B][H][W][3])."""
    import cv2
    from oracle.inputs import letterbox_bgr_u8
    img = cv2.imread(os.path.join(GOLD, "data", "img.jpg"))
    base = letterbox_bgr_u8(img, wl["h"], wl["w"])
    out = np.empty((count, wl["batch"], wl["h"], wl["w"], 3), dtype=np.uint8)
    for s in range(count):
        for i in range(wl["batch"]):
            out[s, i] = np.roll(base, 8 * (i + wl["batch"] * (s + count * rank)), axis=1)
    return out


def dump_device_outputs(out_dir, dets_ptr, counts_ptr, rows, max_faces, device):
    """Writes the records of one rf_detect_batch_device[_allgather] call (rows x max_faces rf_det of 64 bytes, rows int32
    counts; complete in device memory) to out_dir as faces / anchor_index / counts .npy files."""
    import torch

    class DeviceArray:
        def __init__(self, ptr, shape, typestr):
            self.__cuda_array_interface__ = dict(shape=shape, typestr=typestr, data=(ptr, False), version=2)

    rec = torch.as_tensor(DeviceArray(dets_ptr, (rows, max_faces, 64), "|u1"), device=device).cpu().numpy()
    counts = torch.as_tensor(DeviceArray(counts_ptr, (rows,), "<i4"), device=device).cpu().numpy()
    valid = np.arange(max_faces)[None, :] < counts[:, None]
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "faces.npy"), np.where(valid[..., None], rec.view(np.float32)[..., :15], 0).astype(np.float32))
    np.save(os.path.join(out_dir, "anchor_index.npy"), np.where(valid, rec.view(np.int32)[..., 15], -1).astype(np.float64))
    np.save(os.path.join(out_dir, "counts.npy"), counts.astype(np.float64))


class ClockSampler(threading.Thread):
    """SM clock + throttle reasons sampled DURING the timed region: NVML every 2 ms when pynvml can open the device (the
    timed region of the default run is ~0.3 s), else one `nvidia-smi` query per 100 ms.  Rows have nvidia-smi's layout."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu):
        super().__init__(daemon=True)
        self.gpu, self.rows, self.stop_ev = gpu, [], threading.Event()
        self.source = "nvidia-smi"

    def _nvml_loop(self) -> bool:
        try:
            import pynvml as nv
            nv.nvmlInit()
            vis = os.environ.get("CUDA_VISIBLE_DEVICES", "")
            idx = int(vis.split(",")[self.gpu]) if vis and all(x.strip().isdigit() for x in vis.split(",")) else self.gpu
            dev = nv.nvmlDeviceGetHandleByIndex(idx)
            mx = nv.nvmlDeviceGetMaxClockInfo(dev, nv.NVML_CLOCK_SM)
            get_reasons = getattr(nv, "nvmlDeviceGetCurrentClocksEventReasons", None) or nv.nvmlDeviceGetCurrentClocksThrottleReasons
            bits = [nv.nvmlClocksThrottleReasonHwSlowdown, nv.nvmlClocksThrottleReasonHwThermalSlowdown,
                    nv.nvmlClocksThrottleReasonSwThermalSlowdown, nv.nvmlClocksThrottleReasonSwPowerCap]
            nv.nvmlDeviceGetClockInfo(dev, nv.NVML_CLOCK_SM)          # probe once before committing to this source
        except Exception:
            return False
        self.source = "nvml"
        while not self.stop_ev.is_set():
            try:
                sm = nv.nvmlDeviceGetClockInfo(dev, nv.NVML_CLOCK_SM)
                r = int(get_reasons(dev))
                self.rows.append([str(sm), str(mx)] + ["Active" if r & b else "Not Active" for b in bits])
            except Exception:
                pass
            self.stop_ev.wait(0.002)
        return True

    def run(self):
        if self._nvml_loop():
            return
        while not self.stop_ev.is_set():
            try:
                o = subprocess.run(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-i", str(self.gpu)],
                                   capture_output=True, text=True, timeout=5).stdout.strip()
                if o:
                    self.rows.append([x.strip() for x in o.split(",")])
            except Exception:
                pass
            self.stop_ev.wait(0.1)

    def summary(self):
        self.stop_ev.set()
        self.join(timeout=6)
        sm = [float(r[0]) for r in self.rows if r and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for r in self.rows for i in range(4) if len(r) > 2 + i and r[2 + i].lower().startswith("active")})
        return dict(sm_mhz=float(np.median(sm)) if sm else None, sm_max_mhz=max(mx) if mx else None, reasons=reasons,
                    samples=len(self.rows), source=self.source)


# ------------------------------------------------------------------------------------------------
# CPU arm (oracle; the reference's own CPU-Caffe path is unbuildable here)
# ------------------------------------------------------------------------------------------------
class CpuPath:
    def __init__(self, wl, threads):
        import cv2
        import tempfile
        from oracle import topology
        from oracle.postproc import PostprocOracle
        cv2.setNumThreads(threads)
        self.cv2, self.topology, self.wl = cv2, topology, wl
        d = tempfile.mkdtemp()
        p = os.path.join(d, "oracle.prototxt")
        open(p, "w").write(topology.to_prototxt(wl["h"], wl["w"], wl["batch"]))
        self.net = cv2.dnn.readNetFromCaffe(p, os.path.join(GOLD, "weights", wl["model"] + ".caffemodel"))
        self.post = PostprocOracle()
        self.threads = threads

    def step(self, batch_u8):
        """RetinaFace::detect on the CPU: u8->f32 RGB planar, forward, decode+NMS.  Returns #faces."""
        x = np.ascontiguousarray(batch_u8[..., ::-1].transpose(0, 3, 1, 2), dtype=np.float32)
        self.net.setInput(x)
        outs = self.net.forward(self.topology.OUTPUT_BLOBS)
        faces = 0
        for i in range(batch_u8.shape[0]):
            r = self.post.postprocess([o[i] for o in outs], self.wl["h"], self.wl["w"], SCORE_THR, NMS_THR)
            faces += len(r["faces"])
        return faces


def best_cpu_threads(wl, batch):
    """cv2.dnn does not scale to every core of a big host: time one batch at a few thread counts and keep the
    fastest, so the CPU arm runs 'with all the host threads it can use' rather than with all that exist."""
    ncpu = os.cpu_count() or 1
    cands = sorted({t for t in (ncpu, ncpu // 2, 64, 32, 16, 8) if 1 <= t <= ncpu}, reverse=True)
    best, best_t = cands[0], float("inf")
    for t in cands:
        cpu = CpuPath(wl, t)
        cpu.step(batch)
        t0 = time.perf_counter()
        cpu.step(batch)
        dt = time.perf_counter() - t0
        if dt < best_t:
            best, best_t = t, dt
    return best


def cpu_measure(wl, batches, budget_s, min_steps=2, threads=None):
    threads = threads or best_cpu_threads(wl, batches[0])
    cpu = CpuPath(wl, threads)
    cpu.step(batches[0])  # warm-up
    t0 = time.perf_counter()
    faces = steps = 0
    while (time.perf_counter() - t0 < budget_s or steps < min_steps) and steps < 10_000:
        faces += cpu.step(batches[steps % len(batches)])
        steps += 1
    dt = time.perf_counter() - t0
    B = batches[0].shape[0]
    return dict(value=faces / dt, unit="faces/s", cores=threads, kind="port",
                sample=f"{steps} batches of {B} images ({steps * B} images, {dt:.1f} s): cv2.dnn FP32 forward "
                       f"of {wl['model']}.caffemodel + oracle/postproc.c decode/NMS, {threads} threads",
                images_per_s=steps * B / dt, ms_per_batch=dt / steps * 1e3), dt, steps


# ------------------------------------------------------------------------------------------------
_REAL_STDOUT = None


def emit(line: dict) -> None:
    """The ONE JSON line goes to the real stdout; everything else this process (or NCCL / a library) prints was
    redirected to stderr at start-up, so stdout carries exactly one line."""
    data = (json.dumps(line) + "\n").encode()
    if _REAL_STDOUT is None:
        sys.stdout.write(data.decode())
        sys.stdout.flush()
    else:
        os.write(_REAL_STDOUT, data)


def main():
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)            # e.g. "NCCL version ..." banners must not precede the JSON line
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=4000)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default=DEFAULT_WORKLOAD, choices=sorted(WORKLOADS))
    ap.add_argument("--cpu-seconds", type=float, default=12.0, help="budget of the cpu_baseline sample")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extra-configs", action="store_true", help="measure only --workload (skip the `configs` dict)")
    ap.add_argument("--streams", type=int, default=0, help="execution contexts of the engine (0 = library default 2)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the outputs of the last device-timed step of --workload to DIR/*.npy (--impl b200 only)")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of the b200 path only; it cannot be combined with --impl reference")
    wl = dict(WORKLOADS[args.workload])
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    K, W = args.steps, max(args.warmup, 3)
    config = dict(workload=args.workload, model=wl["model"] + ".caffemodel (reference weights)", precision=wl["precision"],
                  batch_per_gpu=wl["batch"], global_batch=wl["batch"] * world, input=f"{wl['w']}x{wl['h']}",
                  score_thr=SCORE_THR, nms_thr=NMS_THR, parallelism=f"dp{world}", input_data="S-real: golden photo letter-boxed, rolled 8*i px")

    if args.impl == "reference":
        # the reference arm: CPU path, rank 0 only
        if rank != 0:
            return
        sample = make_batches(wl, 4, 0)
        cpu = CpuPath(wl, best_cpu_threads(wl, sample[0]))
        for _ in range(min(W, 3)):
            cpu.step(sample[0])
        # each step = one batch; bound the run to a few minutes
        t0 = time.perf_counter()
        faces = 0
        steps = 0
        for s in range(K):
            faces += cpu.step(sample[s % len(sample)])
            steps += 1
            if time.perf_counter() - t0 > 150:
                break
        dt = time.perf_counter() - t0
        v = faces / dt
        line = dict(metric="faces/sec (end-to-end detect)", value=v, unit="faces/s", n_gpus=args.gpus, steps=steps, warmup=W,
                    ms_per_step=dt / steps * 1e3, higher_is_better=True, scaling="weak", vs_baseline=None, dtype="f32",
                    data="synthetic", impl="reference", config=config, images_per_s=steps * wl["batch"] / dt,
                    cpu_baseline=dict(value=v, unit="faces/s", cores=cpu.threads, kind="port",
                                      sample=f"{steps} steps x {wl['batch']} images: cv2.dnn FP32 forward + oracle/postproc.c "
                                             "(the reference's CPU-Caffe path cannot be built: Caffe/OpenCV C++ absent)"),
                    e2e=dict(value=v, unit="faces/s", h2d_bytes_per_step=0, d2h_bytes_per_step=0), gpu_launches=0)
        emit(line)
        return

    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench.py --impl b200 needs a CUDA device: the path has no CPU fallback")
    torch.cuda.set_device(local)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    from retinaface_b200 import RF_PREC_FP16, RF_PREC_FP32, RF_PREC_INT8, Engine
    from retinaface_b200.capi import PIPELINE_DEPTH as depth
    from retinaface_b200.multigpu import init_comm
    precs = {"fp16": RF_PREC_FP16, "fp32": RF_PREC_FP32, "int8": RF_PREC_INT8}
    l2_bytes = 126 * 2**20

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def agree_max(x):
        if world == 1:
            return x
        t = torch.tensor([float(x)], dtype=torch.float64, device=f"cuda:{local}")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t[0])

    def agree_sum(x):
        if world == 1:
            return x
        t = torch.tensor([float(x)], dtype=torch.float64, device=f"cuda:{local}")
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        return float(t[0])

    def measure(name, full):
        """One workload on this rank's GPU: device-timed and end-to-end numbers, each over K timed steps after W warm-up steps."""
        w = dict(WORKLOADS[name])
        prec = precs[w["precision"]]
        B, H, Wd = w["batch"], w["h"], w["w"]
        eng = Engine(os.path.join(GOLD, "weights", w["model"] + ".caffemodel"), H, Wd, precision=prec, max_batch=B,
                     max_faces=128, device=local, streams=args.streams,
                     int8_table=os.path.join(GOLD, "weights", w["model"] + ".table.int8") if prec == RF_PREC_INT8 else None)
        if world > 1:
            init_comm(eng, dist, rank, world, local)
        gather = world > 1
        stream = torch.cuda.ExternalStream(eng.stream_ptr(), device=local)
        img_bytes = B * H * Wd * 3
        ring = max(4, min(256, -(-2 * l2_bytes // img_bytes)))     # input ring > 2 x L2
        host = make_batches(w, ring, rank)
        pinned = torch.from_numpy(host).pin_memory()
        dev = pinned.to(f"cuda:{local}", non_blocking=False)       # device-resident inputs for `value`
        pin_np = pinned.numpy()
        rows = world * B if gather else B
        fbuf = np.empty((rows, eng.max_faces, 15), dtype=np.float32)
        cbuf = np.zeros(rows, dtype=np.int32)

        def pipelined(nsteps, first):
            inflight, nfaces = [], 0
            for i in range(nsteps):
                if len(inflight) == depth:
                    _, c = eng.collect(inflight.pop(0), fbuf, cbuf)
                    nfaces += int(c[rank * B:(rank + 1) * B].sum()) if gather else int(c.sum())
                slot = (first + i) % ring
                inflight.append(eng.submit([pin_np[slot, j] for j in range(B)], SCORE_THR, NMS_THR, allgather=gather))
            while inflight:
                _, c = eng.collect(inflight.pop(0), fbuf, cbuf)
                nfaces += int(c[rank * B:(rank + 1) * B].sum()) if gather else int(c.sum())
            return nfaces

        # faces per ring slot (deterministic; the end-to-end path is also the warm-up of the engine)
        faces_per_slot = np.zeros(ring, dtype=np.int64)
        barrier()
        for s in range(ring):
            faces_per_slot[s] = pipelined(1, s)
        barrier()

        def device_step(slot):
            if gather:
                return eng.detect_device_allgather(B, SCORE_THR, NMS_THR, dev[slot].data_ptr())
            return eng.detect_device(B, SCORE_THR, NMS_THR, dev[slot].data_ptr())

        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        pos = [0]
        last = [None]                       # device (dets, counts) of the last device step

        def dev_block(n):
            barrier()
            ev0.record(stream)
            for _ in range(n):
                last[0] = device_step(pos[0] % ring)
                pos[0] += 1
            eng.fence()                     # stream (context 0) now follows the work queued on every context
            ev1.record(stream)
            barrier()
            return ev0.elapsed_time(ev1)

        def e2e_block(n):
            barrier()
            t0 = time.perf_counter()
            pipelined(n, pos[0])
            pos[0] += n
            barrier()
            return (time.perf_counter() - t0) * 1e3

        lat = [None]

        def blk_block(n):
            barrier()
            t0 = time.perf_counter()
            for _ in range(n):
                lat[0].detect_batch([pin_np[pos[0] % ring, j] for j in range(B)], SCORE_THR, NMS_THR)
                pos[0] += 1
            barrier()
            return (time.perf_counter() - t0) * 1e3

        def timed(block):
            """W untimed warm-up steps, then exactly K timed steps: their time in ms (max over ranks)."""
            block(W)
            return agree_max(block(K))

        mean_faces = float(faces_per_slot.mean())          # per step on this rank (the ring is walked round and round)
        faces_step = agree_sum(mean_faces)                 # whole job
        out = dict(workload=name, precision=w["precision"], batch_per_gpu=B, input=f"{Wd}x{H}", launches_per_step=eng.launches_per_batch(B))
        clock = None
        if full:
            clock = ClockSampler(local)
            clock.start()
        d_ms = timed(dev_block)
        out.update(ms_per_step=d_ms / K, value=faces_step * K / (d_ms * 1e-3), images_per_s=K * B * world / (d_ms * 1e-3), timed_region_s=d_ms * 1e-3)
        if full and args.dump_outputs and rank == 0:
            eng.synchronize()
            dump_device_outputs(args.dump_outputs, *last[0], rows, eng.max_faces, f"cuda:{local}")
        e_ms = timed(e2e_block)
        out["e2e"] = dict(value=faces_step * K / (e_ms * 1e-3), unit="faces/s", h2d_bytes_per_step=img_bytes,
                          d2h_bytes_per_step=(world if gather else 1) * (B * 4 + B * eng.max_faces * 64) + (4 if gather else 0),
                          images_per_s=K * B * world / (e_ms * 1e-3), ms_per_step=e_ms / K, timed_region_s=e_ms * 1e-3,
                          timing=f"host wall clock over {K} rf_submit_batch{'_allgather' if gather else ''}/rf_collect steps, {depth} batches in flight"
                                 + ("; every step's results are the records of ALL ranks, host-visible" if gather else ""))
        if full and not gather:
            # latency mode is its own handle configuration: streams = 1 selects the chain plan (DESIGN.md section 3)
            lat[0] = Engine(os.path.join(GOLD, "weights", w["model"] + ".caffemodel"), H, Wd, precision=prec, max_batch=B, max_faces=128, device=local,
                            streams=1, int8_table=os.path.join(GOLD, "weights", w["model"] + ".table.int8") if prec == RF_PREC_INT8 else None)
            b_ms = timed(blk_block)
            out["e2e"]["blocking"] = dict(value=faces_step * K / (b_ms * 1e-3), ms_per_step=b_ms / K, images_per_s=K * B * world / (b_ms * 1e-3),
                                          launches_per_step=lat[0].launches_per_batch(B),
                                          note="one blocking rf_detect_batch per step on a streams=1 handle (latency mode: chain plan)")
            lat[0].close()
        if clock is not None:
            out["clocks"] = clock.summary()
        if full and rank == 0:
            out["_prof"] = eng.profile_layers(B, iters=max(10, min(K, 100)))
        out["_ring"] = ring
        out["_img_bytes"] = img_bytes
        out["_max_faces"] = eng.max_faces
        eng.close()
        return out

    main_res = measure(args.workload, True)
    extras = {}
    if not args.no_extra_configs:
        for name in (EXTRA_NGPU if world > 1 else EXTRA_1GPU):
            if name == args.workload:
                continue
            try:
                r = measure(name, False)
                extras[name] = {k: v for k, v in r.items() if not k.startswith("_")}
            except Exception as e:                      # a secondary configuration must not take the headline line down
                extras[name] = dict(error=str(e)[:300])

    line = None
    if rank == 0:
        pk = peaks()
        prec = precs[wl["precision"]]
        prof = main_res.pop("_prof")
        ring, img_bytes, mfaces = main_res.pop("_ring"), main_res.pop("_img_bytes"), main_res.pop("_max_faces")
        # ---- roofline of the dominant kernel (direct launches, CUDA events on the library stream) ----
        tot = sum(p["ms"] for p in prof)
        top = max(prof, key=lambda p: p["ms"])
        ach_gbs = top["bytes"] / (top["ms"] * 1e-3) / 1e9
        ach_tf = top["flops"] / (top["ms"] * 1e-3) / 1e12
        traffic, l2b, limiter, tsrc = None, None, None, None
        tp = os.path.join(ROOT, "profiles", "r02_traffic.json")
        if os.path.exists(tp):            # the committed ncu --set full capture of this kernel (not re-measured in this run)
            tj = json.load(open(tp))
            if tj.get("workload") == args.workload and tj.get("kernel") == top["name"]:
                traffic = tj["dram_bytes_read"] + tj["dram_bytes_write"]
                l2b, limiter, tsrc = tj.get("l2_bytes"), tj.get("limiter"), "profiles/r02_traffic.json (ncu --set full capture; file-sourced, not measured in this run)"
        roof = dict(bound="hbm", kernel=top["name"], achieved=ach_gbs, peak=pk["hbm_gbs"], unit="GB/s", frac=ach_gbs / pk["hbm_gbs"],
                    traffic=traffic, traffic_source=tsrc, l2_bytes=l2b, limiter=limiter, peak_source=pk["src"], kernel_ms=top["ms"],
                    kernel_share_of_step=top["ms"] / tot, tensor_tflops=ach_tf, tensor_frac=ach_tf / pk["bf16_tflops"],
                    step_algorithmic_gb=sum(p["bytes"] for p in prof) / 1e9, step_algorithmic_gflop=sum(p["flops"] for p in prof) / 1e9,
                    step_sum_of_kernels_ms=tot,
                    note="kernel time: back-to-back launches of that kernel alone (L2-warm); algorithmic bytes = its input + output tensors")
        line = dict(metric="faces/sec (end-to-end detect)", value=main_res["value"], unit="faces/s", n_gpus=world, steps=K, warmup=W,
                    ms_per_step=main_res["ms_per_step"], higher_is_better=True, scaling="weak", vs_baseline=None,
                    dtype={RF_PREC_FP16: "f16", RF_PREC_FP32: "f32", RF_PREC_INT8: "s8"}[prec], data="synthetic",
                    config=dict(config, execution_contexts=args.streams or 8,
                                l2_policy=f"input ring of {ring} batches = {ring * img_bytes / 2**20:.0f} MiB > 2x L2; activations reused in place",
                                timing=f"{K} timed steps after {W} warm-up steps ({main_res['timed_region_s']:.3f} s timed)",
                                exchange=("detection records of every step stored into every rank's gather window by the NMS kernel (NVLink peer "
                                          "stores, comm.cu); included in value and e2e") if world > 1 else "none (1 GPU)"),
                    images_per_s=main_res["images_per_s"], clocks=main_res.get("clocks"),
                    e2e=main_res["e2e"], gpu_launches=K * main_res["launches_per_step"], launches_per_step=main_res["launches_per_step"],
                    roofline=roof, layers=[dict(name=p["name"], us=round(p["ms"] * 1e3, 2)) for p in prof], configs=extras)
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        host = make_batches(wl, 4, 0)
        cb, _, _ = cpu_measure(wl, host, args.cpu_seconds)
        one, _, _ = cpu_measure(wl, host, max(3.0, args.cpu_seconds / 3), threads=1)
        w1 = dict(wl, batch=1)
        single = make_batches(w1, 4, 0)
        s_all, _, _ = cpu_measure(w1, single, max(3.0, args.cpu_seconds / 4), threads=cb["cores"])
        s_one, _, _ = cpu_measure(w1, single, max(3.0, args.cpu_seconds / 4), threads=1)
        cb["one_core"] = dict(value=one["value"], images_per_s=one["images_per_s"], ms_per_batch=one["ms_per_batch"], cores=1)
        cb["single_image"] = dict(note="BASELINE.json configs[0]: one 448x448 image per call (mnet25 FP32, CPU only)",
                                  all_cores=dict(value=s_all["value"], ms_per_image=s_all["ms_per_batch"], cores=s_all["cores"]),
                                  one_core=dict(value=s_one["value"], ms_per_image=s_one["ms_per_batch"], cores=1))
        cb["host"] = dict(nproc=os.cpu_count())
        line["cpu_baseline"] = cb
    elif rank == 0:
        line["cpu_baseline"] = None
    if rank == 0:
        emit(line)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
