#!/usr/bin/env python
"""Cost of the aligned face crops (rf_detect_align_batch / rf_align_batch_device): mnet25 FP16 at 448x448, batch 8 of 1280x886
photos (S-real: the golden photo rolled by 8 px per image), max_crops 16, 112 x 112 u8 BGR crops.  Measures, in one process:

* align kernel device time: CUDA events around R back-to-back rf_align_batch_device launches on fixed records (one
  rf_detect_batch_device of the letter-boxed batch), sampling the network-sized device images;
* blocking call time of rf_detect_batch against rf_detect_align_batch on the original photos, alternated call by call;
* bytes the kernel moves (crops written + bilinear taps read, 4 taps x 3 bytes per crop pixel, from the face counts) over its time.

Prints one JSON line (and writes it to --out) with the card's name and power limit read in the same run."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def card():
    import torch
    info = {"name": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"], capture_output=True,
                           text=True, timeout=30).stdout.strip()
        info["power_limit"], info["max_sm_clock"] = [s.strip() for s in q.split(",")[:2]]
    except Exception as e:  # noqa: BLE001
        info["power_limit"] = "unread: %s" % str(e)[:80]
    return info


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=2000, help="kernel launches in the event-timed window")
    ap.add_argument("--calls", type=int, default=200, help="blocking calls of each entry point")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import cv2
    import torch
    from oracle.inputs import letterbox_bgr_u8, s_real_batch
    from retinaface_b200 import RF_PREC_FP16, Engine, align_spec
    gold = os.path.join(ROOT, "tests", "golden")
    img = cv2.imread(os.path.join(gold, "data", "img.jpg"))
    B, MC, CROP = 8, 16, 112
    photos = list(s_real_batch(img, B))
    eng = Engine(os.path.join(gold, "weights", "mnet25.caffemodel"), 448, 448, precision=RF_PREC_FP16, max_batch=B, max_image=(896, 1280))
    out = {"tool": "tools/align_rate.py", "card": card(), "model": "mnet25 FP16 448x448", "batch": B, "image": "1280x886",
           "max_crops": MC, "crop": "112x112 u8 BGR", "thr": 0.5, "nms": 0.4}

    # ---- kernel time on fixed records --------------------------------------------------------------------------------------
    net = torch.from_numpy(np.stack([letterbox_bgr_u8(p, 448, 448) for p in photos])).cuda()
    crops = torch.empty((B, MC, CROP, CROP, 3), dtype=torch.uint8, device="cuda")
    torch.cuda.synchronize()
    dets, counts = eng.detect_device(B, 0.5, 0.4, net.data_ptr())
    spec = align_spec((CROP, CROP), max_crops=MC)
    stream = torch.cuda.ExternalStream(eng.last_stream_ptr())
    for _ in range(50):
        eng.align_device(B, net.data_ptr(), dets, counts, crops.data_ptr(), spec)
    eng.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for _ in range(args.reps):
        eng.align_device(B, net.data_ptr(), dets, counts, crops.data_ptr(), spec)
    e1.record(stream)
    e1.synchronize()
    kernel_us = e0.elapsed_time(e1) * 1e3 / args.reps
    faces = eng.detect_batch([p for p in np.asarray(net.cpu())], 0.5, 0.4)
    ncrops = int(sum(min(len(f), MC) for f in faces))
    px = ncrops * CROP * CROP
    bytes_out, bytes_taps = px * 3, px * 4 * 3
    out["kernel"] = {"us_per_launch": kernel_us, "crops": ncrops, "crops_per_image": [int(min(len(f), MC)) for f in faces],
                     "bytes_written": bytes_out, "tap_bytes_read": bytes_taps,
                     "GB_per_s": (bytes_out + bytes_taps) / (kernel_us * 1e-6) / 1e9, "launches_timed": args.reps,
                     "note": "event-timed back-to-back launches on one stream; the source images (4.8 MB) and crops stay in L2"}

    # ---- blocking calls: rf_detect_batch vs rf_detect_align_batch, alternated -------------------------------------------------
    for _ in range(10):
        eng.detect_batch(photos, 0.5, 0.4)
        eng.detect_align(photos, 0.5, 0.4, max_crops=MC)
    t_det, t_al = [], []
    for _ in range(args.calls):
        t0 = time.perf_counter()
        eng.detect_batch(photos, 0.5, 0.4)
        t1 = time.perf_counter()
        per, _ = eng.detect_align(photos, 0.5, 0.4, max_crops=MC)
        t2 = time.perf_counter()
        t_det.append(t1 - t0)
        t_al.append(t2 - t1)
    med = lambda v: float(np.median(v)) * 1e3  # noqa: E731
    out["blocking_ms"] = {"rf_detect_batch": med(t_det), "rf_detect_align_batch": med(t_al), "difference": med(t_al) - med(t_det),
                          "p10_p90_detect": [float(np.percentile(t_det, 10)) * 1e3, float(np.percentile(t_det, 90)) * 1e3],
                          "p10_p90_align": [float(np.percentile(t_al, 10)) * 1e3, float(np.percentile(t_al, 90)) * 1e3],
                          "calls_each": args.calls, "crops_per_call": int(sum(len(p[1]) for p in per)),
                          "note": "host clock around each blocking call (pageable 1280x886 sources, H2D + letter-box + forward + D2H); "
                                  "the align call adds the kernel and the D2H of the crops that exist"}
    eng.close()
    line = json.dumps(out)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
