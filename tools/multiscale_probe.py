"""Multi-scale evaluation of one Potsdam tile: the host composition against the device pass, wall time from call to label map.

    python tools/multiscale_probe.py [--size 6000] [--runs 3] [--out FILE]

Workload: a 6000 x 6000 x 5 float64 Potsdam-shaped tile (synth), dilated_grsl_rate8 in f16, three scales (crops 25, 45,
65, the order validate_test_multiscale would take them in), batch 16.

    host    GpuBackend.scene_mean_logits per scale (the float64 [H, W, K] mean map copied to the host), then NumPy as
            loops.isprs_validate_test_multiscale composes it: astype(float32), reference_softmax, np.sum over the scales,
            np.argmax
    device  GpuBackend.scene_multiscale_labels: the passes, softmax, sum and argmax on the device, the uint8 map copied back

Each path runs once to warm up, then `runs` times, alternating; the median of each is reported.  The two label maps must be
equal.  The card's name and power limit are read in the same run.  Prints one JSON line (also written to --out).
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def card():
    r = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                       text=True)
    name, limit = (x.strip() for x in r.stdout.strip().splitlines()[0].split(","))
    return name, limit


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--size", type=int, default=6000)
    ap.add_argument("--runs", type=int, default=3)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    import drs_b200
    from drs_b200 import backend, loops, synth
    assert torch.cuda.is_available(), "the probe needs a GPU"
    crops, batch, K = [25, 45, 65], 16, 6
    img, lab = synth.scene("potsdam", H=a.size, W=a.size)
    mean, std = synth.normalisation(img)
    s = drs_b200.Session("dilated_grsl_rate8", 5, K, precision="f16", seed=9)
    be = backend.GpuBackend(s, [img], [lab], mean, std)
    H, W = a.size, a.size

    def host_path():
        mean_prob = np.zeros([len(crops), H, W, K], dtype=np.float32)
        for i, c in enumerate(crops):
            mean_prob[i] = be.scene_mean_logits(0, c, batch)
            mean_prob[i, :, :, :] = loops.reference_softmax(mean_prob[i, :, :, :], K)
        return np.argmax(np.sum(mean_prob, axis=0), axis=2)

    def device_path():
        return be.scene_multiscale_labels(0, crops, batch)

    times = {"host": [], "device": []}
    maps = {}
    for it in range(a.runs + 1):
        for name, fn in (("host", host_path), ("device", device_path)):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            maps[name] = fn()
            dt = time.perf_counter() - t0
            if it > 0:
                times[name].append(dt)
    equal = bool(np.array_equal(maps["host"], maps["device"]))
    gpu, power_limit = card()
    res = {"probe": "multiscale", "gpu": gpu, "power_limit": power_limit, "H": H, "W": W, "C": 5, "dtype": "float64",
           "net": "dilated_grsl_rate8", "precision": "f16", "crops": crops, "batch": batch, "runs": a.runs,
           "host_s": float(np.median(times["host"])), "device_s": float(np.median(times["device"])),
           "host_runs_s": [round(t, 3) for t in times["host"]], "device_runs_s": [round(t, 3) for t in times["device"]],
           "labels_equal": equal}
    res["host_over_device"] = res["host_s"] / res["device_s"]
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")
    s.close()
    if not equal:
        sys.exit("label maps differ")


if __name__ == "__main__":
    main()
