#!/usr/bin/env python
"""bench.py -- the hot path's headline metrics on B200 (contract: see the task statement / DESIGN.md section 6).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload train|infer] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

Default workload = BASELINE.json configs[1]: dilated_grsl (Dilated6Pooling), multinomial patch sizes
{25,29,...,49}, update_type acc, batch 64 per GPU, Vaihingen-shaped synthetic scene resident in HBM.
One "step" = the reference's training iteration (isprs:1726-1763): draw a patch size, select the batch, gather +
normalise the patches, sess.run([optimizer, loss, pred_up]) (forward, backward, exchange, momentum update),
per-crop confusion matrix, score update.  metric = train patches/s (whole job).
The same JSON line carries the second headline metric as "inference": full-scene sliding-window inference of a
Potsdam-shaped 6000x6000x5 scene with dilated_grsl_rate8 (configs[3]) in Mpixel/s.

--impl reference times the reference-equivalent CPU path (TensorFlow is not installable here: the oracle's
PyTorch-CPU restatement of the graph + the NumPy restatement of the host loops) on a bounded sample.

--dump-outputs DIR writes, after the timed steps, what the timed path computed in its last timed step as DIR/<name>.npy
(float32 / float64, rank 0 only), so that two builds can be compared output for output on the same seeded inputs:
  train_loss, train_confusion, train_n_correct, train_pred   what the training step returns (loss, per-crop confusion
                                                               matrix, correct pixels, predicted labels [B, crop, crop])
  train_var__<scope>__<name>                                   every variable and momentum slot after that step
  infer_label_counts                                           pixels per class of the last timed scene pass's label map
  infer_labels_sample, infer_labels_sample_index               2^20 of its pixels at fixed seeded flat indices
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

TRAIN_CFG = dict(net="dilated_grsl", dataset="vaihingen", C=4, K=6, batch=64, values=[25, 29, 33, 37, 41, 45, 49],
                 distribution="multinomial", update="acc", lr=0.01, wd=0.005)
INFER_CFG = dict(net="dilated_grsl_rate8", dataset="potsdam", C=5, K=6, crop=25, batch=64, H=6000, W=6000)


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm=d["hbm_gbs"], tc_burst=d["bf16_tflops"], tc_sustained=d["bf16_tflops_sustained"], source="measured")
    return dict(hbm=6650.0, tc_burst=1590.0, tc_sustained=1400.0, source="fallback")


class ClockSampler:
    """SM clock / power / throttle reasons DURING the timed region (B200_PROFILING.md) through NVML.  The thread is started
    well before the region (NVML initialisation and the first queries take a driver lock that kernel launches also need: inside
    a 40 ms region they cost up to a second) and polls every 25 ms; begin() / stop() mark the region and only the samples between
    them are reported (the nearest one if the region was shorter than a period).  Falls back to one nvidia-smi query."""
    PERIOD = 0.025

    def __init__(self, index):
        self.index, self.samples, self.stop_flag, self.thread, self.nv = index, [], False, None, None
        self.t_begin = self.t_end = None

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.handle = pynvml.nvmlDeviceGetHandleByIndex(self.index)
            self._query()
            self.thread = threading.Thread(target=self._loop, daemon=True)
            self.thread.start()
        except Exception:
            self.nv = None

    def _query(self):
        nv = self.nv
        sm = nv.nvmlDeviceGetClockInfo(self.handle, nv.NVML_CLOCK_SM)
        pw = nv.nvmlDeviceGetPowerUsage(self.handle) / 1000.0
        rs = nv.nvmlDeviceGetCurrentClocksEventReasons(self.handle) if hasattr(nv, "nvmlDeviceGetCurrentClocksEventReasons") \
            else nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.handle)
        return (time.perf_counter(), sm, pw, rs)

    def _loop(self):
        while not self.stop_flag:
            try:
                self.samples.append(self._query())
            except Exception:
                pass
            time.sleep(self.PERIOD)

    def begin(self):
        self.t_begin = time.perf_counter()

    def stop(self):
        self.t_end = time.perf_counter()
        if self.nv is None:
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=clocks.sm,clocks.max.sm,power.draw",
                                      "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=10).stdout.split(",")
                return {"sm_mhz": float(out[0]), "sm_max_mhz": float(out[1]), "power_w_max": float(out[2]), "samples": 1,
                        "reasons": [], "note": "single nvidia-smi sample after the timed region (NVML unavailable)"}
            except Exception:
                return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.stop_flag = True
        self.thread.join(timeout=1.0)
        nv = self.nv
        try:
            mx = float(nv.nvmlDeviceGetMaxClockInfo(self.handle, nv.NVML_CLOCK_SM))
        except Exception:
            mx = None
        t0 = self.t_begin if self.t_begin is not None else 0.0
        inside = [x for x in self.samples if t0 <= x[0] <= self.t_end]
        note = None
        if not inside and self.samples:
            mid = 0.5 * (t0 + self.t_end)
            inside = [min(self.samples, key=lambda x: abs(x[0] - mid))]
            note = "timed region shorter than the %.0f ms polling period: nearest sample" % (self.PERIOD * 1e3)
        names = {"hw_slowdown": 0x8, "sw_power_cap": 0x4, "hw_thermal_slowdown": 0x40, "sw_thermal_slowdown": 0x20,
                 "hw_power_brake_slowdown": 0x80}
        reasons = set()
        for _, _, _, r in inside:
            for k, bit in names.items():
                if r & bit:
                    reasons.add(k)
        sm = [x[1] for x in inside]
        out = {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx,
               "power_w_max": max([x[2] for x in inside]) if inside else None, "samples": len(sm), "reasons": sorted(reasons)}
        if note:
            out["note"] = note
        return out


def profiled_traffic(which):
    """DRAM bytes per launch of the dominant kernel from the committed ncu --set full capture (profiles/)."""
    for name in ("r2c_traffic.json", "r2_traffic.json"):          # newest capture first
        try:
            return float(json.load(open(os.path.join(ROOT, "profiles", name)))[which]["dram_bytes_per_launch"])
        except Exception:
            continue
    return None


def dist_env():
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    return rank, world, local


# ----------------------------------------------------------------------------------------------------------------
# the workload both arms run: the drop-in training loop (loops.isprs_train == isprs:1621-1851) on one synthetic scene
# ----------------------------------------------------------------------------------------------------------------
SEED = 77


def isprs_workload(cfg, test_hw=(300, 300)):
    """What isprs_dilated_random.py builds before it calls train (isprs:2066-2115), on a synthetic Vaihingen-shaped scene:
    class distributions, rotation table, normalisation, score arrays -- under the seeds both arms share."""
    import random
    from drs_b200 import host, synth
    img, lab = synth.scene(cfg["dataset"])
    timg, tlab = synth.scene(cfg["dataset"], H=test_hw[0], W=test_hw[1], seed=4321)
    np.random.seed(SEED)
    random.seed(SEED)
    tr_distr = host.create_distributions_over_classes([lab], 25, 25, cfg["K"], verbose=False)
    te_distr = host.create_distributions_over_classes([tlab], 25, 25, cfg["K"], verbose=False)
    rot = host.create_rotation_distribution(tr_distr, verbose=False)
    mean, std = synth.normalisation(img)
    values = cfg["values"]
    probs = host.define_multinomial_probs(values) if cfg["distribution"] == "multinomial" else None
    pal, occ, chosen = host.init_score_arrays(cfg["distribution"], values)
    return dict(train_data=[img], train_labels=[lab], test_data=[timg], test_labels=[tlab], tr_distr=tr_distr, te_distr=te_distr,
                rot=rot, mean=mean, std=std, probs=probs, pal=pal, occ=occ, chosen=chosen)


def run_isprs_loop(backend, wl, cfg, batch_size, niter, hook, depth=None):
    """loops.isprs_train with the log lines discarded (the JSON line must be the only output) and its cache/checkpoint files in
    a scratch directory; display / epoch / validation intervals beyond niter, so that every iteration is a plain training step."""
    import contextlib
    import tempfile
    from drs_b200 import loops
    far = 10 ** 9
    cwd = os.getcwd()
    if depth is not None:
        os.environ["DRS_PREFETCH"] = str(depth)
    with tempfile.TemporaryDirectory() as tmp, open(os.devnull, "w") as null:
        os.chdir(tmp)
        try:
            with contextlib.redirect_stdout(null):
                loops.isprs_train(backend, wl["train_data"], wl["train_labels"], wl["tr_distr"], wl["rot"], wl["test_data"],
                                  wl["test_labels"], wl["te_distr"], ["t"], batch_size, niter, cfg["update"], cfg["distribution"],
                                  cfg["values"], wl["pal"], wl["occ"], wl["chosen"], wl["probs"], 20, tmp + "/", far, "bench", "",
                                  cfg["K"], epoch_number=far, val_inteval=far, final_validation=False, step_hook=hook)
        finally:
            os.chdir(cwd)


def conv_flops_train(net, C, K, M):
    """Algorithmic FLOPs of one training step: fprop + dgrad + wgrad of every conv, minus conv1's dgrad."""
    from drs_b200 import nets
    plan, cls_in = nets.layer_plan(net, C)
    macs = 0
    for i, (_, k, r, ci, co) in enumerate(plan):
        macs += k * k * ci * co * (3 if i > 0 else 2)
    macs += 3 * cls_in * K
    return 2.0 * macs * M


# ----------------------------------------------------------------------------------------------------------------
# ours
# ----------------------------------------------------------------------------------------------------------------
def run_train_ours(args, rank, world, local, cfg=None, sync_bn=False, extras=True, outputs=None):
    """`outputs`: a dict that receives the results of the last timed step and the variables it left (see --dump-outputs)."""
    import torch
    import torch.distributed as dist
    import drs_b200
    from drs_b200 import dist as ddist, host
    from drs_b200.backend import GpuBackend
    cfg = cfg or TRAIN_CFG
    dev = torch.device("cuda", local)
    torch.cuda.set_device(dev)
    wl = isprs_workload(cfg)
    s = drs_b200.Session(cfg["net"], cfg["C"], cfg["K"], weight_decay=cfg["wd"], lr_initial=cfg["lr"], precision="bf16",
                         device=local, seed=5)
    be = GpuBackend(s, wl["train_data"] + wl["test_data"], wl["train_labels"] + wl["test_labels"], wl["mean"], wl["std"],
                    device=local, rank=rank, world=world)
    if world > 1:
        ddist.attach_nccl(s, sync_bn=sync_bn)
    B = cfg["batch"]
    W, K = args.warmup, args.steps
    depth = int(os.environ.get("DRS_PREFETCH", "2"))
    tail = depth + 2                 # untimed steps behind the timed ones: the planner thread runs ahead of the device by the
    niter = W + K + tail             # same margin at both ends of the timed region (steady state, K plans per K steps)
    crops, launches = [], [0, 0]
    ev = [torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)]
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()              # before the warm-up steps: NVML initialisation stays out of the timed region
    clocks = [None]
    orig_submit = be.submit_train

    def submit(plan, loss_mask=None):
        crops.append(int(plan.crop))
        return orig_submit(plan, loss_mask)

    be.submit_train = submit
    last_result = [None]
    if outputs is not None:
        orig_result = be.train_result

        def train_result(ticket):
            last_result[0] = orig_result(ticket)
            return last_result[0]

        be.train_result = train_result

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def hook(step, pipe):
        # called after step `step` has been enqueued and before step+1 is: the event recorded here fires when `step` is done
        if step == W:
            pipe.flush()
            barrier()
            sampler.begin()
            launches[0] = s.launch_count
            ev[0].record()
        elif step == W + K:
            ev[1].record()
            launches[1] = s.launch_count
            pipe.flush()
            barrier()
            clocks[0] = sampler.stop() if rank == 0 else None
            if outputs is not None:
                # the flush handed over this step's result last; step W+K+1 has not been enqueued, so the prediction buffer
                # and the variables are still those of step W+K
                loss, cm, n_correct = last_result[0]
                c = crops[-1]
                outputs["train_loss"] = np.array([loss], dtype=np.float64)
                outputs["train_confusion"] = cm.astype(np.float64)
                outputs["train_n_correct"] = np.array([n_correct], dtype=np.float64)
                outputs["train_pred"] = be._pred[:B * c * c].cpu().numpy().astype(np.float32).reshape(B, c, c)
                for name, v in s.variables().items():
                    outputs["train_var__" + name.replace("/", "__")] = np.asarray(v, dtype=np.float32)

    run_isprs_loop(be, wl, cfg, B * world, niter, hook)
    ms = ev[0].elapsed_time(ev[1])
    timed_crops = crops[W:W + K]
    px = sum(B * c * c for c in timed_crops)
    if world > 1:
        t = torch.tensor([ms], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    value = B * world * K / (ms / 1e3)
    out = dict(metric="train patches/s", value=value, unit="patches/s", ms_per_step=ms / K, dtype="bf16", scaling="weak",
               gpu_launches=launches[1] - launches[0], clocks=clocks[0],
               # the drawn patch sizes differ from run to run (and with the global batch): the pixel rate is the size-neutral view
               patch_mpixels_per_s=px * world / (ms / 1e3) / 1e6)
    if not extras:
        s.close()
        return out

    # ---- data-parallel check (SURVEY 8e): every rank must hold bit-identical variables and optimizer slots after the run
    if world > 1:
        out["dp_check"] = dp_check(s, be, cfg, rank, world, dev, sync_bn)

    # ---- kernel timing pass: the same patch sizes again with a CUDA event pair around every tensor-core launch.  Timing
    # single launches needs them serialised, so this pass runs the filter gradients on the main stream instead of overlapping
    # them with the backward's HBM-bound kernels (which is what the timed region above does); its step time is reported too.
    planner = host.NativePlanner()
    hw = np.asarray([wl["train_data"][0].shape[:2]], dtype=np.int32)
    rs = np.random.RandomState(1)
    inst = np.zeros((B * world, 4), dtype=np.int64)
    inst[:, 1], inst[:, 2], inst[:, 3] = rs.randint(0, 1900, B * world), rs.randint(0, 2400, B * world), rs.randint(0, 360, B * world)
    s.set_profiling(True)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    s.profile_read()
    e0.record()
    for c in timed_crops:
        be.train_on_plan(planner.plan(hw, inst, c, cfg["C"], own=be.own_rows(B * world)))
    e1.record()
    barrier()
    ms_prof = e0.elapsed_time(e1)
    conv_ms, conv_n, conv_fl = s.profile_read()
    s.set_profiling(False)
    planner.close()

    # ---- end to end through the sess.run seam: host x / y in pinned memory, host loss / pred / confusion back
    host_batches = {}
    rs = np.random.RandomState(3)
    for c in sorted(set(timed_crops)):
        xh = torch.from_numpy(rs.randn(B, c * c * cfg["C"]).astype(np.float32)).pin_memory()
        yh = torch.from_numpy(rs.randint(0, cfg["K"], size=(B, c * c)).astype(np.float32)).pin_memory()
        host_batches[c] = (xh.numpy(), yh.numpy(), xh, yh)
    for c in timed_crops[:3]:
        s.train_step(host_batches[c][0], host_batches[c][1], c, want_cm=True)
    barrier()
    e0.record()
    bi = bo = 0
    for c in timed_crops:
        s.train_step(host_batches[c][0], host_batches[c][1], c, want_cm=True)
        bi += B * c * c * (cfg["C"] + 1) * 4
        bo += B * c * c * 8 + 4 + (cfg["K"] ** 2 + 1) * 4
    e1.record()
    barrier()
    ms2 = e0.elapsed_time(e1)
    if world > 1:
        t = torch.tensor([ms2], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms2 = float(t.item())
    out["e2e"] = {"value": B * world * K / (ms2 / 1e3), "unit": "patches/s", "h2d_bytes_per_step": bi // K, "d2h_bytes_per_step": bo // K,
                  "api": "Session.train_step == drs_train_step_host (sess.run seam, host feeds/fetches)"}
    s.close()

    pk = peaks()
    capped = bool(clocks[0] and "sw_power_cap" in (clocks[0].get("reasons") or []))
    peak = pk["tc_sustained"] if capped else pk["tc_burst"]
    ach = (conv_fl / (conv_ms * 1e-3) / 1e12) if conv_ms > 0 else None
    out["roofline"] = {"bound": "tensor", "kernel": "tcgen05 kernels of the step: conv_tc_kernel (fprop + dgrad) and wgrad_tc_kernel",
                       "achieved": ach, "peak": peak, "unit": "TFLOP/s", "frac": (ach / peak) if ach else None,
                       "traffic": profiled_traffic("train"),
                       "peak_source": pk["source"] + (" bf16 sustained (sw_power_cap seen during the timed region)" if capped
                                                      else " bf16 burst (no power cap during the timed region)"),
                       "launches": conv_n, "kernel_ms_per_step": conv_ms / K, "ms_per_step_timing_pass": ms_prof / K,
                       "step_tflops_all_kernels": conv_flops_train(cfg["net"], cfg["C"], cfg["K"], px) / (ms * 1e-3) / 1e12}
    out["config"] = {"workload": "configs[1]: isprs_dilated_random.py dilated_grsl multinomial {25..49} acc, batch 64/GPU, Vaihingen-shaped "
                                 "2000x2500x4 float64 scene resident in HBM; one step = one iteration of the drop-in loop "
                                 "(loops.isprs_train: draw size, select_batch, dynamically_create_patches decisions incl. np.random.normal "
                                 "noise, gather+rotate+flip+normalise, sess.run(train), calc_accuracy_by_crop, score update)",
                     "net": cfg["net"], "batch_per_gpu": B, "global_batch": B * world, "patch_sizes_drawn": timed_crops,
                     "parallelism": "dp%d" % world, "sync_bn": bool(sync_bn), "cuda_graphs": os.environ.get("DRS_GRAPHS", "1") != "0",
                     "host_plan": "native planner thread %d steps ahead (bit-exact np.random stream), results taken one step late; "
                                  "%d untimed tail steps keep the planner's lead equal at both ends of the timed region" % (depth, tail),
                     "l2": "per-step working set (activations %.0f-%.0f MB) exceeds the 126 MB L2; no explicit flush" %
                           (B * 25 * 25 * 896 * 6 / 1e6, B * 49 * 49 * 896 * 6 / 1e6)}
    return out


class TimedLoop:
    """The timing protocol of run_train_ours as a reusable piece: wraps a backend, records the patch sizes it is fed, and
    provides the step hook that brackets steps W+1 .. W+K with CUDA events (barrier + synchronize on both sides)."""

    def __init__(self, be, session, W, K, local, world=1):
        import torch
        self.torch, self.be, self.s, self.W, self.K, self.world = torch, be, session, W, K, world
        self.crops, self.launches = [], [0, 0]
        self.ev = [torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)]
        self.depth = int(os.environ.get("DRS_PREFETCH", "2"))
        self.niter = W + K + self.depth + 2
        orig = be.submit_train

        def submit(plan, loss_mask=None):
            self.crops.append(int(plan.crop))
            return orig(plan, loss_mask)

        be.submit_train = submit

    def barrier(self):
        if self.world > 1:
            import torch.distributed as dist
            dist.barrier()
        self.torch.cuda.synchronize()

    def hook(self, step, pipe):
        if step == self.W:
            pipe.flush()
            self.barrier()
            self.launches[0] = self.s.launch_count
            self.ev[0].record()
        elif step == self.W + self.K:
            self.ev[1].record()
            self.launches[1] = self.s.launch_count
            pipe.flush()
            self.barrier()

    def result(self, batch, unit="patches/s"):
        ms = self.ev[0].elapsed_time(self.ev[1])
        crops = self.crops[self.W:self.W + self.K]
        return {"value": batch * self.K / (ms / 1e3), "unit": unit, "us_per_step": ms / self.K * 1e3, "steps": self.K,
                "gpu_launches_per_step": (self.launches[1] - self.launches[0]) / self.K, "patch_sizes_drawn": crops,
                "patch_pixels_per_step": int(sum(batch * c * c for c in crops) / self.K)}


def quiet_loop(fn):
    """Run a training loop of loops.py with its log lines discarded and its files in a scratch directory."""
    import contextlib
    import tempfile
    cwd = os.getcwd()
    with tempfile.TemporaryDirectory() as tmp, open(os.devnull, "w") as null:
        os.chdir(tmp)
        try:
            with contextlib.redirect_stdout(null):
                fn(tmp + "/")
        finally:
            os.chdir(cwd)


def run_extra_configs(args, local):
    """The other BASELINE.json configs as extra keys of the line (1 GPU, short runs of the same drop-in loops):
    configs[0] Dilated6 single_fixed 25 batch 16 (the launch-bound case), configs[2] DenseDilated6 uniform 25..65 on a
    Potsdam-shaped tile, configs[4] contest + coffee multi_fixed / loss, and configs[3] at crop 65."""
    import random
    import torch
    import drs_b200
    from drs_b200 import host, loops, synth
    from drs_b200.backend import GpuBackend
    dev = torch.device("cuda", local)
    W, K = 5, max(20, min(args.steps, 50))
    far = 10 ** 9
    out = {}

    def isprs_case(key, cfg, note):
        wl = isprs_workload(cfg)
        s = drs_b200.Session(cfg["net"], cfg["C"], cfg["K"], weight_decay=cfg["wd"], lr_initial=cfg["lr"], precision="bf16", device=local, seed=5)
        be = GpuBackend(s, wl["train_data"] + wl["test_data"], wl["train_labels"] + wl["test_labels"], wl["mean"], wl["std"], device=local)
        tl = TimedLoop(be, s, W, K, local)
        run_isprs_loop(be, wl, cfg, cfg["batch"], tl.niter, tl.hook)
        r = tl.result(cfg["batch"])
        r["tflops_all_kernels"] = conv_flops_train(cfg["net"], cfg["C"], cfg["K"], r["patch_pixels_per_step"]) / (r["us_per_step"] * 1e-6) / 1e12
        r["workload"] = note
        s.close()
        out[key] = r

    isprs_case("configs[0]", dict(net="dilated_icpr_original", dataset="vaihingen", C=4, K=6, batch=16, values=[25], distribution="single_fixed",
                                  update="acc", lr=0.01, wd=0.005),
               "isprs_dilated_random.py dilated_icpr_original single_fixed 25, batch 16, Vaihingen-shaped 2000x2500x4 scene (the reference's "
               "CPU-runnable case; launch-bound on a B200: whole-step CUDA graph)")
    isprs_case("configs[2]", dict(net="dilated_icpr_rate6_densely", dataset="potsdam", C=5, K=6, batch=16, values=[25, 65], distribution="uniform",
                                  update="acc", lr=0.01, wd=0.005),
               "isprs_dilated_random.py dilated_icpr_rate6_densely uniform 25..65, batch 16 per GPU (global 128 on 8 GPUs), Potsdam-shaped "
               "6000x6000x5 tile")

    # ---- contest (contest_dilated_random.py ... multi_fixed loss): one training scene, label 7 = unlabelled
    np.random.seed(SEED); random.seed(SEED)
    # (label blocks of 20 px: the contest's class distribution skips single-class windows, contest:172-189)
    img, lab = synth.scene("contest", unlabelled=True, block=20)
    timg, tlab = synth.scene("contest", H=600, W=500, seed=99, unlabelled=True, block=20)
    distr = host.contest_create_distributions_over_classes(lab, 25, 50, 7, verbose=False)
    assert len(distr) > 64 * 3, "synthetic contest scene has too few multi-class windows"
    mean, std = synth.normalisation(img)
    values = [25, 33, 41, 49]
    pal, occ, chosen = host.init_score_arrays("multi_fixed", values, occur_init=1)
    s = drs_b200.Session("dilated_grsl_rate8", 3, 7, weight_decay=0.005, lr_initial=0.01, decay_rate=0.1, precision="bf16", device=local, seed=5)
    be = GpuBackend(s, [img, timg], [lab, tlab], mean, std, device=local)
    tl = TimedLoop(be, s, W, K, local)
    quiet_loop(lambda outp: loops.contest_train(be, img, lab, tlab, distr, outp, "", 64, tl.niter, "multi_fixed", "loss", pal, occ, chosen,
                                                None, values, 7, display_step=far, epoch_number=far, val_inteval=far, final_test=False,
                                                step_hook=tl.hook))
    r = tl.result(64)
    r["tflops_all_kernels"] = conv_flops_train("dilated_grsl_rate8", 3, 7, r["patch_pixels_per_step"]) / (r["us_per_step"] * 1e-6) / 1e12
    r["workload"] = "contest_dilated_random.py dilated_grsl_rate8 multi_fixed 25,33,41,49 loss, batch 64, GRSS-DFC2014-shaped 3989x2830x3 float32 scene"
    s.close()
    out["configs[4] contest"] = r

    # ---- coffee (coffee_dilated_random.py ... multi_fixed loss): 500x500x3 float32 tiles, float16 training patches
    np.random.seed(SEED); random.seed(SEED)
    tiles = [synth.scene("coffee", seed=200 + i) for i in range(4)]
    tdata, tlabs = [t[0] for t in tiles[:3]], [t[1] for t in tiles[:3]]
    distr = host.coffee_create_distributions_over_classes(tlabs, 25, 25, 2)
    mean, std = synth.normalisation(tdata[0])
    values = [25, 33, 41]
    pal, occ, chosen = host.init_score_arrays("multi_fixed", values)
    s = drs_b200.Session("dilated_grsl", 3, 2, weight_decay=0.005, lr_initial=0.01, decay_rate=0.1, precision="bf16", device=local, seed=5)
    be = GpuBackend(s, tdata + [tiles[3][0]], tlabs + [tiles[3][1]], mean, std, device=local, train_fp16_patches=True)
    tl = TimedLoop(be, s, W, K, local)
    quiet_loop(lambda outp: loops.coffee_train(be, tdata, [tiles[3][1]], distr, outp, "", 64, tl.niter, "multi_fixed", "loss", pal, occ, chosen,
                                               None, values, 2, display_step=far, epoch_number=far, val_inteval=far, final_test=False,
                                               step_hook=tl.hook))
    r = tl.result(64)
    r["tflops_all_kernels"] = conv_flops_train("dilated_grsl", 3, 2, r["patch_pixels_per_step"]) / (r["us_per_step"] * 1e-6) / 1e12
    r["workload"] = "coffee_dilated_random.py dilated_grsl multi_fixed 25,33,41 loss, batch 64, three 500x500x3 float32 tiles, float16 training patches"
    s.close()
    out["configs[4] coffee"] = r
    return out


def dp_check(s, be, cfg, rank, world, dev, sync_bn):
    """(1) After the timed steps every rank's variables, BN statistics and momentum slots must be bit-identical: one checksum per
    rank, all-gathered.  (2) One SyncBN fp32 step on a global batch split over the ranks against the same step done by a single
    process on the whole batch (the parity mode of SURVEY 8e): loss and every updated variable."""
    import torch
    import torch.distributed as dist
    import drs_b200
    from drs_b200 import dist as ddist
    import hashlib
    names = [n for n, _ in s.variable_names()]
    local_stats = [n for n in names if n.endswith("/moving_mean") or n.endswith("/moving_variance")]
    h = hashlib.sha256()
    for n in names:
        if n in local_stats and not sync_bn:
            continue                      # rank-local by design without SyncBN (averaged before evaluation / save)
        h.update(np.ascontiguousarray(s.get_variable(n)).tobytes())
    digest = np.frombuffer(h.digest()[:8], dtype=np.int64).copy()
    t = torch.from_numpy(digest).to(dev)
    allv = [torch.empty_like(t) for _ in range(world)]
    dist.all_gather(allv, t)
    replicas_equal = all(bool((v == allv[0]).all().item()) for v in allv)
    # (2) SyncBN parity step in fp32
    B, crop, C, K = 4 * world, 25, cfg["C"], cfg["K"]
    rs = np.random.RandomState(11)
    x = rs.randn(B, crop * crop * C).astype(np.float32)
    y = rs.randint(0, K, size=(B, crop * crop)).astype(np.float32)
    sp = drs_b200.Session(cfg["net"], C, K, weight_decay=cfg["wd"], lr_initial=cfg["lr"], precision="fp32", device=dev.index, seed=5)
    sp.set_stream(torch.cuda.current_stream(dev).cuda_stream)
    ddist.attach_nccl(sp, sync_bn=True)
    per = B // world
    loss_dp, _ = sp.train_step(x[rank * per:(rank + 1) * per], y[rank * per:(rank + 1) * per], crop)
    worst = 0.0
    loss_ref = None
    if rank == 0:
        def single(xx):
            s1 = drs_b200.Session(cfg["net"], C, K, weight_decay=cfg["wd"], lr_initial=cfg["lr"], precision="fp32", device=dev.index, seed=5)
            s1.set_stream(torch.cuda.current_stream(dev).cuda_stream)
            l1, _ = s1.train_step(xx, y, crop)
            v = {n: s1.get_variable(n) for n, _ in s1.variable_names()}
            s1.close()
            return l1, v

        loss_ref, ref = single(x)
        # the conditioning of the step itself: the same single-process step with x perturbed by 1e-7 relative (the size of the
        # only difference data parallelism introduces, the summation order of the BN statistics); see tools/dp_parity.py
        _, ptb = single((x * (1.0 + 1e-7 * np.random.RandomState(9).randn(*x.shape))).astype(np.float32))
        within, worst_p = True, 0.0
        for n in ref:
            den = np.abs(ref[n]).max() + 1e-12
            err = float(np.abs(ref[n] - sp.get_variable(n)).max() / den)
            err_p = float(np.abs(ref[n] - ptb[n]).max() / den)
            within = within and err < max(5e-4, 3.0 * err_p)
            worst, worst_p = max(worst, err), max(worst_p, err_p)
    sp.close()
    ok = replicas_equal
    res = {"replicas_bit_identical": bool(replicas_equal)}
    if rank == 0:
        res.update(syncbn_loss=float(loss_dp), single_process_loss=float(loss_ref), syncbn_worst_rel_diff=worst,
                   perturbation_1e7_worst_rel_diff=worst_p)
        res["tolerance"] = "every variable incl. momentum slots: max(5e-4, 3 x what a 1e-7 input perturbation of the single-process step moves it by)"
        ok = ok and abs(float(loss_dp) - float(loss_ref)) < 2e-5 * max(1.0, abs(float(loss_ref))) and within
    res["result"] = "ok" if ok else "FAILED"
    return res


def run_infer_ours(args, rank, world, local, steps=3, cfg=None, outputs=None):
    """Full-scene sliding-window inference (isprs:1241-1284), row stripes over the ranks, label map assembled on rank 0.
    `steps` whole passes are timed one by one (barrier + synchronize on both sides of each); value = median pass.
    `outputs`: a dict that receives a fixed sample of the last timed pass's label map (see --dump-outputs)."""
    import torch
    import torch.distributed as dist
    import drs_b200
    from drs_b200 import dist as ddist, synth
    cfg = cfg or INFER_CFG
    dev = torch.device("cuda", local)
    torch.cuda.set_device(dev)
    H, W = cfg["H"], cfg["W"]
    if args.small:
        H = W = 1500
    img, _ = synth.scene(cfg["dataset"], H=H, W=W)
    mean, std = synth.normalisation(img)
    s = drs_b200.Session(cfg["net"], cfg["C"], cfg["K"], precision="f16", device=local, seed=9)
    s.set_stream(torch.cuda.current_stream(dev).cuda_stream)
    s.set_normalization(mean, std)
    if world > 1:
        ddist.attach_nccl(s)
    cuts = ddist.stripe_bounds(H, world)
    r0, r1 = cuts[rank], cuts[rank + 1]

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def one_pass():
        if world == 1:
            return s.scene_infer(0, cfg["crop"], cfg["batch"], H, W)
        # the stripe stays on the device; NCCL send/recv assembles the map on rank 0, one device-to-host copy there
        s.scene_infer(0, cfg["crop"], cfg["batch"], H, W, row_begin=r0, row_end=r1, keep_on_device=True)
        return s.scene_gather_labels(H, W, cuts, rank)

    # a rank keeps only the scene rows its stripe needs (the stripe plus the patch rows straddling its borders)
    u0, u1 = ddist.stripe_rows_needed(H, cfg["crop"], r0, r1) if world > 1 else (None, None)
    s.upload_scene(0, img, None, u0, u1)
    s.scene_infer(0, cfg["crop"], cfg["batch"], H, W, row_begin=r0, row_end=min(r1, r0 + 40))   # warm-up stripe (kernels)
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    one_pass()                                   # warm-up pass: stripe-sized buffers, geometry tables, first collective
    barrier()
    sampler.begin()
    times, launches = [], 0
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for _ in range(steps):
        barrier()
        l0 = s.launch_count
        e0.record()
        labels = one_pass()
        e1.record()
        barrier()
        times.append(e0.elapsed_time(e1))
        launches = s.launch_count - l0
    clocks = sampler.stop() if rank == 0 else None
    if outputs is not None:
        # the whole map as float32 would exceed the dump's 64 MB: class counts of every pixel plus a fixed seeded sample
        flat = np.asarray(labels).reshape(-1)
        idx = np.sort(np.random.RandomState(0).randint(0, flat.size, size=1 << 20))
        outputs["infer_label_counts"] = np.bincount(flat, minlength=cfg["K"]).astype(np.float64)
        outputs["infer_labels_sample"] = flat[idx].astype(np.float32)
        outputs["infer_labels_sample_index"] = idx.astype(np.float64)
    # kernel timing pass (roofline): the same pass once more with a CUDA-event pair around every tensor-core launch
    s.set_profiling(True)
    s.scene_infer(0, cfg["crop"], cfg["batch"], H, W, row_begin=r0, row_end=r1, keep_on_device=True)
    barrier()
    conv_ms, conv_n, conv_fl = s.profile_read()
    s.set_profiling(False)
    # end to end: host scene -> HBM -> label map on the host
    e2e_times = []
    for _ in range(max(1, min(steps, 2))):
        barrier()
        e0.record()
        if world == 1:
            # a fresh tile: the upload is streamed ahead of the chunks that read it (drs_scene_infer_host)
            s.scene_infer_host(0, img, cfg["crop"], cfg["batch"])
        else:
            s.upload_scene(0, img, None, u0, u1)
            one_pass()
        e1.record()
        barrier()
        e2e_times.append(e0.elapsed_time(e1))
    ms, ms2 = float(np.median(times)), float(np.median(e2e_times))
    if world > 1:
        t = torch.tensor([ms, ms2], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms, ms2 = float(t[0].item()), float(t[1].item())
    s.close()
    pk = peaks()
    capped = bool(clocks and "sw_power_cap" in (clocks.get("reasons") or []))
    peak = pk["tc_sustained"] if capped else pk["tc_burst"]
    ach = (conv_fl / (conv_ms * 1e-3) / 1e12) if conv_ms > 0 else None
    return dict(metric="full-scene inference Mpixel/s", value=H * W / 1e6 / (ms / 1e3), unit="Mpixel/s", ms_per_step=ms,
                passes_ms=[round(t, 2) for t in times], dtype="f16", scaling="strong",
                e2e={"value": H * W / 1e6 / (ms2 / 1e3), "unit": "Mpixel/s", "h2d_bytes_per_step": int(img.nbytes if u0 is None else img[u0:u1].nbytes),
                     "d2h_bytes_per_step": int(H * W), "api": "Session.scene_infer_host (host scene in, upload streamed under the pass, host label map out)" if world == 1 else
                            "Session.upload_scene + Session.scene_infer + scene_gather_labels (host stripe in, host label map out on rank 0)"},
                gpu_launches=launches, clocks=clocks,
                roofline={"bound": "tensor", "kernel": "conv_tc_kernel (tcgen05 fprop)", "achieved": ach, "peak": peak,
                          "unit": "TFLOP/s", "frac": ach / peak if ach else None, "traffic": profiled_traffic("inference"),
                          "peak_source": pk["source"] + (" bf16 sustained (sw_power_cap seen)" if capped else " bf16 burst"), "launches": conv_n,
                          "kernel_ms_per_step": conv_ms},
                config={"workload": "configs[3]: %s full-scene sliding-window inference, %s-shaped %dx%dx%d "
                                    "float64, crop %d stride %d, row stripes over %d GPU(s); median of %d passes" %
                                    (cfg["net"], cfg["dataset"], H, W, cfg["C"], cfg["crop"], cfg["crop"] // 2, world, steps),
                        "net": cfg["net"], "crop": cfg["crop"], "patches": int(len(drs_b200.grid_positions(H, W, cfg["crop"], cfg["batch"]))),
                        "parallelism": "stripes%d" % world, "l2": "scene (%.0f MB) and activations exceed L2" % (img.nbytes / 1e6)})


# ----------------------------------------------------------------------------------------------------------------
# reference-equivalent CPU path (oracle): the checker timed as the baseline
# ----------------------------------------------------------------------------------------------------------------
def cli_rate(cfg, iters=300, first=100):
    """The drop-in command line itself: ``isprs_dilated_random.py ... training`` on the same synthetic scene written as .npy,
    rate taken from the script's own "Iter N -- Time ..." log lines (isprs:1766-1772) between iteration `first` and `iters`."""
    import datetime
    import re
    import tempfile
    from drs_b200 import synth
    with tempfile.TemporaryDirectory() as tmp:
        data, out = os.path.join(tmp, "vaihingen"), os.path.join(tmp, "out")
        os.makedirs(data)
        os.makedirs(out)
        img, lab = synth.scene(cfg["dataset"])
        timg, tlab = synth.scene(cfg["dataset"], H=300, W=300, seed=4321)
        np.save(os.path.join(data, "1_image.npy"), img)
        np.save(os.path.join(data, "1_labels.npy"), lab)
        np.save(os.path.join(data, "2_image.npy"), timg)
        np.save(os.path.join(data, "2_labels.npy"), tlab)
        argv = [sys.executable, os.path.join(ROOT, "isprs_dilated_random.py"), data + "/", out + "/", "", "1", "2", str(cfg["lr"]),
                str(cfg["wd"]), str(cfg["batch"]), str(iters), "25", "25", cfg["net"], cfg["distribution"],
                ",".join(str(v) for v in cfg["values"]), cfg["update"], "training"]
        env = dict(os.environ, PYTHONPATH=ROOT, DRS_SEED="5")
        for k in ("RANK", "WORLD_SIZE", "LOCAL_RANK", "MASTER_ADDR", "MASTER_PORT"):
            env.pop(k, None)
        t0 = time.perf_counter()
        r = subprocess.run(argv, cwd=tmp, env=env, capture_output=True, text=True, timeout=900)
        wall = time.perf_counter() - t0
    if r.returncode != 0:
        return {"error": (r.stdout[-400:] + r.stderr[-400:])}
    stamps = {}
    for m in re.finditer(r"^Iter (\d+) -- Time (\d+):(\d+):(\d+\.?\d*)", r.stdout, re.M):
        stamps[int(m.group(1))] = int(m.group(2)) * 3600 + int(m.group(3)) * 60 + float(m.group(4))
    if first not in stamps or iters not in stamps:
        return {"error": "log lines of iterations %d / %d not found" % (first, iters)}
    dt = (stamps[iters] - stamps[first]) % 86400
    return {"patches_per_s": cfg["batch"] * (iters - first) / dt, "iterations": iters - first, "ms_per_step": dt / (iters - first) * 1e3,
            "wall_s_whole_command": wall,
            "cmd": "isprs_dilated_random.py <data>/ <out>/ '' 1 2 %g %g %d %d 25 25 %s %s %s %s training" %
                   (cfg["lr"], cfg["wd"], cfg["batch"], iters, cfg["net"], cfg["distribution"], ",".join(str(v) for v in cfg["values"]),
                    cfg["update"]),
            "how": "timestamps of the script's own 'Iter N -- Time' lines, iterations %d..%d" % (first, iters)}


class OracleBackend:
    """The reference-equivalent CPU path behind the loop's backend interface (checker code timed as the baseline): NumPy
    gather / flip / normalise of the plan (scipy rotation already applied by the Python planner, as the reference does it on
    the host), the PyTorch-CPU fp32 restatement of the TF graph for sess.run(train), and the reference's Python-loop
    calc_accuracy_by_crop."""

    def __init__(self, cfg, wl):
        import torch
        from oracle import nets_torch
        self.cfg, self.wl, self.torch = cfg, wl, torch
        self.net = nets_torch.OracleNet(cfg["net"], cfg["C"], cfg["K"], nets_torch.init_params(cfg["net"], cfg["C"], cfg["K"], seed=5))
        self.crops = []

    def train_on_plan(self, plan, loss_mask=None):
        from oracle import host_np
        cfg, wl, torch = self.cfg, self.wl, self.torch
        self.crops.append(int(plan.crop))
        xs, ys = host_np.apply_plan(wl["train_data"], wl["train_labels"], plan.inst, plan.flips, plan.crop, wl["mean"], wl["std"],
                                    plan.noise, plan.noise_on, plan.over_x, plan.over_y, plan.over_on)
        B = len(plan.inst)
        loss, pred, _ = self.net.train_step(torch.from_numpy(xs.reshape(B, -1)), torch.from_numpy(ys.reshape(B, -1)), plan.crop,
                                            cfg["lr"], cfg["wd"])
        masks = None if plan.acc_mask is None else plan.acc_mask.astype(bool)
        acc, _, cm = host_np.confusion_by_crop(ys.astype(np.int64), pred.numpy(), cfg["K"], masks)
        return loss, cm, acc

    def save(self, path):
        pass


def cpu_train_baseline(steps, warmup, cfg=None):
    """The SAME seeded loop as the GPU arm (same scene, same seeds -> same patch sizes, batches and augmentations), strictly
    sequential like the reference (no planner thread), on the host cores."""
    import torch
    cfg = cfg or TRAIN_CFG
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    wl = isprs_workload(cfg)
    be = OracleBackend(cfg, wl)
    B = cfg["batch"]
    t = [0.0, 0.0]

    def hook(step, pipe):
        if step == warmup:
            pipe.flush()
            t[0] = time.perf_counter()
        elif step == warmup + steps:
            pipe.flush()
            t[1] = time.perf_counter()

    if warmup == 0:
        t[0] = time.perf_counter()
    run_isprs_loop(be, wl, cfg, B, warmup + steps, hook, depth=0)
    dt = t[1] - t[0]
    crops = be.crops[warmup:warmup + steps]
    return dict(value=B * steps / dt, unit="patches/s", cores=cores, kind="port", ms_per_step=dt / steps * 1e3, steps=steps,
                patch_sizes_drawn=crops,
                sample="%d full iterations (batch 64, crops %s) of the same seeded drop-in loop on the same 2000x2500x4 scene: Python "
                       "dynamically_create_patches decisions + scipy order-0 rotation + np.random.normal noise + NumPy gather/normalise, "
                       "PyTorch-CPU fp32 graph fwd+bwd+momentum, Python-loop calc_accuracy_by_crop; TensorFlow not installable "
                       "(SURVEY F13)" % (steps, crops))


def cpu_infer_baseline(batches=6):
    import torch
    from drs_b200 import synth
    from oracle import host_np, nets_torch
    cfg = INFER_CFG
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    img, _ = synth.scene(cfg["dataset"], H=300, W=400)
    mean, std = synth.normalisation(img)
    orc = nets_torch.OracleNet(cfg["net"], cfg["C"], cfg["K"], nets_torch.init_params(cfg["net"], cfg["C"], cfg["K"], seed=9))
    crop, B = cfg["crop"], cfg["batch"]
    stride = host_np.sliding_stride(crop)
    prob = np.zeros((300, 400, cfg["K"]), dtype=np.float32)
    occ = np.zeros((300, 400, cfg["K"]), dtype=np.uint32)

    def one(i):
        pos = host_np.patch_positions(300, 400, crop, stride, i, B, "isprs")
        xs, _ = host_np.apply_plan([img], None, [(0, r, c) for r, c in pos], None, crop, mean, std)
        _, logits = orc.infer(torch.from_numpy(xs.reshape(len(pos), -1)), crop)
        lg = logits.numpy()
        for j, (r, c) in enumerate(pos):
            prob[r:r + crop, c:c + crop] += lg[j]
            occ[r:r + crop, c:c + crop] += 1
        return len(pos)

    one(0)
    t0 = time.perf_counter()
    n = sum(one(i) for i in range(1, 1 + batches))
    dt = time.perf_counter() - t0
    # scene pixels per second = patches/s * (H*W / patches of the full scene); extrapolated linearly by patch count
    total_patches = 499 * 499
    sec_full = total_patches / (n / dt)
    return dict(value=cfg["H"] * cfg["W"] / 1e6 / sec_full, unit="Mpixel/s", cores=cores, kind="port", patches_per_s=n / dt,
                sample="%d batches of 64 patches (crop 25) through the PyTorch-CPU fp32 graph + NumPy accumulate, extrapolated "
                       "linearly to the 249001 patches of a 6000x6000 scene" % batches)


def run_reference(args, rank, world):
    if rank != 0:
        return None
    if args.workload == "infer":
        b = cpu_infer_baseline(batches=max(4, min(args.steps, 16)))
        line = dict(metric="full-scene inference Mpixel/s", value=b["value"], unit=b["unit"], ms_per_step=None, dtype="f32",
                    scaling="strong", config={"workload": "configs[3] on the host cores (bounded sample, extrapolated)"})
    else:
        b = cpu_train_baseline(args.steps, args.warmup)
        line = dict(metric="train patches/s", value=b["value"], unit=b["unit"], ms_per_step=b["ms_per_step"], dtype="f32",
                    scaling="weak", config={"workload": "configs[1] on the host cores: " + b["sample"], "net": TRAIN_CFG["net"],
                                            "batch_per_gpu": TRAIN_CFG["batch"], "global_batch": TRAIN_CFG["batch"],
                                            "patch_sizes_drawn": b["patch_sizes_drawn"]})
    line.update(impl="reference", cpu_baseline=b, gpu_launches=0,
                e2e={"value": b["value"], "unit": b["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0})
    return line


DUMP_LIMIT = 64 << 20


def write_outputs(path, outputs):
    """--dump-outputs: one float32 / float64 .npy per array, 64 MB in all at most."""
    total = sum(a.nbytes for a in outputs.values())
    if total > DUMP_LIMIT:
        raise SystemExit("bench.py: %d bytes of outputs exceed the %d-byte dump limit" % (total, DUMP_LIMIT))
    os.makedirs(path, exist_ok=True)
    for name, a in outputs.items():
        assert a.dtype in (np.float32, np.float64), (name, a.dtype)
        np.save(os.path.join(path, name + ".npy"), a)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="train", choices=["train", "infer"])
    ap.add_argument("--no-secondary", action="store_true", help="skip the second headline metric")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-cli", action="store_true", help="skip the command-line level rate")
    ap.add_argument("--no-extra", action="store_true", help="skip the other BASELINE configs (configs[0], [2], [4], [3] at crop 65)")
    ap.add_argument("--small", action="store_true", help="1500x1500 inference scene (profiling runs)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step computed as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs dumps the GPU path (--impl ours)")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    rank, world, local = dist_env()
    base = dict(n_gpus=world, steps=args.steps, warmup=args.warmup, higher_is_better=True, vs_baseline=None, data="synthetic")
    outputs = {} if args.dump_outputs and rank == 0 else None

    if args.impl == "reference":
        line = run_reference(args, rank, world)
        if line is not None:
            base.update(line)
            print(json.dumps(base), flush=True)
        return 0

    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the product path has no CPU fallback (use --impl reference for the CPU baseline)")
    import torch.distributed as dist
    if world > 1:
        torch.cuda.set_device(local)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    try:
        if args.workload == "train":
            line = run_train_ours(args, rank, world, local, outputs=outputs)
            if world > 1 and not args.no_secondary:
                # the parity mode of data parallelism (SURVEY 8e): BN statistics over the global batch, forward and backward
                sb = run_train_ours(args, rank, world, local, sync_bn=True, extras=False)
                line["sync_bn"] = {k: sb[k] for k in ("value", "unit", "ms_per_step", "gpu_launches")}
            second = None if args.no_secondary else run_infer_ours(args, rank, world, local, outputs=outputs)
        else:
            line = run_infer_ours(args, rank, world, local, steps=args.steps, outputs=outputs)
            second = None
        if rank == 0:
            base.update(line)
            base["impl"] = "ours"
            if second is not None:
                base["inference"] = second
            if world == 1 and not args.no_extra and args.workload == "train":
                base["configs"] = run_extra_configs(args, local)
                if second is not None:
                    c65 = run_infer_ours(args, rank, world, local, steps=3, cfg=dict(INFER_CFG, crop=65))
                    base["configs"]["configs[3] crop 65"] = {k: c65[k] for k in ("value", "unit", "ms_per_step", "passes_ms", "gpu_launches")}
                    base["configs"]["configs[3] crop 65"]["roofline_frac"] = c65["roofline"]["frac"]
            if world == 1 and not args.no_cli and args.workload == "train":
                base["cli"] = cli_rate(TRAIN_CFG)
            if world == 1 and not args.no_cpu:
                base["cpu_baseline"] = cpu_train_baseline(8, 2) if args.workload == "train" else cpu_infer_baseline()
                if second is not None:
                    base["inference"]["cpu_baseline"] = cpu_infer_baseline()
            if outputs is not None:
                write_outputs(args.dump_outputs, outputs)
            print(json.dumps(base), flush=True)
    finally:
        if world > 1:
            dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
