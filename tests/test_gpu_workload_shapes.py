"""Every layer at the shapes of the benchmark workloads, and the graph-replayed training step tied to those checks.

Workloads (bench.py; test_workload_table_matches_bench pins TRAIN_CFG and INFER_CFG to this table):

    configs[0]          dilated_icpr_original      C 4  K 6  batch 16          single_fixed 25
    configs[1]          dilated_grsl               C 4  K 6  batch 64          multinomial {25, 29, .., 49}: draws 25..49
    configs[2]          dilated_icpr_rate6_densely C 5  K 6  batch 16 per GPU  uniform 25..65
    configs[3]          dilated_grsl_rate8         C 5  K 6  inference, scene chunks of a 6000 x 6000 scene, crops 25 and 65
    configs[4] contest  dilated_grsl_rate8         C 3  K 7  batch 64          multi_fixed 25, 33, 41, 49, ignore label 7
    configs[4] coffee   dilated_grsl               C 3  K 2  batch 64          multi_fixed 25, 33, 41

The launch decisions that depend on the shape are mirrored on the host (regime_signature): per convolution on the tensor
cores (forward and data gradient) the pairing mt, two CTAs per SM, whether the grid is the tile count or the CTA limit and
the ConvSched round class; per filter gradient on the tensor cores T, the limit that chose the split count and whether the
pixels split into whole 64-pixel chunks; per pooling layer the row-segment regime and the segment length mod 3 of the
training pool forward and the fused pool + BN backward; conv1's tile count against its grid.  select_crops picks, per
training workload, crops that reach every value any crop of the interval reaches, the smallest and largest included.

Training (GPU), per workload, a seeded sequence of 6 to 8 steps over the selected crops with repeats, from the same
variables twice:
  E  eager under DRS_DEBUG_KEEP=1, bn_decay = 0, weight_decay = 0: after every step the forward checks of
     test_gpu_forward_layers (train_forward_checks) and every backward stage of test_gpu_backward_layers (check_step) on the
     step's own taps, against the variables read before the step;
  P  the product path: no DRS_DEBUG_KEEP, reserve(B, largest crop), the ignore label, CUDA graphs captured up front for
     every crop the loop can draw (backend.prepare_training), steps submitted with train_step_async and their results
     fetched two steps late.
Halfway, one validation infer at the largest crop with 16x the batch grows the arena (free device memory drops), which
forces P to capture its graphs again.  P must equal E bit for bit: loss, confusion counts and pred of every step, then
every variable, momentum slot and global_step.  A set_variable after the capture, made on both, keeps them equal; without
it on P the first step already differs.

Inference (GPU): InferRun at the scene pass's own chunk sizes (scene_infer_impl: chunk = min(P, sm 40 128 / crop^2), and
the last partial chunk of the 6000 x 6000 grid), f16 and bf16, sampled pixels.
"""
import re
import time
from math import ceil

import numpy as np
import pytest

from test_gpu_backward_layers import TrainRun, _assert_within, _subset_cols, check_step, pool_nseg, \
    wgrad_tc_supported
from test_gpu_forward_layers import REPORT, InferRun, _print_report, net_layers, nseg_class, params_with_stats, sample_pixels, \
    train_forward_checks
from test_gpu_parity import rounded

B200_SMS = 148
BM = 128                                            # CONV_TC_BM: pixels per tile

# name -> (net, C, K, batch, crops the loop can draw, ignore label, isprs loop (accuracy mask))
TRAIN_WORKLOADS = {
    "configs[0]": ("dilated_icpr_original", 4, 6, 16, [25], None, True),
    "configs[1]": ("dilated_grsl", 4, 6, 64, list(range(25, 50)), None, True),
    "configs[2]": ("dilated_icpr_rate6_densely", 5, 6, 16, list(range(25, 66)), None, True),
    "configs[4] contest": ("dilated_grsl_rate8", 3, 7, 64, [25, 33, 41, 49], 7, False),
    "configs[4] coffee": ("dilated_grsl", 3, 2, 64, [25, 33, 41], None, False),
}
# name -> (net, C, K, crops, scene H, W)
INFER_WORKLOADS = {
    "configs[3]": ("dilated_grsl_rate8", 5, 6, (25, 65), 6000, 6000),
    "configs[4] contest": ("dilated_grsl_rate8", 3, 7, (25,), 6000, 6000),
}


def _ids(table):
    """configs[4] contest -> configs4_contest"""
    return [re.sub(r"\W+", "_", n.replace("[", "").replace("]", "")) for n in table]


def test_workload_table_matches_bench():
    """The table above is bench.py's: TRAIN_CFG is configs[1] (the multinomial over 25..49 lists 25, 29, .., 49), INFER_CFG
    is configs[3] at its first crop."""
    import bench
    t = bench.TRAIN_CFG
    net, C, K, B, crops, ign, _ = TRAIN_WORKLOADS["configs[1]"]
    assert (t["net"], t["C"], t["K"], t["batch"]) == (net, C, K, B)
    assert t["distribution"] == "multinomial" and list(range(t["values"][0], t["values"][-1] + 1)) == crops
    assert t["values"] == list(range(25, 50, 4))
    i = bench.INFER_CFG
    net, C, K, icrops, H, W = INFER_WORKLOADS["configs[3]"]
    assert (i["net"], i["C"], i["K"], i["crop"], i["H"], i["W"]) == (net, C, K, icrops[0], H, W)


# ------------------------------------------------------------------------------------------------ host mirrors
def conv_sched_class(U, mt, G):
    """Round structure of ConvSched (conv_tc.cuh:79-94) for U units on G CTAs."""
    if mt == 1:
        return "singles"
    rounds = U // (2 * G)
    r = U - 2 * G * rounds
    if rounds == 0:
        return "mixed round only"
    return "pairs, r=0" if r == 0 else ("pairs, r<=G" if r <= G else "pairs, r>G")


def conv_tc_launch(M, co, sm):
    """(mt, two CTAs, grid, units) of launch_conv_tc_t (conv_tc.cuh:597, 612, 621 and 638-639) for one N tile of co."""
    units = -(-M // BM)
    mt = 2 if co <= 128 and M > BM else 1
    two = co <= 64                                  # conv_tc_two_cta; EPI_C == 32 follows (launch_conv_tc, 668)
    grid = min(units, 2 * sm if two else sm)
    return mt, two, grid, units


def n_tiles_of(co):
    """The N tiles run_conv (drs_api.cu:721-727) splits co into."""
    n = 1
    while co // n > 256 or co % n or (co // n) % 32:
        n += 1
    return [co // n] * n


def wgrad_tc_launch(M, k, ci, co, sm, part_cap):
    """(T, which limit chose the split count, whole 64-pixel chunks) of launch_wgrad_tc (wgrad_tc.cuh:317-347)."""
    ci_pad, co_pad = -(-ci // 64) * 64, -(-co // 64) * 64
    n_tiles = (k * k * (ci_pad // 64) + 1) // 2
    acc = 64 if co_pad <= 64 else (128 if co_pad <= 128 else 256)
    T = 512 // acc
    while T > 1 and 3 * (T * 2 * 8192 + (co_pad // 64) * 8192) > 227 * 1024 - 2048:
        T -= 1
    T = min(T, n_tiles)
    n_groups = -(-n_tiles // T)
    n_chunks = -(-M // 64)
    lim = {"SM fill": max(1, sm // n_groups), "chunks/8": max(1, n_chunks // 8),
           "workspace": part_cap // (k * k * ci_pad * co_pad)}
    splits = min(lim.values())
    return T, next(n for n, v in lim.items() if v == splits), M % 64 == 0


def regime_signature(net, C, B, crop, sm):
    """{(layer, quantity, value)} of the bf16 training step at (B, crop): see the module docstring."""
    layers, _, _ = net_layers(net, C)
    M = B * crop * crop
    part_cap = max(L["k"] ** 2 * L["ci"] * L["co"] for L in layers) * 48      # TrainWs::layout, part_w_cap
    sig = set()
    for j, L in enumerate(layers):
        sc = L["scope"]
        if j == 0:                                   # conv1_tc (conv1_tc.cuh:330, 354), its filter gradient from xcol
            tiles = -(-M // BM)
            sig.add((sc, "conv1 tiles", "< SMs" if tiles < sm else ("multiple of SMs" if tiles % sm == 0 else "SMs + part")))
            wg = wgrad_tc_launch(M, 1, 128, L["co"], sm, part_cap)
        else:
            for what, ci, co in (("fwd", L["ci"], L["co"]), ("dgrad", L["co"], L["ci"])):
                for co_t in sorted(set(n_tiles_of(co))):
                    mt, two, grid, units = conv_tc_launch(M, co_t, sm)
                    sig.add((sc, "%s N%d" % (what, co_t), (mt, two, "tiles" if grid == units else "CTA limit",
                                                             conv_sched_class(units, mt, grid))))
            wg = wgrad_tc_launch(M, L["k"], L["ci"], L["co"], sm, part_cap) if wgrad_tc_supported(L["ci"], L["co"]) else None
        if wg:
            sig.add((sc, "wgrad_tc", wg))
        if L["post"] == ("max",):                    # launch_maxpool3_fwd (ops.cuh:386-389), _bwd_apply (474-477)
            _, seg, regime = pool_nseg(B, crop, L["co"], sm)
            for what in ("pool fwd", "pool bwd"):
                sig.add((sc, what, (regime, seg % 3)))
    return sig


def conv_units(net, C, B, crop, sm):
    """{(units, mt, grid)} of every tensor-core convolution launch of the step."""
    layers, _, _ = net_layers(net, C)
    M = B * crop * crop
    out = set()
    for L in layers[1:]:
        for co in (L["co"], L["ci"]):
            for co_t in set(n_tiles_of(co)):
                mt, _, grid, units = conv_tc_launch(M, co_t, sm)
                out.add((units, mt, grid))
    return out


def select_crops(net, C, B, crops, sm):
    """The smallest and the largest crop (every crop of an interval of at most four), then greedily the crop that adds the
    most signature values not yet reached (ties: the smaller crop), until every value of the interval is reached.  Returns
    (crops, coverage of the interval)."""
    sigs = {c: regime_signature(net, C, B, c, sm) for c in crops}
    want = set().union(*sigs.values())
    sel = sorted(set(crops) if len(crops) <= 4 else {min(crops), max(crops)})
    got = set().union(*(sigs[c] for c in sel))
    while got != want:
        c = max(crops, key=lambda c: (len(sigs[c] - got), -c))
        sel.append(c)
        got |= sigs[c]
    return sorted(sel), want


def test_crop_selection_covers_the_interval():
    """For every training workload the selected crops reach every signature value that any crop of its interval reaches;
    the smallest and largest crops are selected, and the regimes the selection is meant to tell apart do occur."""
    seen = set()
    for name, (net, C, K, B, crops, _, _) in TRAIN_WORKLOADS.items():
        sel, want = select_crops(net, C, B, crops, B200_SMS)
        assert min(crops) in sel and max(crops) in sel and set(sel) <= set(crops), name
        assert set().union(*(regime_signature(net, C, B, c, B200_SMS) for c in sel)) == want, name
        seen |= {v[3] for (_, q, v) in want if q.startswith(("fwd", "dgrad"))}
        print(name, "crops", sel, "of", len(crops), "reach", len(want), "signature values")
    assert {"singles", "mixed round only", "pairs, r<=G", "pairs, r>G"} <= seen, seen


def _sched_class_enumerated(lib, U, mt, G):
    """The round class read off the schedule drs_debug_conv_schedule enumerates (the kernel's own ConvSched): the full
    rounds are the pairs of the last CTA (it never takes a pair in the last round), the last round holds the rest."""
    from test_abi import _schedule
    sched = _schedule(lib, U, mt, G)
    pairs = sum(p for items in sched for _, p in items)
    if mt == 1:
        assert pairs == 0
        return "singles"
    rounds = sum(p for _, p in sched[G - 1])
    rest = U - 2 * G * rounds
    last_pairs = pairs - G * rounds
    assert 0 <= last_pairs and 0 <= rest < 2 * G
    if rounds == 0:
        return "mixed round only"
    return "pairs, r=0" if rest == 0 else ("pairs, r<=G" if last_pairs == 0 else "pairs, r>G")


def test_conv_sched_mirror_matches_enumeration(drs):
    """conv_sched_class agrees with the schedule the library enumerates for every (units, mt, grid) of every training
    workload's crops, on 148 SMs."""
    from drs_b200 import lib
    l = lib.load()
    shapes = set()
    for net, C, K, B, crops, _, _ in TRAIN_WORKLOADS.values():
        for c in crops:
            shapes |= conv_units(net, C, B, c, B200_SMS)
    classes = set()
    for U, mt, G in sorted(shapes):
        cls = conv_sched_class(U, mt, G)
        assert _sched_class_enumerated(l, U, mt, G) == cls, (U, mt, G)
        classes.add(cls)
    assert {"singles", "mixed round only", "pairs, r<=G", "pairs, r>G"} <= classes, classes


# ------------------------------------------------------------------------------------------------ training (GPU)
def draw_sequence(sel, rs):
    """Every selected crop once and two to five more drawn with repeats (6 to 8 steps in all), in a seeded order."""
    n = min(8, max(6, len(sel) + 2))
    seq = list(sel) + list(rs.choice(sel, n - len(sel)))
    return [int(c) for c in rs.permutation(seq)]


def _feeds(seq, B, C, K, ignore, isprs, seed):
    """Per step (x, y, accuracy mask or None) drawn from the seed; about 20 % of the labels are the ignored label."""
    rs = np.random.RandomState(seed)
    out = []
    for crop in seq:
        px = crop * crop
        x = rs.randn(B, px * C).astype(np.float32)
        y = rs.randint(0, K, size=(B, px)).astype(np.float32)
        if ignore is not None:
            y = np.where(rs.rand(B, px) < 0.2, ignore, y).astype(np.float32)
        am = (rs.rand(B, px) > 0.1).astype(np.uint8) if isprs else None
        out.append((x, y, am))
    return out


def _trainables(s):
    return {n: v for n, v in s.variables().items() if not n.endswith("/Momentum") and n != "global_step"}


def _nudge(s, scope):
    """The change of the sensitivity check: a layer's weights scaled by 17/16."""
    s.set_variable(scope + "/weights", s.get_variable(scope + "/weights") * np.float32(1.0625))


def run_eager_checked(drs, monkeypatch, wl, seq, feeds, p, mid, val, rs):
    """E: the sequence eager under DRS_DEBUG_KEEP=1, every step checked.  Returns per-step (loss, cm, n_correct, pred),
    the validation outputs and the final variables."""
    net, C, K, B, crops, ign, _ = TRAIN_WORKLOADS[wl]
    r = TrainRun(drs, monkeypatch, net, C, K, "bf16", B, seq[0], ignore=ign is not None, step=False)
    layers, _, act = net_layers(net, C)
    r.s.load_variables(p)
    _nudge(r.s, layers[1]["scope"])
    steps, vout = [], None
    try:
        for i, (crop, (x, y, am)) in enumerate(zip(seq, feeds)):
            if i == mid:                                 # (no tap copies of the validation pass: it is compared, not checked)
                monkeypatch.delenv("DRS_DEBUG_KEEP")
                vout = r.s.infer(val, max(crops))
                monkeypatch.setenv("DRS_DEBUG_KEEP", "1")
            r.crop, r.M, r.x, r.y = crop, B * crop * crop, x, y
            r.p = _trainables(r.s)                       # the weights move between steps
            loss, r.pred, r.cm, r.n_correct = r.s.train_step(x, y, crop, want_cm=True, acc_mask=am)
            r.loss = float(loss)
            steps.append((loss, r.cm, r.n_correct, r.pred.reshape(-1).astype(np.uint8)))
            r.collect()
            tag = "%s crop%d" % (wl, crop)
            idx = sample_pixels(B, crop, rs)
            taps = dict(r.taps, x=rounded(x.reshape(B, crop, crop, C), "bf16"))
            stats = {L["scope"]: (r.s.get_variable(L["scope"] + "/moving_mean"), r.s.get_variable(L["scope"] + "/moving_variance"))
                     for L in layers}
            res = train_forward_checks(layers, act, r.p, taps, stats, "bf16", B, crop, idx, tag)
            res.update(check_step([r], tag, idx=idx, wcols=_subset_cols(rs)))
            _assert_within(res, (wl, i, crop))
        final = r.s.variables()
    finally:
        r.close()
    return steps, vout, final


class ProductRun:
    """P: the product loop's use of a session (backend.GpuBackend): device buffers for the largest crop, reserve, the ignore
    label, graphs captured for every crop of the interval, train_step_async on its own stream, results fetched late."""

    def __init__(self, drs, wl, p, nudge=True, prepare=None):
        import torch
        net, C, K, B, crops, ign, isprs = TRAIN_WORKLOADS[wl]
        self.torch, self.B, self.C, self.K = torch, B, C, K
        self.stream = torch.cuda.Stream()
        n = B * max(crops) ** 2
        dev = torch.device("cuda")
        self.x = torch.empty(n * C, dtype=torch.float32, device=dev)
        self.y = torch.empty(n, dtype=torch.float32, device=dev)
        self.pred = torch.empty(n, dtype=torch.uint8, device=dev)
        self.amask = torch.empty(n, dtype=torch.uint8, device=dev) if isprs else None
        s = self.s = drs.Session(net, C, K, precision="bf16", bn_decay=0.0, weight_decay=0.0)
        s.load_variables(p)
        s.set_stream(self.stream.cuda_stream)
        s.reserve(B, max(crops), training=True)
        if ign is not None:
            s.set_ignore_label(ign)
        s.prepare_training(self.x, self.y, B, crops if prepare is None else prepare, pred_dev=self.pred, acc_mask_dev=self.amask)
        if nudge:
            _nudge(s, net_layers(net, C)[0][1]["scope"])
        self.tickets, self.preds, self.results = [], [], {}

    def submit(self, crop, x, y, am):
        """Copy the feeds into the fixed buffers on the session's stream (as the gather does), enqueue the step, keep a
        device copy of its pred behind it."""
        torch, n = self.torch, self.B * crop * crop
        with torch.cuda.stream(self.stream):
            self.x[:n * self.C].copy_(torch.from_numpy(x.reshape(-1)).pin_memory(), non_blocking=True)
            self.y[:n].copy_(torch.from_numpy(y.reshape(-1)).pin_memory(), non_blocking=True)
            if self.amask is not None:
                self.amask[:n].copy_(torch.from_numpy(am.reshape(-1)).pin_memory(), non_blocking=True)
            t = self.s.train_step_async(self.x, self.y, self.B, crop, pred_dev=self.pred, acc_mask_dev=self.amask)
            self.preds.append(self.pred[:n].clone())
        self.tickets.append(t)

    def fetch(self, keep=2):
        """Results of every step but the last `keep`."""
        for i, t in enumerate(self.tickets[:len(self.tickets) - keep]):
            if i not in self.results:
                self.results[i] = self.s.train_result(t)


def run_product(drs, monkeypatch, wl, seq, feeds, p, mid, val):
    """P: the sequence through prepared graphs, the validation infer at step `mid`.  Returns per-step results, the
    validation outputs, the drop of free device memory across the validation and the final variables."""
    import torch
    monkeypatch.delenv("DRS_DEBUG_KEEP", raising=False)
    net, C, K, B, crops, _, _ = TRAIN_WORKLOADS[wl]
    P = ProductRun(drs, wl, p)
    try:
        vdev = torch.from_numpy(val.reshape(-1)).cuda()
        nv = val.shape[0] * max(crops) ** 2
        vlog = torch.empty(nv * K, dtype=torch.float32, device="cuda")
        vpred = torch.empty(nv, dtype=torch.uint8, device="cuda")
        drop = None
        for i, (crop, (x, y, am)) in enumerate(zip(seq, feeds)):
            if i == mid:
                P.fetch(keep=0)
                torch.cuda.synchronize()
                free0 = torch.cuda.mem_get_info()[0]
                with torch.cuda.stream(P.stream):
                    P.s.infer_dev(vdev, val.shape[0], max(crops), vlog, vpred)
                P.s.synchronize()
                drop = free0 - torch.cuda.mem_get_info()[0]
            P.submit(crop, x, y, am)
            P.fetch()
        P.fetch(keep=0)
        P.s.synchronize()
        steps = [(P.results[i][0], P.results[i][1], P.results[i][2], P.preds[i].cpu().numpy()) for i in range(len(seq))]
        vout = (vpred.cpu().numpy(), vlog.cpu().numpy())
        final = P.s.variables()
    finally:
        P.s.close()
    return steps, vout, drop, final


def _same_step(a, b):
    return (np.float32(a[0]).tobytes() == np.float32(b[0]).tobytes() and np.array_equal(a[1], b[1]) and a[2] == b[2]
            and np.array_equal(a[3], b[3]))


@pytest.mark.gpu
@pytest.mark.parametrize("wl", list(TRAIN_WORKLOADS), ids=_ids(TRAIN_WORKLOADS))
def test_workload_training_sequence(drs, monkeypatch, wl):
    import torch
    net, C, K, B, crops, ign, isprs = TRAIN_WORKLOADS[wl]
    sm = torch.cuda.get_device_properties(0).multi_processor_count
    t0 = time.time()
    sel, want = select_crops(net, C, B, crops, sm)
    rs = np.random.RandomState(61 + list(TRAIN_WORKLOADS).index(wl))
    seq = draw_sequence(sel, rs)
    reached = set().union(*(regime_signature(net, C, B, c, sm) for c in seq))
    print("\n%s: crops %s of %d-%d, sequence %s, %d of %d signature values reached" % (wl, sel, min(crops), max(crops), seq,
                                                                                     len(reached), len(want)))
    assert reached == want, sorted(want - reached)
    feeds = _feeds(seq, B, C, K, ign, isprs, 67)
    from oracle import nets_torch
    p = nets_torch.init_params(net, C, K, seed=5)
    mid = len(seq) // 2
    val = rs.randn(16 * B, max(crops) ** 2 * C).astype(np.float32)     # a validation batch larger than the reserved one
    e_steps, e_val, e_final = run_eager_checked(drs, monkeypatch, wl, seq, feeds, p, mid, val, rs)
    _print_report("%s, E checked" % wl, time.time() - t0)
    p_steps, p_val, drop, p_final = run_product(drs, monkeypatch, wl, seq, feeds, p, mid, val)
    print("%s: validation infer at B %d, crop %d: free device memory dropped by %.0f MB" % (wl, 16 * B, max(crops), drop / 2 ** 20))
    # the grown arena: nothing else an infer_dev on caller buffers allocates (the folded eval weights) takes more than a few MB
    assert drop > 32 * 2 ** 20, drop
    bad = [i for i, (a, b) in enumerate(zip(e_steps, p_steps)) if not _same_step(a, b)]
    assert not bad, ("steps differ between eager and graph replay", [(i, seq[i], e_steps[i][0], p_steps[i][0]) for i in bad])
    assert np.array_equal(e_val[0].reshape(-1), p_val[0].astype(np.int64)) and np.array_equal(e_val[1].reshape(-1), p_val[1]), wl
    assert set(e_final) == set(p_final)
    diff = [n for n in e_final if not np.array_equal(e_final[n], p_final[n])]
    assert not diff, ("variables differ", diff)
    assert e_final["global_step"][0] == len(seq)
    # the comparison can fail: without the change made after prepare, the first step already differs
    monkeypatch.delenv("DRS_DEBUG_KEEP", raising=False)
    P0 = ProductRun(drs, wl, p, nudge=False, prepare=[seq[0]])
    try:
        P0.submit(seq[0], *feeds[0])
        P0.fetch(keep=0)
        P0.s.synchronize()
        assert not _same_step(e_steps[0], (P0.results[0][0], P0.results[0][1], P0.results[0][2], P0.preds[0].cpu().numpy()))
    finally:
        P0.s.close()
    print("%s: %d steps bit-identical eager vs replayed, %.1f s" % (wl, len(seq), time.time() - t0))


# ------------------------------------------------------------------------------------------------ inference (GPU)
def scene_chunks(crop, H, W, sm):
    """Batches of scene_infer_impl (drs_scene_api.cuh:466-470) over an H x W scene: the chunk and the last partial one."""
    from drs_b200 import session
    P = len(session.grid_positions(H, W, crop, 64))
    chunk = max(1, min(P, sm * 40 * BM // (crop * crop)))
    return sorted({chunk, P - (ceil(P / chunk) - 1) * chunk})


@pytest.mark.gpu
@pytest.mark.parametrize("wl", list(INFER_WORKLOADS), ids=_ids(INFER_WORKLOADS))
def test_workload_inference_chunks(drs, wl):
    """InferRun at the scene pass's chunk sizes, f16 and bf16, sampled pixels; prints the maxpool3_classifier regime."""
    net, C, K, icrops, H, W = INFER_WORKLOADS[wl]
    import torch
    sm = torch.cuda.get_device_properties(0).multi_processor_count
    rs = np.random.RandomState(71)
    p = params_with_stats(net, C, K, 5)
    layers, _, _ = net_layers(net, C)
    t0 = time.time()
    for crop in icrops:
        for B in scene_chunks(crop, H, W, sm):
            print("%s crop %d batch %d: maxpool3_classifier nseg %s" % (wl, crop, B, nseg_class(B, crop, layers[-1]["co"], sm)))
            x = rs.randn(B, crop * crop * C).astype(np.float32)
            for prec in ("f16", "bf16"):
                run = InferRun(drs, net, C, K, prec, p, x, B, crop)
                _assert_within(run.check("%s crop%d B%d" % (wl, crop, B), sample_pixels(B, crop, rs)), (wl, prec, B, crop))
                del run
    _print_report(wl + " inference", time.time() - t0)
