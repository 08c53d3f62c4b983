"""The full-scene pass at the benchmark's inference shapes, bit for bit against a checked reference, and contest grids that
visit a lattice cell more than twice.

Workloads (the nets of test_gpu_workload_shapes.INFER_WORKLOADS, the scenes of synth, batch 64 as bench.INFER_CFG):

    configs[3]          dilated_grsl_rate8  C 5  K 6  potsdam 6000 x 6000 float64  isprs grid    crops 25, 65
    configs[4] contest  dilated_grsl_rate8  C 3  K 7  contest 3989 x 2830 float32  contest grid  crops 25, 49

Sessions are f16 as in the bench, plus bf16 at crop 65, with the variables of params_with_stats (non-trivial folded BN).
On a square scene the contest grid equals the isprs grid, hence the contest-shaped scene.

Host mirrors (CPU):
  pass_chunk     the chunk size of scene_infer_impl (drs_scene_api.cuh): min(P, SMs * waves * 128 / crop^2), waves 40;
  accum_ranges   the split of every chunk into visit ranges that accumulate_kernel can order in one launch (at most
                 ACCUM_MAX_CONTRIB = 32 contributions per pixel), restated per pixel; coverage() checks each range by brute
                 force, and that a range ended by a split could not have taken one more visit.

E, the checked reference (GPU + NumPy): the pass's grid chunk by chunk, gather_dev and infer_dev into device buffers, the
logits streamed to the host and added into a float32 [H, W, K] map in visit order with the visit counts (host_np's
accumulate_argmax without holding every logit), then the float64 mean and the first argmax.  Gathered patches of the first
and last chunk and every patch on the right or bottom edge equal host_np.apply_plan; the first, a middle and the last
partial chunk run through InferRun (the float64 layer checks of test_gpu_forward_layers) and its logits equal E's.

P, the product path as bench.py runs it: the session on a torch stream, the warm-up stripe, the resident scene_infer, the
same pass profiled, DRS_CHUNK_WAVES=7, row stripes of 2, 4 and 8 ranks from partial uploads, and scene_infer_host
(streamed upload) on a fresh session.  Every one equals E's label map and float64 mean map bit for bit, and a pass launches
exactly E's gathers and forwards plus one accumulation per range and the argmax.

Tall contest scenes (3000 x 300 crop 25, 3989 x 600 crop 49) visit a cell up to 11 and 8 times; before the chunks were
split into ranges, their accumulation failed with "a pixel is covered by more than 32 patch visits".

The GPU tests take about 3.5 minutes on one B200 (1000 W power limit): 31 to 47 s per scene-pass case, 22 to 28 s of it the
InferRun layer checks, and under 2 s for each tall-scene test.  Peak host memory is 8.2 GB, reached by configs[3] at crop
25: the float64 scene (1.4 GB), the float32 sum map (0.9 GB) and two float64 mean maps (1.7 GB each).
"""
import resource
import time

import numpy as np
import pytest

from test_gpu_backward_layers import _assert_within
from test_gpu_forward_layers import InferRun, params_with_stats, sample_pixels
from test_gpu_workload_shapes import B200_SMS, BM, INFER_WORKLOADS, _ids

BATCH = 64
ACCUM_MAX_CONTRIB = 32                               # scene.cuh
# name -> (workload of INFER_WORKLOADS, synth scene, grid, crops)
SCENE_PASSES = {
    "configs[3]": ("configs[3]", "potsdam", "isprs", (25, 65)),
    "configs[4] contest": ("configs[4] contest", "contest", "contest", (25, 49)),
}
CASES = [("configs[3]", 25, "f16"), ("configs[3]", 65, "f16"), ("configs[3]", 65, "bf16"),
         ("configs[4] contest", 25, "f16"), ("configs[4] contest", 49, "f16")]
CASE_IDS = ["%s-crop%d-%s" % (_ids([wl])[0], crop, prec) for wl, crop, prec in CASES]
# contest grids on tall scenes: (H, W, crop)
TALL = ((3000, 300, 25), (3989, 600, 49))
COFFEE = (500, 500, (25, 33, 41))                    # bench's coffee tiles (square) and crops


def scene_shape(wl):
    from drs_b200 import synth
    sp = synth.SHAPES[SCENE_PASSES[wl][1]]
    return sp["H"], sp["W"]


def geometries():
    """(name, H, W, crop, grid) of every scene pass of the table."""
    out = []
    for wl, (_, _, grid, crops) in SCENE_PASSES.items():
        H, W = scene_shape(wl)
        out += [("%s crop %d" % (wl, c), H, W, c, grid) for c in crops]
    return out


# ------------------------------------------------------------------------------------------------ host mirrors
def pass_chunk(P, crop, sm, waves=40):
    """Patches per chunk of scene_infer_impl (drs_scene_api.cuh: chunk = whole 128-pixel tiles for `waves` waves)."""
    return max(1, min(P, sm * waves * BM // (crop * crop)))


def accum_ranges(pos, H, W, crop, chunk, limit=ACCUM_MAX_CONTRIB):
    """accum_ranges of drs_scene_api.cuh, per pixel: every chunk starts a range; a range ends before the visit that would
    give a pixel it covers more than `limit` contributions.  Returns the cuts, ranges [cuts[r], cuts[r + 1])."""
    cnt = np.zeros((H, W), np.uint8)
    cuts, lo, hi = [], H, 0
    for p, (y, x) in enumerate(np.asarray(pos).tolist()):
        win = cnt[y:y + crop, x:x + crop]
        if p % chunk == 0 or win.max() >= limit:
            cuts.append(p)
            cnt[lo:hi] = 0
            lo, hi = H, 0
        win += 1
        lo, hi = min(lo, y), max(hi, y + crop)
    return cuts + [len(pos)]


def coverage(pos, crop, W):
    """Largest number of the given patches that cover one pixel (brute force over the rows they touch)."""
    pos = np.asarray(pos, dtype=np.int64)
    y0 = int(pos[:, 0].min())
    r, c = pos[:, 0] - y0, pos[:, 1]
    d = np.zeros((int(r.max()) + crop + 1, W + 1), np.int32)
    for dr, dc, v in ((0, 0, 1), (crop, 0, -1), (0, crop, -1), (crop, crop, 1)):
        np.add.at(d, (r + dr, c + dc), v)
    return int(d.cumsum(0).cumsum(1).max())


def check_ranges(name, pos, H, W, crop, chunk):
    """The mirrored ranges of a pass: within the limit (brute force), maximal where they split, every chunk starting one.
    Returns (cuts, per-chunk peak contributions of one pixel)."""
    P = len(pos)
    cuts = accum_ranges(pos, H, W, crop, chunk)
    starts = set(range(0, P, chunk))
    assert starts <= set(cuts[:-1]) and cuts[-1] == P and cuts == sorted(set(cuts)), name
    for a, b in zip(cuts[:-1], cuts[1:]):
        assert coverage(pos[a:b], crop, W) <= ACCUM_MAX_CONTRIB, (name, a, b)
        if b < P and b not in starts:
            assert coverage(pos[a:b + 1], crop, W) > ACCUM_MAX_CONTRIB, (name, a, b)
    peaks = [coverage(pos[s:s + chunk], crop, W) for s in range(0, P, chunk)]
    return cuts, peaks


def cell_visits(pos):
    """Largest number of visits of one lattice cell (a cell is a patch origin)."""
    _, n = np.unique(np.asarray(pos), axis=0, return_counts=True)
    return int(n.max())


def test_grid_positions_match_the_numpy_grid(drs):
    """The library's visiting order equals host_np's restatement of create_patches_per_map at every workload shape, on
    the tall contest scenes and on the coffee tiles."""
    from oracle import host_np
    shapes = [(H, W, c, g) for _, H, W, c, g in geometries()] + [(H, W, c, "contest") for H, W, c in TALL]
    shapes += [(COFFEE[0], COFFEE[1], c, "coffee") for c in COFFEE[2]]
    for H, W, crop, grid in shapes:
        pos = drs.grid_positions(H, W, crop, BATCH, grid)
        ref = np.array(host_np.all_patch_positions(H, W, crop, BATCH, grid), dtype=np.int32)
        assert np.array_equal(pos, ref), (H, W, crop, grid)


def test_workload_table_matches_bench_and_synth():
    """Batch and net of configs[3] are bench.INFER_CFG's; the synth scenes have the channels and classes of the nets."""
    import bench
    from drs_b200 import synth
    assert bench.INFER_CFG["batch"] == BATCH and bench.INFER_CFG["dataset"] == SCENE_PASSES["configs[3]"][1]
    for wl, (iwl, kind, _, crops) in SCENE_PASSES.items():
        net, C, K, _, _, _ = INFER_WORKLOADS[iwl]
        assert (synth.SHAPES[kind]["C"], synth.SHAPES[kind]["K"]) == (C, K), wl
        assert INFER_WORKLOADS[iwl][3][0] == crops[0]
    assert SCENE_PASSES["configs[3]"][3] == INFER_WORKLOADS["configs[3]"][3]


def test_chunk_rule_reaches_the_edges(drs):
    """At 148 SMs every workload shape ends in a partial chunk and has chunks that start inside a grid row; the isprs grid
    reaches the shifted last row and column, the contest grid the shifted last column, leaves the bottom rows unvisited
    and visits some cell three times."""
    visits = {}
    for name, H, W, crop, grid in geometries():
        pos = drs.grid_positions(H, W, crop, BATCH, grid)
        P, stride = len(pos), crop // 2
        chunk = pass_chunk(P, crop, B200_SMS)
        starts = np.arange(0, P, chunk)
        inside = int((pos[starts, 1] != 0).sum())
        visits[name] = cell_visits(pos)
        print("%s: %d patches, chunk %d, %d chunks, last %d, %d chunks start inside a grid row, cells visited up to %d times"
              % (name, P, chunk, len(starts), P - starts[-1], inside, visits[name]))
        assert P % chunk != 0, name
        assert inside > 0, name
        assert (H - crop) % stride and (W - crop) % stride, name
        assert (pos[:, 1] == W - crop).any(), name
        if grid == "isprs":
            assert visits[name] == 1 and (pos[:, 0] == H - crop).any(), name
        else:
            # contest: the batch offsets divide by the row count, so the walk stops short of the bottom of a scene taller
            # than wide; those rows keep occur 0 (-> 1) and label 0 (bug F10)
            assert pos[:, 0].max() + crop < H, name
    assert max(v for n, v in visits.items() if "contest" in n) >= 3, visits


def test_accumulation_ranges_stay_within_the_kernel_limit(drs):
    """Every mirrored range keeps each pixel within 32 contributions and ends only where the next visit would exceed it;
    the isprs and coffee grids never split a chunk, the tall contest scenes must."""
    rows = []
    for name, H, W, crop, grid in geometries():
        pos = drs.grid_positions(H, W, crop, BATCH, grid)
        chunk = pass_chunk(len(pos), crop, B200_SMS)
        cuts, peaks = check_ranges(name, pos, H, W, crop, chunk)
        rows.append((name, chunk, max(peaks), len(cuts) - 1, -(-len(pos) // chunk)))
        if grid == "isprs":
            assert cuts == list(range(0, len(pos), chunk)) + [len(pos)], name
    for crop in COFFEE[2]:
        H, W = COFFEE[:2]
        pos = drs.grid_positions(H, W, crop, BATCH, "coffee")
        name = "coffee %dx%d crop %d" % (H, W, crop)
        cuts, peaks = check_ranges(name, pos, H, W, crop, len(pos))
        assert cuts == [0, len(pos)], name
        rows.append((name, len(pos), max(peaks), 1, 1))
    for H, W, crop in TALL:
        pos = drs.grid_positions(H, W, crop, BATCH, "contest")
        name = "contest %dx%d crop %d" % (H, W, crop)
        for chunk in (pass_chunk(len(pos), crop, B200_SMS), len(pos)):       # the scene pass, accumulate_argmax
            cuts, peaks = check_ranges(name, pos, H, W, crop, chunk)
            assert max(peaks) > ACCUM_MAX_CONTRIB and len(cuts) - 1 > -(-len(pos) // chunk), name
            rows.append((name, chunk, max(peaks), len(cuts) - 1, -(-len(pos) // chunk)))
    for name, chunk, peak, n, nch in rows:
        print("%-34s chunk %6d: peak %3d contributions per pixel and chunk, %4d ranges for %4d chunks" % (name, chunk, peak, n, nch))


# ------------------------------------------------------------------------------------------------ E, the checked reference (GPU)
def _same_bits(a, b):
    a, b = np.ascontiguousarray(a), np.ascontiguousarray(b)
    return a.shape == b.shape and a.dtype == b.dtype and np.array_equal(a.view(np.uint8), b.view(np.uint8))


def _mean_of(prob, occ):
    """host_np.accumulate_argmax's tail: occur 0 -> 1, float64 divide."""
    mean = prob.astype(np.float64)
    mean /= np.maximum(occ, 1)[..., None].astype(np.float64)
    return mean


def _add_clipped(band, y_lo, lg, pos, crop):
    """Add the logits of the patches at `pos` to the rows [y_lo, y_lo + len(band)) of a map, in order."""
    y_hi = y_lo + band.shape[0]
    for j, (y, x) in enumerate(pos):
        a, b = max(y, y_lo), min(y + crop, y_hi)
        if a < b:
            band[a - y_lo:b - y_lo, x:x + crop] += lg[j, a - y:b - y]


def checked_reference(drs, s, img, mean_full, std_full, pos, crop, chunk, K, keep):
    """E (see the module docstring).  `keep`: chunk indices whose gathered input and logits are returned.  Also returns
    two wrong references: the middle chunk added in reverse visit order, and the last chunk dropped (as bands of rows)."""
    import torch
    from oracle import host_np
    H, W, C = img.shape
    P = len(pos)
    starts = list(range(0, P, chunk))
    rev, last = len(starts) // 2, len(starts) - 1
    x = torch.empty(chunk * crop * crop * C, dtype=torch.float32, device="cuda")
    lg = torch.empty(chunk * crop * crop * K, dtype=torch.float32, device="cuda")
    lg_host = torch.empty(chunk * crop * crop * K, dtype=torch.float32, pin_memory=True)
    prob = np.zeros((H, W, K), np.float32)
    occ = np.zeros((H, W), np.uint32)
    kept, rev_band, drop_band, n_gather = {}, None, None, 0
    for ci, s0 in enumerate(starts):
        nb = min(chunk, P - s0)
        cp = pos[s0:s0 + nb]
        inst = np.concatenate([np.zeros((nb, 1), np.int32), cp], 1)
        s.gather_dev(inst, None, crop, x)
        s.infer_dev(x, nb, crop, lg)
        s.synchronize()
        n = nb * crop * crop
        lg_host[:n * K].copy_(lg[:n * K])
        L = lg_host[:n * K].numpy().reshape(nb, crop, crop, K)
        # gathered patches: whole first and last chunk, every patch on the right or bottom edge
        sel = np.arange(nb) if ci in (0, last) else np.nonzero((cp[:, 0] == H - crop) | (cp[:, 1] == W - crop))[0]
        if len(sel):
            got = x[:n * C].view(nb, crop, crop, C)[torch.from_numpy(sel).cuda()].cpu().numpy()
            ref, _ = host_np.apply_plan([img], None, inst[sel], None, crop, mean_full, std_full)
            assert _same_bits(got, ref.astype(np.float32)), ("gathered patches differ", ci)
            n_gather += len(sel)
        if ci in keep:
            kept[ci] = (x[:n * C].cpu().numpy().reshape(nb, -1), L.copy())
        y_lo, y_hi = int(cp[:, 0].min()), int(cp[:, 0].max()) + crop
        if ci == last:
            drop_band = (y_lo, prob[y_lo:y_hi].copy(), occ[y_lo:y_hi].copy())
        if ci == rev:
            rev_band = (y_lo, prob[y_lo:y_hi].copy())
            _add_clipped(rev_band[1], y_lo, L[::-1], cp[::-1], crop)
        elif rev_band is not None:
            _add_clipped(rev_band[1], rev_band[0], L, cp, crop)
        for j, (y, xx) in enumerate(cp.tolist()):
            prob[y:y + crop, xx:xx + crop] += L[j]
            occ[y:y + crop, xx:xx + crop] += 1
    mean = _mean_of(prob, occ)
    del prob
    labels = np.argmax(mean, axis=2).astype(np.uint8)
    y0, band = rev_band
    rev_mean = _mean_of(band, occ[y0:y0 + band.shape[0]])
    y1, dprob, docc = drop_band
    drop_mean = _mean_of(dprob, docc)
    return labels, mean, kept, (y0, rev_mean), (y1, drop_mean), n_gather


def _peak_rss_gb():
    return resource.getrusage(resource.RUSAGE_SELF).ru_maxrss / 2 ** 20


@pytest.mark.gpu
@pytest.mark.parametrize("wl,crop,prec", CASES, ids=CASE_IDS)
def test_scene_pass_equals_checked_reference(drs, monkeypatch, wl, crop, prec):
    import torch
    from drs_b200 import dist as ddist, synth
    t0 = time.time()
    iwl, kind, grid, _ = SCENE_PASSES[wl]
    net, C, K, _, _, _ = INFER_WORKLOADS[iwl]
    img, _ = synth.scene(kind)
    H, W = img.shape[:2]
    mean_full, std_full = synth.normalisation(img)
    p = params_with_stats(net, C, K, 5)
    sm = torch.cuda.get_device_properties(0).multi_processor_count
    pos = drs.grid_positions(H, W, crop, BATCH, grid)
    P = len(pos)
    chunk = pass_chunk(P, crop, sm)
    n_chunks = -(-P // chunk)
    cuts = accum_ranges(pos, H, W, crop, chunk)
    tag = "%s crop %d %s" % (wl, crop, prec)
    print("\n%s: %d patches, chunk %d, %d chunks, %d accumulation ranges" % (tag, P, chunk, n_chunks, len(cuts) - 1))
    stream = torch.cuda.Stream()

    def session():
        s = drs.Session(net, C, K, precision=prec)
        s.load_variables(p)
        s.set_stream(stream.cuda_stream)
        s.set_normalization(mean_full, std_full)
        return s

    def same_as_e(got, what, rows=(0, H)):
        gl, gm = got
        assert np.array_equal(gl, e_labels[rows[0]:rows[1]]), (tag, what, "labels")
        assert _same_bits(gm, e_mean[rows[0]:rows[1]]), (tag, what, "mean")

    s = session()
    try:
        s.upload_scene(0, img, None)
        s.scene_infer(0, crop, BATCH, H, W, variant=grid, row_begin=0, row_end=40)        # the bench's warm-up stripe
        l0 = s.launch_count
        keep = (0, n_chunks // 2, n_chunks - 1)
        e_labels, e_mean, kept, (y_rev, rev_mean), (y_drop, drop_mean), n_gather = checked_reference(
            drs, s, img, mean_full, std_full, pos, crop, chunk, K, keep)
        e_launches = s.launch_count - l0
        t_e = time.time() - t0
        # P: the resident pass, as the bench times it
        l0 = s.launch_count
        got = s.scene_infer(0, crop, BATCH, H, W, variant=grid, want_mean=True)
        launches = s.launch_count - l0
        print("%s: E %d launches, pass %d launches (%d ranges + argmax more)" % (tag, e_launches, launches, len(cuts) - 1))
        assert launches == e_launches + len(cuts) - 1 + 1, (launches, e_launches, len(cuts))
        same_as_e(got, "resident")
        # the wrong references differ from the product's map
        assert not _same_bits(got[1][y_rev:y_rev + len(rev_mean)], rev_mean), (tag, "reversed chunk not detected")
        assert not _same_bits(got[1][y_drop:y_drop + len(drop_mean)], drop_mean), (tag, "dropped chunk not detected")
        del got
        s.set_profiling(True)
        got = s.scene_infer(0, crop, BATCH, H, W, variant=grid, want_mean=True)
        conv_ms, conv_n, _ = s.profile_read()
        s.set_profiling(False)
        assert conv_n > 0 and conv_ms > 0, (conv_ms, conv_n)
        same_as_e(got, "profiled")
        del got
        monkeypatch.setenv("DRS_CHUNK_WAVES", "7")
        assert pass_chunk(P, crop, sm, 7) < chunk
        same_as_e(s.scene_infer(0, crop, BATCH, H, W, variant=grid, want_mean=True), "DRS_CHUNK_WAVES=7")
        monkeypatch.delenv("DRS_CHUNK_WAVES")
        if grid == "contest":
            wrong = s.scene_infer(0, crop, BATCH, H, W, variant="isprs")
            assert not np.array_equal(wrong, e_labels), (tag, "isprs grid on the contest scene not detected")
        for world in (2, 4, 8):
            for r in range(world):
                a, b = ddist.stripe_bounds(H, world, r)
                lo, hi = ddist.stripe_rows_needed(H, crop, a, b)
                s.upload_scene(0, img, None, lo, hi)
                same_as_e(s.scene_infer(0, crop, BATCH, H, W, variant=grid, row_begin=a, row_end=b, want_mean=True),
                          "stripe %d of %d" % (r, world), (a, b))
    finally:
        s.close()
    s = session()
    try:
        same_as_e(s.scene_infer_host(0, img, crop, BATCH, variant=grid, want_mean=True), "streamed upload")
    finally:
        s.close()
    t_p = time.time() - t0 - t_e
    # E tied to the float64 layer checks: its logits are those of InferRun on the same gathered input
    rs = np.random.RandomState(73)
    for ci in keep:
        xk, lk = kept[ci]
        nb = xk.shape[0]
        run = InferRun(drs, net, C, K, prec, p, xk, nb, crop)
        _assert_within(run.check("%s chunk %d" % (tag, ci), sample_pixels(nb, crop, rs)), (tag, ci))
        assert _same_bits(run.logits.reshape(lk.shape), lk), (tag, "chunk %d logits differ from InferRun's" % ci)
        del run
    print("%s: %d gathered patches checked; E %.0f s, P %.0f s, layer checks %.0f s; peak host memory %.1f GB"
          % (tag, n_gather, t_e, t_p, time.time() - t0 - t_e - t_p, _peak_rss_gb()))


# ------------------------------------------------------------------------------------------------ tall contest scenes (GPU)
@pytest.mark.gpu
@pytest.mark.parametrize("H,W,crop", TALL)
def test_tall_contest_accumulate_argmax(drs, H, W, crop):
    """accumulate_argmax on a contest grid that visits a cell up to 11 (8) times equals host_np bit for bit, in one launch
    per mirrored range plus the argmax; the isprs grid of the same scene takes one launch."""
    import torch
    from oracle import host_np
    K = 7
    s = drs.Session("dilated_grsl", 3, K, precision="fp32")
    try:
        for grid in ("contest", "isprs"):
            pos = drs.grid_positions(H, W, crop, BATCH, grid)
            g = torch.Generator(device="cuda").manual_seed(17)
            logits = torch.randn(len(pos), crop, crop, K, device="cuda", generator=g)
            l0 = s.launch_count
            labels, mean = s.accumulate_argmax(logits, pos, crop, H, W, want_mean=True)
            launches = s.launch_count - l0
            ranges = len(accum_ranges(pos, H, W, crop, len(pos))) - 1
            print("%dx%d crop %d %s grid: cells visited up to %d times, %d ranges" % (H, W, crop, grid, cell_visits(pos), ranges))
            assert launches == ranges + 1, (grid, launches, ranges)
            assert (ranges > 1) == (grid == "contest")
            ref_l, ref_m = host_np.accumulate_argmax(logits.cpu().numpy(), pos, H, W, crop, return_mean=True)
            assert np.array_equal(labels, ref_l.astype(np.uint8)) and _same_bits(mean, ref_m), grid
    finally:
        s.close()


@pytest.mark.gpu
def test_tall_contest_scene_infer_matches_patchwise_loop(drs):
    """scene_infer on the 3000 x 300 contest grid == grid -> gather -> normalise -> net -> ordered accumulate -> argmax run
    patch-wise through the same session (as test_scene_infer_matches_patchwise_oracle_loop)."""
    from drs_b200 import synth
    from oracle import host_np
    H, W, crop = TALL[0]
    img, _ = synth.scene("contest", H=H, W=W, seed=31)
    mean_full, std_full = synth.normalisation(img)
    s = drs.Session("dilated_grsl", 3, 7, precision="f16", seed=2)
    try:
        s.upload_scene(0, img, None)
        s.set_normalization(mean_full, std_full)
        labels, mean = s.scene_infer(0, crop, BATCH, H, W, variant="contest", want_mean=True)
        pos = np.array(host_np.all_patch_positions(H, W, crop, BATCH, "contest"), dtype=np.int32)
        xr, _ = host_np.apply_plan([img], None, [(0, r, c) for r, c in pos], None, crop, mean_full, std_full)
        _, logits = s.infer(xr.reshape(len(pos), -1), crop)
    finally:
        s.close()
    ref_l, ref_m = host_np.accumulate_argmax(logits, pos, H, W, crop, return_mean=True)
    assert np.array_equal(labels, ref_l.astype(np.uint8)) and _same_bits(mean, ref_m)
