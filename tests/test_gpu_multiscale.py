"""GPU: the multi-scale evaluation on the device (drs_scene_infer_multiscale) against the NumPy composition of
validate_test_multiscale (isprs:1380-1411), bit for bit.

H, the host composition: for each crop in order, the mean map of one scene pass (scene_infer(want_mean=True): prob_im /
occur_im in float64), cast to float32, loops.reference_softmax; np.sum over the scales; np.argmax.  The device pass must
return the same label map and the same float32 sum, on the isprs grid of a Vaihingen-shaped scene that takes several chunks
per pass (DRS_CHUNK_WAVES=3) and on a tall contest scene whose grid visits lattice cells several times, in f16 and fp32;
in row stripes; with the device confusion matrix; and refusing bad calls without leaving anything half done.  The kernel
alone is also fed means over the whole float32 range of exp, for every class count up to 8.
"""
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

# (synth kind, H, W, net channels, classes, grid, crops in evaluation order)
SCENES = (("vaihingen", 400, 300, 4, 6, "isprs", (31, 25, 45)),
          ("contest", 600, 120, 3, 7, "contest", (25, 33, 19)))


def host_composition(s, scene_id, crops, batch, H, W, variant, row_begin=0, row_end=None):
    """(labels, float32 sum) of validate_test_multiscale's NumPy composition over the device's mean maps."""
    K = s.num_classes
    probs = []
    for c in crops:
        _, mean = s.scene_infer(scene_id, c, batch, H, W, variant=variant, row_begin=row_begin, row_end=row_end, want_mean=True)
        probs.append(loops_softmax(mean.astype(np.float32), K))
    psum = np.sum(np.stack(probs), axis=0)
    return np.argmax(psum, axis=2), psum


def loops_softmax(a, K):
    from drs_b200 import loops
    return loops.reference_softmax(a, K)


def same_bits(a, b):
    return a.dtype == b.dtype == np.float32 and np.array_equal(a.view(np.uint32), b.view(np.uint32))


def session_with_scene(drs, kind, H, W, C, K, prec, seed=3, labels=True):
    from drs_b200 import synth
    img, lab = synth.scene(kind, H=H, W=W, block=16, unlabelled=True)
    mean, std = synth.normalisation(img)
    s = drs.Session("dilated_grsl", C, K, precision=prec, seed=seed)
    s.set_normalization(mean, std)
    s.upload_scene(0, img, lab if labels else None)
    return s, img, lab, mean, std


@pytest.mark.parametrize("prec", ["f16", "fp32"])
def test_multiscale_equals_host_composition(drs, monkeypatch, prec):
    """1, 2 and 3 scales: labels and the float32 sum equal the host composition bit for bit, on a chunked isprs pass and on a
    contest grid that visits cells several times."""
    monkeypatch.setenv("DRS_CHUNK_WAVES", "3")            # ~90 patches of crop 25 per chunk: several chunks per pass
    batch = 16
    for kind, H, W, C, K, grid, crops in SCENES:
        s, *_ = session_with_scene(drs, kind, H, W, C, K, prec)
        with s:
            for n in (1, 2, 3):
                ref_l, ref_sum = host_composition(s, 0, crops[:n], batch, H, W, grid)
                lab, psum = s.scene_infer_multiscale(0, crops[:n], batch, H, W, variant=grid, want_sum=True)
                assert lab.shape == (H, W) and psum.shape == (H, W, K)
                assert same_bits(psum, ref_sum), (kind, prec, n)
                assert np.array_equal(lab, ref_l), (kind, prec, n)
                if n == 1:                                 # one scale: the softmax of the single-scale mean map
                    single = s.scene_infer(0, crops[0], batch, H, W, variant=grid)
                    assert (lab == single).mean() > 0.999


@pytest.mark.parametrize("K", [2, 6, 7, 8])
def test_multiscale_kernel_over_the_whole_range_of_means(drs, K):
    """The device build of the softmax (multiscale_softmax_add_kernel, one launch per scale through
    drs_debug_multiscale_softmax_add) on means a trained or an untrained net may give: logit-like values, the whole of
    [-104, 89], the band [-104, -87.3] whose exp is denormal, and means above 88.72 whose exp overflows (the NumPy sum is then
    NaN and np.argmax takes the first NaN); counts 0 (read as 1) to 12.  Two scales: the float32 sum equals the NumPy
    composition bit for bit (NaN where it has NaN) and the labels equal its np.argmax, for every class count up to 8."""
    from drs_b200 import loops
    rs = np.random.RandomState(K)
    n = 1_000_000

    def scale():
        m = rs.uniform(-104.0, 89.0, size=(n, K))
        m[: n // 2] = rs.uniform(-20.0, 20.0, size=(n // 2, 1)) + rs.randn(n // 2, K) * 3.0
        m[n // 2: n // 2 + 20000] = rs.uniform(-104.0, -87.3, size=(20000, K))
        m[n // 2 + 20000: n // 2 + 21000, 0] = rs.uniform(88.73, 89.0, size=1000)
        occ = rs.randint(0, 13, size=n).astype(np.uint32)
        prob = (m * np.maximum(occ, 1)[:, None]).astype(np.float32)                # the pass's sums
        mean = (prob.astype(np.float64) / np.maximum(occ, 1).astype(np.float64)[:, None]).astype(np.float32)
        return prob, occ, mean

    (p1, o1, m1), (p2, o2, m2) = scale(), scale()
    with np.errstate(over="ignore", under="ignore", invalid="ignore"):
        ref = np.sum(np.stack([loops.reference_softmax(m1, K), loops.reference_softmax(m2, K)]), axis=0)
    ref_l = np.argmax(ref, axis=1)
    assert np.isnan(ref).any() and ((ref > 0) & (ref < np.finfo(np.float32).tiny)).any()
    with drs.Session("dilated_grsl", 4, K, precision="f16") as s:
        acc, none = s.debug_multiscale_softmax_add(p1, o1, want_labels=False)
        acc, lab = s.debug_multiscale_softmax_add(p2, o2, acc=acc)
    assert none is None
    nan = np.isnan(ref)
    assert np.array_equal(np.isnan(acc), nan)
    assert np.array_equal(acc[~nan].view(np.uint32), ref[~nan].view(np.uint32))
    assert np.array_equal(lab, ref_l)


def test_multiscale_row_stripes_equal_the_full_pass(drs):
    """2 and 3 row stripes of one GPU (row_begin / row_end), concatenated, equal the whole-scene pass bit for bit."""
    for kind, H, W, C, K, grid, crops in SCENES:
        s, *_ = session_with_scene(drs, kind, H, W, C, K, "f16")
        with s:
            full_l, full_sum = s.scene_infer_multiscale(0, crops, 16, H, W, variant=grid, want_sum=True)
            for n in (2, 3):
                cuts = [(r * H) // n + (7 if 0 < r < n else 0) for r in range(n + 1)]
                parts = [s.scene_infer_multiscale(0, crops, 16, H, W, variant=grid, row_begin=a, row_end=b, want_sum=True)
                         for a, b in zip(cuts[:-1], cuts[1:])]
                assert np.array_equal(np.concatenate([p[0] for p in parts]), full_l), (kind, n)
                assert same_bits(np.concatenate([p[1] for p in parts]), full_sum), (kind, n)


def test_multiscale_confusion_and_the_next_single_scale_pass(drs):
    """drs_scene_confusion after a multi-scale pass counts that pass's label map (eroded label 6 ignored), also when the map
    stayed on the device; a single-scale pass afterwards is bit-identical to a fresh session's."""
    from drs_b200 import loops
    kind, H, W, C, K, grid, crops = SCENES[0]
    s, img, lab, mean, std = session_with_scene(drs, kind, H, W, C, K, "f16")
    with s:
        assert (lab == 6).any()
        labels = s.scene_infer_multiscale(0, crops, 16, H, W)
        cm, correct = s.scene_confusion(0, K, 6)
        ref = loops.confusion_counts(lab, labels, K, ignore_label=6)
        assert np.array_equal(cm, ref) and correct == int(np.trace(ref))
        assert s.scene_infer_multiscale(0, crops, 16, H, W, keep_on_device=True) is None
        cm2, _ = s.scene_confusion(0, K, 6)
        assert np.array_equal(cm2, ref)
        after_l, after_m = s.scene_infer(0, 25, 16, H, W, want_mean=True)
    fresh, *_ = session_with_scene(drs, kind, H, W, C, K, "f16")
    with fresh:
        ref_l, ref_m = fresh.scene_infer(0, 25, 16, H, W, want_mean=True)
    assert np.array_equal(after_l, ref_l) and np.array_equal(after_m.view(np.uint64), ref_m.view(np.uint64))


def test_multiscale_refuses_bad_calls_and_leaves_nothing_half_done(drs):
    """No scale, a crop larger than the scene and a stripe whose rows are not resident each raise DrsError before any
    launch; the next pass is bit-identical to the one before the refused calls, and the confusion still counts it."""
    from drs_b200 import lib, loops
    kind, H, W, C, K, grid, crops = SCENES[0]
    s, img, lab, mean, std = session_with_scene(drs, kind, H, W, C, K, "f16")
    with s:
        ref_l, ref_sum = s.scene_infer_multiscale(0, crops, 16, H, W, want_sum=True)
        with pytest.raises(lib.DrsError, match="at least one scale"):
            s.scene_infer_multiscale(0, [], 16, H, W)
        with pytest.raises(lib.DrsError, match="does not fit"):
            s.scene_infer_multiscale(0, [25, W + 1], 16, H, W)
        for _ in range(2):                                 # a refused geometry is not memoised as an empty pass
            with pytest.raises(lib.DrsError, match="does not fit"):
                s.scene_infer(0, W + 1, 16, H, W)
        cm, _ = s.scene_confusion(0, K, 6)                 # the refused calls left the last map alone
        assert np.array_equal(cm, loops.confusion_counts(lab, ref_l, K, ignore_label=6))
        # rows [0, 200) + labels resident: the stripe [150, 250) needs patches that reach below row 200
        s.upload_scene(1, img, lab, row_begin=0, row_end=200)
        with pytest.raises(lib.DrsError, match="resident"):
            s.scene_infer_multiscale(1, crops, 16, H, W, row_begin=150, row_end=250)
        part_l = s.scene_infer_multiscale(1, crops, 16, H, W, row_begin=0, row_end=150)
        assert np.array_equal(part_l, ref_l[:150])
        again_l, again_sum = s.scene_infer_multiscale(0, crops, 16, H, W, want_sum=True)
        assert np.array_equal(again_l, ref_l) and same_bits(again_sum, ref_sum)


def _cli_dataset(tmp_path, drs):
    """A Vaihingen-shaped dataset, a saved model and the score arrays of step 3 for the isprs command line."""
    from drs_b200 import synth
    data, out = tmp_path / "vaihingen", tmp_path / "out"
    data.mkdir()
    out.mkdir()
    for i, name in enumerate(("1", "5")):
        img, lab = synth.scene("vaihingen", H=180, W=150, seed=40 + i, block=16)
        np.save(data / (name + "_image.npy"), img)
        np.save(data / (name + "_labels.npy"), lab)
    with drs.Session("dilated_grsl", 4, 6, precision="bf16", seed=9) as s:
        s.save(str(out / "model-3"))
    np.save(out / "patch_acc_loss_step_3.npy", np.array([2.0, 4.5, 3.0], dtype=np.float32))
    np.save(out / "patch_occur_step_3.npy", np.array([4, 5, 5], dtype=np.int32))
    args = [str(data) + "/", str(out) + "/", str(out / "model-3"), "1", "5", "0.01", "0.005", "16", "10", "25", "25",
            "dilated_grsl", "multi_fixed", "25,31,40", "acc", "validate_test"]
    return args


def _free_port():
    import socket
    with socket.socket() as sk:
        sk.bind(("127.0.0.1", 0))
        return sk.getsockname()[1]


# GpuBackend.scene_multiscale_labels through cli.make_backend, in one process or one per rank under torchrun: every rank
# saves the map it returns (the assembled [H, W] map on every rank)
_MAPS_SCRIPT = """
import sys
import numpy as np
sys.path.insert(0, sys.argv[1])
import drs_b200  # noqa: F401
from drs_b200 import cli, synth
img, lab = synth.scene("vaihingen", H=303, W=250, seed=44, block=16)
mean, std = synth.normalisation(img)
be = cli.make_backend("dilated_grsl", 4, 6, 0.005, 0.01, 0.5, [img], [lab], mean, std, True, False, seed=9)
m = be.scene_multiscale_labels(0, [31, 25, 45], 16)
np.save(sys.argv[2] + "_rank%d.npy" % be.rank, m)
"""


def _metric_lines(stdout):
    return [l for l in stdout.splitlines() if l.startswith("---- Iter")]


def test_isprs_cli_multiscale_validate_test(drs, tmp_path):
    """isprs_dilated_random.py ... validate_test with DRS_NUM_SCALES=3: the multi-scale evaluation over the three patch sizes,
    with the metric lines of the host composition (same session, same model)."""
    import io
    import types
    from contextlib import redirect_stdout
    from drs_b200 import backend, loops
    args = _cli_dataset(tmp_path, drs)
    env = dict(os.environ, PYTHONPATH=ROOT, DRS_NUM_SCALES="3")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "isprs_dilated_random.py")] + args, cwd=tmp_path, env=env,
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    lines = _metric_lines(r.stdout)
    assert len(lines) == 2 and "Test ALL MAPS" in lines[1]
    # the host composition of the same evaluation (mean / std from the cache files the run wrote)
    img = np.load(tmp_path / "vaihingen" / "5_image.npy")
    lab = np.load(tmp_path / "vaihingen" / "5_labels.npy")
    tag = str(tmp_path) + "/dataset_vaihingen_crop_25_stride_25"
    mean, std = np.load(tag + "_mean.npy"), np.load(tag + "_std.npy")
    with drs.Session("dilated_grsl", 4, 6, precision="f16") as s:
        be = backend.GpuBackend(s, [img], [lab], mean, std)
        be.restore(args[2])

        host_only = types.SimpleNamespace(scene_mean_logits=be.scene_mean_logits)   # the NumPy composition
        buf = io.StringIO()
        with redirect_stdout(buf):
            loops.isprs_validate_test_multiscale(host_only, [img], [lab], ["5"], 16, 3, "multi_fixed", np.array([25, 31, 40]),
                                                 "acc", 3, False, args[1])
    assert _metric_lines(buf.getvalue()) == lines


def test_isprs_cli_multiscale_two_ranks_when_two_gpus(drs, tmp_path):
    """Under torchrun on 2 ranks (row stripes, labels gathered over NCCL) the backend returns the 1-rank label map on every
    rank, and the command line prints the metric lines of the 1-rank run."""
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    env = dict(os.environ, PYTHONPATH=ROOT, DRS_NUM_SCALES="3")
    run = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1"]
    script = tmp_path / "maps.py"
    script.write_text(_MAPS_SCRIPT)
    one = subprocess.run([sys.executable, str(script), ROOT, str(tmp_path / "one")], cwd=tmp_path, env=env, capture_output=True,
                         text=True, timeout=600)
    assert one.returncode == 0, one.stdout[-3000:] + one.stderr[-3000:]
    two = subprocess.run(run + ["--master-port", str(_free_port()), str(script), ROOT, str(tmp_path / "two")], cwd=tmp_path,
                         env=env, capture_output=True, text=True, timeout=900)
    assert two.returncode == 0, two.stdout[-3000:] + two.stderr[-3000:]
    ref = np.load(tmp_path / "one_rank0.npy")
    assert ref.shape == (303, 250)
    for r in (0, 1):
        assert np.array_equal(np.load(tmp_path / ("two_rank%d.npy" % r)), ref), r

    args = _cli_dataset(tmp_path, drs)
    cli_script = os.path.join(ROOT, "isprs_dilated_random.py")
    one = subprocess.run([sys.executable, cli_script] + args, cwd=tmp_path, env=env, capture_output=True, text=True, timeout=600)
    assert one.returncode == 0, one.stdout[-3000:] + one.stderr[-3000:]
    two = subprocess.run(run + ["--master-port", str(_free_port()), cli_script] + args, cwd=tmp_path, env=env,
                         capture_output=True, text=True, timeout=900)
    assert two.returncode == 0, two.stdout[-3000:] + two.stderr[-3000:]
    lines = _metric_lines(one.stdout)
    assert len(lines) == 2
    # every rank prints the metrics of the assembled map
    assert sorted(_metric_lines(two.stdout)) == sorted(lines * 2)
