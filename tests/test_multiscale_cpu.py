"""CPU: the arithmetic of the device's multi-scale evaluation, compiled for the host, against NumPy; and the multi-scale loop
driving a backend that composes the scales itself.

The kernel (multiscale_softmax_add_kernel, csrc/scene.cuh) and drs_debug_np_softmax share one source (csrc/np_softmax.h),
so a bit-exact match here pins the formula the device evaluates; the GPU tests (test_gpu_multiscale.py) then hold the
device to the same NumPy composition.
"""
import io
import os
from contextlib import redirect_stdout

import numpy as np
import pytest

from oracle import host_np
from oracle.fake_net import fake_logits


def _bits_equal(a, b):
    return np.array_equal(np.asarray(a, np.float32).view(np.uint32), np.asarray(b, np.float32).view(np.uint32))


@pytest.mark.parametrize("K", [2, 6, 7, 8])
def test_softmax_equals_reference_softmax_bit_for_bit(drs, K):
    """drs_debug_np_softmax == loops.reference_softmax (np.exp, np.sum over the last axis, np.repeat, np.divide in float32)
    up to the 8 classes a session takes (np.sum adds K < 8 values in order but K = 8 as a tree), on 2 M random means over
    [-100, 80] -- exp results down in the denormal range included -- and on runs of equal values."""
    from drs_b200 import loops
    from drs_b200.session import np_softmax
    rs = np.random.RandomState(K)
    n = 2_000_000
    m = rs.uniform(-100.0, 80.0, size=(n, K)).astype(np.float32)
    # means of one pixel close together (the usual case: softmax of logits a few units apart), some far apart
    m[: n // 2] = (rs.uniform(-20.0, 20.0, size=(n // 2, 1)) + rs.randn(n // 2, K) * 3.0).astype(np.float32)
    m[n // 2: n // 2 + 1000] = rs.uniform(-104.0, -87.0, size=(1000, K)).astype(np.float32)   # exp denormal
    ref = loops.reference_softmax(m, K)
    got = np_softmax(m)
    assert _bits_equal(got, ref)
    assert (np.exp(m[n // 2: n // 2 + 1000]) < np.finfo(np.float32).tiny).any()
    # runs of equal values: ties of the argmax downstream, and exactly representable quotients
    ties = np.repeat(rs.uniform(-50.0, 50.0, size=(5000, 1)).astype(np.float32), K, axis=1)
    ties[::2, -1] = ties[::2, 0] - 1.0
    ties[::3, 0] = 0.0
    assert _bits_equal(np_softmax(ties), loops.reference_softmax(ties, K))


def test_exp_restatement_equals_numpy_exp():
    """The restatement of NumPy's float32 exp (csrc/np_softmax.h: np_expf) == np.exp, bit for bit, on every float32 with
    0.5 <= |x| < 4 (50 M values: the band the softmax of nearby logits lives in), on 24 M random bit patterns of
    [-104, 89] (every exponent, so tiny arguments too), on 12 M values drawn uniformly from [-104, 89] (denormal results of
    [-104, -87.3] included) and on the overflow / underflow borders and the specials.

    The exhaustive sweep was run once, outside the suite: the restatement matched np.exp (numpy 2.3.5, AVX-512F path) on
    every one of the 4,278,190,080 finite float32 inputs.  It takes far longer than a unit test should, so the suite keeps
    this sample."""
    from drs_b200.session import np_expf

    def bits(lo, hi):                                      # every float32 in [lo, hi), 0 < lo < hi
        return np.arange(np.float32(lo).view(np.uint32), np.float32(hi).view(np.uint32), dtype=np.uint32).view(np.float32)

    band = bits(0.5, 4.0)
    rs = np.random.RandomState(7)
    top_neg = int(np.float32(104.0).view(np.uint32))
    top_pos = int(np.float32(89.0).view(np.uint32))
    rnd_bits = np.concatenate([rs.randint(0, top_neg + 1, size=12_000_000, dtype=np.uint64),
                               rs.randint(0, top_pos + 1, size=12_000_000, dtype=np.uint64)]).astype(np.uint32)
    rnd_bits[:12_000_000] |= np.uint32(0x80000000)
    uniform = rs.uniform(-104.0, 89.0, size=12_000_000).astype(np.float32)
    edges = np.array([88.72283935546875, np.nextafter(np.float32(88.72283935546875), np.float32(0)), 88.7228, -87.33654,
                      -103.97208404541015625, np.nextafter(np.float32(-103.97208404541015625), np.float32(0)), -103.9721,
                      0.0, -0.0, 1e-30, -1e-30, np.inf, -np.inf, np.nan, 3.4e38, -3.4e38], dtype=np.float32)
    with np.errstate(over="ignore", under="ignore"):
        for x in (band, -band, rnd_bits.view(np.float32), uniform, edges):
            got, ref = np_expf(x), np.exp(x)
            nan = np.isnan(ref)
            assert np.array_equal(np.isnan(got), nan)
            bad = got[~nan].view(np.uint32) != ref[~nan].view(np.uint32)
            assert not bad.any(), x[~nan][bad][:8]
        e = np.exp(uniform)
    assert ((e > 0) & (e < np.finfo(np.float32).tiny)).any()         # denormal results were compared


def test_softmax_rejects_bad_arguments(drs):
    from drs_b200 import lib
    from drs_b200.session import np_softmax
    with pytest.raises(lib.DrsError, match="at most 8 classes"):
        np_softmax(np.zeros((4, 9), np.float32))


def test_multiscale_loop_with_a_backend_that_composes_the_scales(tmp_path):
    """loops.isprs_validate_test_multiscale with a stand-in backend that has scene_multiscale_labels (what GpuBackend
    offers): it receives the crops of the reference's own run (multiscale_golden.npz, both update types) in order and
    returns the label map of their composition, which equals the reference's; the printed lines are those of the host
    composition."""
    from drs_b200 import loops
    g = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "multiscale_golden.npz"))
    img, lab, mean, std, values = g["ms_scene"], g["ms_gt"], g["ms_mean"], g["ms_std"], g["ms_values"]

    def mean_map(crop, batch):
        h, w = img.shape[:2]
        pos = host_np.all_patch_positions(h, w, crop, batch)
        inst = np.array([[0, r, c] for r, c in pos], dtype=np.int32)
        x, _ = host_np.apply_plan([img], [lab], inst, None, crop, mean, std, cast=False)
        logits = fake_logits(x.reshape(len(inst), -1), crop, 4, 6)
        _, m = host_np.accumulate_argmax(logits, pos, h, w, crop, return_mean=True)
        return m

    class HostBackend:
        """Only the per-scale maps: the loop composes them in NumPy."""

        def scene_mean_logits(self, scene_id, crop, batch, variant="isprs"):
            return mean_map(crop, batch)

    class ComposingBackend:
        def __init__(self):
            self.calls = []

        def scene_multiscale_labels(self, scene_id, crops, batch, variant="isprs"):
            self.calls.append((scene_id, list(crops), batch, variant))
            psum = sum(loops.reference_softmax(mean_map(c, batch).astype(np.float32), 6) for c in crops)
            return np.argmax(psum, axis=2).astype(np.uint8)

    for ci in (0, 1):
        out = str(tmp_path) + "/"
        np.save(out + "patch_acc_loss_step_5.npy", g["ms_%d_pal" % ci])
        np.save(out + "patch_occur_step_5.npy", g["ms_%d_occ" % ci])
        be = ComposingBackend()
        log = io.StringIO()
        with redirect_stdout(log):
            maps = loops.isprs_validate_test_multiscale(be, [img], [lab], ["1"], 7, 5, "multi_fixed", values.copy(),
                                                        str(g["ms_updates"][ci]), 3, False, out)
        ref_crops = g["ms_%d_crops" % ci]
        order = [int(c) for i, c in enumerate(ref_crops) if i == 0 or c != ref_crops[i - 1]]
        assert be.calls == [(0, order, 7, "isprs")]
        assert np.array_equal(maps[0], g["ms_%d_labels" % ci])
        host_log = io.StringIO()
        with redirect_stdout(host_log):
            host_maps = loops.isprs_validate_test_multiscale(HostBackend(), [img], [lab], ["1"], 7, 5, "multi_fixed",
                                                             values.copy(), str(g["ms_updates"][ci]), 3, False, out)
        assert np.array_equal(host_maps[0], maps[0])
        assert log.getvalue() == host_log.getvalue()
