"""Closing a session returns every device allocation it made: workspace, scene buffers, captured graphs and the per-layer
copies that DRS_DEBUG_KEEP=1 keeps from the last step."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu


def one_session(drs, monkeypatch, rs):
    from drs_b200 import synth
    C, K, B, crop = 4, 6, 16, 25
    s = drs.Session("dilated_grsl", C, K, precision="bf16", seed=1)
    s.reserve(B, crop)
    x = rs.randn(B, crop * crop * C).astype(np.float32)
    y = rs.randint(0, K, size=(B, crop * crop)).astype(np.float32)
    s.train_step(x, y, crop)
    monkeypatch.setenv("DRS_DEBUG_KEEP", "1")         # the kept copies of this step are still alive when the session closes
    s.train_step(x, y, crop)
    monkeypatch.delenv("DRS_DEBUG_KEEP")
    img, lab = synth.scene("vaihingen", H=150, W=170, block=16, unlabelled=True)
    mean, std = synth.normalisation(img)
    s.set_normalization(mean, std)
    s.upload_scene(0, img, lab)
    s.scene_infer(0, crop, 16, 150, 170)
    s.scene_confusion(0, K, 6)
    w = (rs.randn(3, 3, 64, 64) / 24.0).astype(np.float32)
    s.debug_conv(rs.randn(2, 9, 9, 64).astype(np.float32), w, np.ones(64, np.float32), np.zeros(64, np.float32), 1, 1, "bf16")
    s.close()


def test_session_close_frees_device_memory(drs, monkeypatch):
    import torch
    rs = np.random.RandomState(0)
    free = []
    for _ in range(8):
        one_session(drs, monkeypatch, rs)
        torch.cuda.synchronize()
        free.append(torch.cuda.mem_get_info()[0])
    lost = free[0] - free[-1]
    assert lost <= 128 << 20, "free device memory fell by %.1f MiB over 7 sessions: %s" % (
        lost / 2.0**20, [f >> 20 for f in free])
