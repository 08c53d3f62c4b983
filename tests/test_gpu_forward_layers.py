"""Teacher-forced per-layer checks of the forward path against a float64 reference.

Each layer's reference is computed from the GPU's own input to that layer: the exact 16-bit values the kernel read, fetched
with debug_activation.  Errors cannot pile up across layers, so at every depth the bound of a stored output is one rounding
plus the fp32 accumulation:

    |y_gpu - y_ref| <= u |y_ref| + (1 + u) gamma(n) * sum |x| |w| |scale| + tiny

  * u = 2^-11 (f16), 2^-8 (bf16), 2^-24 (fp32 storage);
  * products of 16-bit operands are exact in fp32; gamma(n) = (n + 4) 2^-23 bounds an n-term fp32 sum in any order, with
    adds that truncate (2^-23 each, the tensor cores' accumulation) rather than round, plus the folded BN affine of the
    epilogue;
  * tiny = 2^-24 in f16 (its subnormal spacing), negligible otherwise.
Max-pool and the activations are 1-Lipschitz, so a pooled output's bound is the largest bound in its window; an average
pool's is the mean of its window's bounds plus its own fp32 sum and rounding.  Conv weights are rounded to the session
precision, as the packers round them.  Nothing here is fitted to observed errors.

At scene-chunk sizes only sampled pixels are evaluated, each from its receptive field in the previous tap (for a pooled
layer the 3x3 conv outputs around it): image corners and borders of the first and last image, both sides of every 128-pixel
tile boundary that splits an image, the last pixel, and random ones.
"""
import os
import time

import numpy as np
import pytest

from test_gpu_parity import NETS, TRAIN_NETS, act_np, rounded, torch_conv

pytestmark = pytest.mark.gpu

EPS = 0.001                                    # batch_norm epsilon (isprs:658)
U = {"f16": 2.0 ** -11, "bf16": 2.0 ** -8, "fp32": 2.0 ** -24}
TINY = {"f16": 2.0 ** -24, "bf16": 1e-30, "fp32": 1e-30}
E24 = 2.0 ** -24
REPORT = {}                                    # (case, precision, layer) -> largest err / bound


def gamma(n):
    return (n + 4) * 2.0 ** -23


# ------------------------------------------------------------------------------------------------ network description
def net_layers(net, C):
    """[{scope, k, rate, ci, co, post, inputs}] in execution order, and the classifier's input scopes.  ``inputs`` name the
    taps whose channel concatenation is the layer's input ("x": the network input); ``post`` is None, ("max",),
    ("avg", k) or ("se", r, name)."""
    from oracle import nets_torch as nt
    spec = nt.NET_SPECS[net]
    plan, _ = nt.layer_plan(net, C)
    n_plain = len(spec["convs"])
    posts = spec.get("post")
    layers = []
    for i, (scope, k, r, ci, co) in enumerate(plan[:n_plain]):
        post = ("max",) if spec["pool"] else (posts[i] if posts else None)
        inputs = ["x"] if i == 0 else ([p[0] for p in plan[:i]] if spec["dense"] else [plan[i - 1][0]])
        layers.append(dict(scope=scope, k=k, rate=r, ci=ci, co=co, post=post, inputs=inputs))
    prev = [p[0] for p in plan[:n_plain]] if spec["dense"] else [plan[n_plain - 1][0]]
    by_scope = {p[0]: p for p in plan}
    for (name, _, _, _, _, _) in spec.get("squeeze", ()):
        for part, inputs in (("_s1", prev), ("_s2_1", [name + "_s1"]), ("_s2_2", [name + "_s1"])):
            _, k, r, ci, co = by_scope[name + part]
            layers.append(dict(scope=name + part, k=k, rate=r, ci=ci, co=co, post=None, inputs=list(inputs)))
        prev = [name + "_s2_1", name + "_s2_2"]
    act = 1 if spec["act"] == "relu" else 2
    return layers, prev, act


def nseg_of(B, crop, ci, sm_count):
    """Row segments per image of maxpool3_classifier_kernel (launch_maxpool3_classifier, ops.cuh)."""
    base = B * ((crop + 1) // 2) * (ci // 8)
    n0 = min(max(1, -(-sm_count * 2048 // base)), max(1, crop // 4))
    seg = -(-crop // n0)
    return -(-crop // seg)


def nseg_class(B, crop, ci, sm_count):
    """(nseg, which limit chose it): the crop/4 cap, the SM-fill term at its floor of 1, or the SM-fill term above 1."""
    base = B * ((crop + 1) // 2) * (ci // 8)
    fill = max(1, -(-sm_count * 2048 // base))
    return nseg_of(B, crop, ci, sm_count), ("crop/4" if fill >= crop // 4 > 1 else ("1" if fill == 1 else "intermediate"))


# ------------------------------------------------------------------------------------------------ float64 reference
def pixel_coords(idx, B, crop):
    b, rem = np.divmod(idx, crop * crop)
    i, j = np.divmod(rem, crop)
    return b, i, j


def conv_at(Xs, w, rate, idx, crop, pad_before=None, chunk=2048):
    """SAME dilated convolution at flat pixel indices ``idx`` of the channel concatenation of ``Xs`` ([B,crop,crop,*] each):
    (sum x w, sum |x| |w|), [len(idx), Co] float64.  ``pad_before``: override of TF SAME's floor(total / 2)."""
    k = w.shape[0]
    pb = (k - 1) * rate // 2 if pad_before is None else pad_before
    b, i, j = pixel_coords(idx, Xs[0].shape[0], crop)
    offs = np.arange(k) * rate - pb
    wm = w.reshape(-1, w.shape[-1]).astype(np.float64)
    wa = np.abs(wm)
    out = np.empty((len(idx), wm.shape[1]))
    sab = np.empty_like(out)
    for c0 in range(0, len(idx), chunk):
        sl = slice(c0, c0 + chunk)
        r, c = i[sl, None] + offs, j[sl, None] + offs
        valid = (((r >= 0) & (r < crop))[:, :, None] & ((c >= 0) & (c < crop))[:, None, :])[..., None]
        rc, cc = np.clip(r, 0, crop - 1), np.clip(c, 0, crop - 1)
        bb = b[sl, None, None]
        p = np.concatenate([X[bb, rc[:, :, None], cc[:, None, :]] for X in Xs], -1).astype(np.float64) * valid
        p = p.reshape(p.shape[0], -1)
        out[sl] = p @ wm
        sab[sl] = np.abs(p) @ wa
    return out, sab


def window(idx, B, crop, r, shift=0):
    """Flat indices of the (2r+1)^2 SAME window around each pixel (-1: outside the image), [len(idx), (2r+1)^2]."""
    b, i, j = pixel_coords(idx, B, crop)
    d = np.arange(-r, r + 1)
    ii = i[:, None, None] + d[None, :, None]
    jj = j[:, None, None] + d[None, None, :] + shift
    ok = (ii >= 0) & (ii < crop) & (jj >= 0) & (jj < crop)
    q = b[:, None, None] * crop * crop + ii * crop + jj
    return np.where(ok, q, -1).reshape(len(idx), -1)


def post_needs(L, idx, B, crop, mut):
    """The pixels whose pre-post values the layer's outputs at idx depend on, and the windows (None: no window)."""
    post = L["post"]
    if post is None:
        return idx, None
    if post[0] == "se":
        return np.arange(B * crop * crop), None
    r = 1 if post[0] == "max" else post[1] // 2
    win = window(idx, B, crop, r, mut.get("pool_shift", 0) if post[0] == "max" else 0)
    return np.unique(win[win >= 0]), win


def apply_post(L, a, ba, need, win, idx, B, crop, p, prec):
    """Pool / average pool / SE gate of the activations ``a`` (with bounds ``ba``) at pixels ``need`` -> outputs at idx."""
    post = L["post"]
    u, tiny = U[prec], TINY[prec]
    if post is None:
        return a, ba
    if post[0] == "se":
        px = crop * crop
        A, BA = a.reshape(B, px, -1), ba.reshape(B, px, -1)
        w1, b1 = [np.asarray(p[post[2] + "_fc1/" + n], np.float64) for n in ("weights", "biases")]
        w2, b2 = [np.asarray(p[post[2] + "_fc2/" + n], np.float64) for n in ("weights", "biases")]
        m = A.mean(1)
        dm = BA.mean(1) + gamma(px) * np.abs(A).mean(1)
        h = np.maximum(m @ w1 + b1, 0)
        dh = dm @ np.abs(w1) + gamma(w1.shape[0]) * (np.abs(m) @ np.abs(w1) + np.abs(b1))
        g = 1.0 / (1.0 + np.exp(-(h @ w2 + b2)))
        dg = 0.25 * (dh @ np.abs(w2) + gamma(w2.shape[0]) * (np.abs(h) @ np.abs(w2) + np.abs(b2))) + 4 * E24
        out = A * g[:, None, :]
        bound = np.abs(g)[:, None, :] * BA + (np.abs(A) + BA) * dg[:, None, :] + (u + 2 * E24) * np.abs(out) + tiny
        return out.reshape(-1, out.shape[-1])[idx], bound.reshape(-1, out.shape[-1])[idx]
    ok = win >= 0
    pos = np.searchsorted(need, np.where(ok, win, need[0]))
    Aw, Bw = a[pos], ba[pos]
    okc = ok[..., None]
    if post[0] == "max":
        return np.where(okc, Aw, -np.inf).max(1), np.where(okc, Bw, 0.0).max(1)
    cnt = ok.sum(1)[:, None]
    ref = np.where(okc, Aw, 0.0).sum(1) / cnt
    mb = np.where(okc, Bw, 0.0).sum(1) / cnt
    ma = np.where(okc, np.abs(Aw), 0.0).sum(1) / cnt
    return ref, mb + gamma(ok.shape[1]) * ma + u * (np.abs(ref) + mb) + tiny


def eval_layer(L, taps, p, prec, act, idx, B, crop, mut=None):
    """Reference inference output of layer L at pixels idx from the GPU's input taps, and its bound."""
    mut = mut or {}
    s = L["scope"]
    w = rounded(np.asarray(p[s + "/weights"], np.float32), prec).astype(np.float64)
    if mut.get("drop_last_input_channel") and L["inputs"] == ["x"]:
        w[:, :, -1, :] = 0.0
    pb = None
    if mut.get("swap_pads") == s:
        total = (L["k"] - 1) * L["rate"]
        pb = total - total // 2
    need, win = post_needs(L, idx, B, crop, mut)
    z, sab = conv_at([taps[n] for n in L["inputs"]], w, L["rate"], need, crop, pb)
    b, mm, mv = [np.asarray(p[s + n], np.float64) for n in ("/biases", "/moving_mean", "/moving_variance")]
    scale = 1.0 / np.sqrt(mv + EPS)
    a = act_np((z + b - mm) * scale, act)
    ba = U[prec] * np.abs(a) + (1 + U[prec]) * gamma(w.shape[0] * w.shape[1] * w.shape[2]) * (sab + np.abs(b) + np.abs(mm)) * scale + TINY[prec]
    return apply_post(L, a, ba, need, win, idx, B, crop, p, prec)


def classify(xc, bx, p, K, k_off=0):
    """1x1 classifier on [n, cls_in] inputs with input bounds bx (None: exact GPU values), fp32 weights as stored."""
    wc = np.asarray(p["conv_classifier/weights"], np.float64).reshape(-1, K)
    bc = np.asarray(p["conv_classifier/biases"], np.float64)
    if k_off:                                  # the weight matrix read with one class too few: the last class keeps its bias
        kk = K - k_off
        wc = np.concatenate([wc.reshape(-1)[:wc.shape[0] * kk].reshape(-1, kk), np.zeros((wc.shape[0], k_off))], 1)
    lg = xc @ wc + bc
    bound = gamma(xc.shape[1]) * (np.abs(xc) @ np.abs(wc) + np.abs(bc)) + 2 * E24 * np.abs(lg) + 1e-30
    if bx is not None:
        bound = bound + bx @ np.abs(wc)
    return lg, bound


def ratio(key, got, ref, bound):
    r = float((np.abs(got.astype(np.float64) - ref) / bound).max())
    REPORT[key] = max(REPORT.get(key, 0.0), r)
    return r


def sample_pixels(B, crop, rs, n_random=1024):
    """Image corners and borders of the first and last image, both sides of every 128-pixel tile boundary that splits an
    image, the last pixel, and n_random more."""
    P, M = crop * crop, B * crop * crop
    e = np.arange(crop)
    border = np.unique(np.concatenate([e, (crop - 1) * crop + e, e * crop, e * crop + crop - 1]))
    t = np.arange(128, M, 128)
    t = t[t % P != 0]
    idx = np.concatenate([border, (B - 1) * P + border, t - 1, t, [M - 1], rs.randint(0, M, n_random)])
    return np.unique(idx)


def params_with_stats(net, C, K, seed):
    """Initial variables with non-trivial moving statistics, as in test_network_inference_vs_oracle."""
    from oracle import nets_torch
    p = nets_torch.init_params(net, C, K, seed=seed)
    rs = np.random.RandomState(seed + 1)
    for k in p:
        if k.endswith("moving_mean"):
            p[k] = (rs.randn(*p[k].shape) * 0.2).astype(np.float32)
        if k.endswith("moving_variance"):
            p[k] = (0.5 + rs.rand(*p[k].shape)).astype(np.float32)
    return p


# ------------------------------------------------------------------------------------------------ inference
class InferRun:
    """One s.infer and every activation tap it recorded.  DRS_DEBUG_KEEP=1 makes the forward keep a copy of each layer's
    output: its feature buffers rotate, so without copies only the last layers' taps survive the pass."""

    def __init__(self, drs, net, C, K, prec, p, x, B, crop):
        self.layers, self.cls_inputs, self.act = net_layers(net, C)
        s = drs.Session(net, C, K, precision=prec)
        s.load_variables(p)
        keep = os.environ.get("DRS_DEBUG_KEEP")
        os.environ["DRS_DEBUG_KEEP"] = "1"
        try:
            self.pred, self.logits = s.infer(x, crop)
        finally:
            if keep is None:
                del os.environ["DRS_DEBUG_KEEP"]
            else:
                os.environ["DRS_DEBUG_KEEP"] = keep
        self.taps = {"x": rounded(x.reshape(B, crop, crop, C), prec)}
        for L in self.layers:
            try:
                self.taps[L["scope"]] = s.debug_activation(L["scope"], B, crop, L["co"])
            except drs.lib.DrsError:           # the pooled last layer of a fused pool + classifier has no tap
                assert L is self.layers[-1] and L["post"] == ("max",) and prec != "fp32", L["scope"]
        s.close()
        self.net, self.C, self.K, self.prec, self.p, self.B, self.crop = net, C, K, prec, p, B, crop

    def check(self, tag, idx=None, mut=None):
        """Largest err / bound per layer and for the logits ({name: ratio}); pred checked on the way."""
        B, crop, K, prec = self.B, self.crop, self.K, self.prec
        idx = np.arange(B * crop * crop) if idx is None else idx
        out = {}
        for L in self.layers:
            if L["scope"] not in self.taps:
                continue
            ref, bound = eval_layer(L, self.taps, self.p, prec, self.act, idx, B, crop, mut)
            got = self.taps[L["scope"]].reshape(-1, L["co"])[idx]
            out[L["scope"]] = ratio((tag, prec, L["scope"]), got, ref, bound)
        last = self.layers[-1]
        if last["scope"] in self.taps:
            xc = np.concatenate([self.taps[n].reshape(-1, self.taps[n].shape[-1])[idx] for n in self.cls_inputs], 1).astype(np.float64)
            lg, lb = classify(xc, None, self.p, K, (mut or {}).get("k_off", 0))
        else:
            # last layer fused with the pool + classifier: conv L from tap L-1, pool, classify (bounds carried through)
            pooled, pb = eval_layer(last, self.taps, self.p, prec, self.act, idx, B, crop, mut)
            lg, lb = classify(pooled, pb, self.p, K, (mut or {}).get("k_off", 0))
        got = self.logits.reshape(-1, K)[idx]
        out["logits"] = ratio((tag, prec, "logits"), got, lg, lb)
        if mut is None:
            assert np.array_equal(self.pred.reshape(-1), np.argmax(self.logits.reshape(-1, K), -1)), (tag, prec)
            top2 = np.sort(lg, -1)
            decided = top2[:, -1] - top2[:, -2] > 2 * lb.max(-1)
            assert np.array_equal(self.pred.reshape(-1)[idx][decided], np.argmax(lg, -1)[decided]), (tag, prec)
        return out


def _assert_within(res, what):
    bad = {k: v for k, v in res.items() if not v <= 1.0}
    assert not bad, (what, bad)


INFER_NETS = NETS + (("dilated_grsl", 4, 2), ("dilated_grsl", 4, 3), ("dilated_grsl_rate8", 5, 8))
FP32_NETS = {"dilated_grsl", "dilated_icpr_rate6_densely", "dilated_icpr_old", "dilated_icpr_rate6_avgpool",
             "dilated_icpr_rate6_SE", "dilated_icpr_rate6_squeeze"}


@pytest.mark.parametrize("net,C,K", INFER_NETS)
def test_inference_layers_full(drs, net, C, K):
    """Every layer and the logits of s.infer, whole tensors, at small shapes: (3, 25), (5, 7), (2, 12) and crops 3 and 5, where
    the 5x5 window is wider than the image.  Squeeze nets check each expand convolution's own output slice."""
    rs = np.random.RandomState(4)
    p = params_with_stats(net, C, K, 3)
    t0 = time.time()
    for prec in ("f16", "bf16") + (("fp32",) if net in FP32_NETS else ()):
        for B, crop in ((3, 25), (5, 7), (2, 12), (4, 3), (3, 5)):
            x = rs.randn(B, crop * crop * C).astype(np.float32)
            run = InferRun(drs, net, C, K, prec, p, x, B, crop)
            _assert_within(run.check("%s K%d" % (net, K)), (net, K, prec, B, crop))
    _print_report(net, time.time() - t0)


SCENE_NETS = (("dilated_grsl", 4, 6), ("dilated_grsl_rate8", 5, 6), ("dilated_icpr_original", 4, 6),
              ("dilated_icpr_rate6_densely", 5, 6))


@pytest.mark.parametrize("net,C,K", SCENE_NETS)
def test_inference_layers_scene_chunk(drs, net, C, K):
    """Scene-chunk sizes, sampled pixels: M = 300 000 (B = 480 at crop 25) and the odd crop 49 (B = 128, M = 307 328).  The
    persistent convolution kernels cycle their stage and TMEM rings many times per CTA and the tile count is not a multiple
    of the grid; conv1 runs 2 344 tiles."""
    rs = np.random.RandomState(7)
    p = params_with_stats(net, C, K, 5)
    t0 = time.time()
    for prec in ("f16", "bf16"):
        for B, crop in ((480, 25), (128, 49)):
            x = rs.randn(B, crop * crop * C).astype(np.float32)
            run = InferRun(drs, net, C, K, prec, p, x, B, crop)
            idx = sample_pixels(B, crop, rs)
            _assert_within(run.check("%s scene" % net, idx), (net, prec, B, crop, len(idx)))
    _print_report(net, time.time() - t0)


def test_pool_classifier_row_segments_and_class_counts(drs):
    """maxpool3_classifier_kernel at every row-segment regime -- nseg = crop/4 (few patches), an intermediate value and 1
    (crop 13, B = 1 400) -- and with K = 2, 3 and 8 classes (its KC = 2, KC = 6 with masked classes, KC = 8)."""
    sm = _sm_count()
    seen_nseg, seen_k = {}, set()
    rs = np.random.RandomState(9)
    t0 = time.time()
    for net, C, K, prec, B, crop in (("dilated_grsl", 4, 2, "bf16", 3, 25), ("dilated_grsl_rate8", 5, 3, "f16", 200, 25),
                                     ("dilated_grsl", 4, 8, "bf16", 1400, 13), ("dilated_grsl_rate8", 5, 8, "f16", 2, 16)):
        layers, _, _ = net_layers(net, C)
        n, cls = nseg_class(B, crop, layers[-1]["co"], sm)
        seen_nseg.setdefault(cls, []).append((net, B, crop, n))
        seen_k.add(K)
        p = params_with_stats(net, C, K, 11)
        x = rs.randn(B, crop * crop * C).astype(np.float32)
        run = InferRun(drs, net, C, K, prec, p, x, B, crop)
        assert layers[-1]["scope"] not in run.taps          # the fused kernel ran
        idx = None if B * crop * crop < 4096 else sample_pixels(B, crop, rs)
        _assert_within(run.check("%s K%d nseg%d" % (net, K, n), idx), (net, K, prec, B, crop, n))
    print("pool + classifier row segments covered:", seen_nseg, "class counts:", sorted(seen_k))
    assert set(seen_nseg) == {"crop/4", "intermediate", "1"}, seen_nseg
    assert {2, 3, 8} <= seen_k
    _print_report("pool_classifier", time.time() - t0)


def test_wrong_references_break_the_bounds(drs):
    """The bounds tell a right answer from a wrong one: on the same f16 GPU outputs, a reference with the pads of the k=4 rate-3
    layer swapped (4/5 <-> 5/4), conv1's last input channel dropped, the pool window shifted by one column, or the
    classifier's weights read with one class too few exceeds its bound by at least 10x."""
    net, C, K, B, crop = "dilated_grsl", 4, 6, 3, 25
    rs = np.random.RandomState(13)
    p = params_with_stats(net, C, K, 3)
    x = rs.randn(B, crop * crop * C).astype(np.float32)
    run = InferRun(drs, net, C, K, "f16", p, x, B, crop)
    _assert_within(run.check("sensitivity"), "right reference")
    got = {}
    for name, mut, where in ((("swap_pads", {"swap_pads": "conv3"}, "conv3")), ("drop_last_input_channel", {"drop_last_input_channel": 1}, "conv1"),
                             ("pool_shift", {"pool_shift": 1}, "conv1"), ("k_off", {"k_off": 1}, "logits")):
        got[name] = run.check("wrong:" + name, mut=mut)[where]
    print("wrong references, largest err / bound:", got)
    assert all(v >= 10.0 for v in got.values()), got


def _sm_count():
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count


def _print_report(what, seconds):
    rows = sorted((k, v) for k, v in REPORT.items())
    print("\n%s: largest err / bound per (case, precision, layer), %.1f s" % (what, seconds))
    for (case, prec, layer), v in rows:
        print("  %-44s %-5s %-14s %.3f" % (case, prec, layer, v))
    REPORT.clear()


# ------------------------------------------------------------------------------------------------ conv1 unit cases
@pytest.mark.parametrize("prec", ["f16", "bf16"])
def test_conv1_tensor_core_kernel(drs, prec):
    """conv1_tc_kernel through debug_conv: C in {1, 3, 4, 5, 8}, Co in {32, 64}, crops 3 .. 25, M < 128, tiles spanning
    images, a partial last tile and more tiles than SMs; all three activations.  Bound of test_single_convolution, and the
    derived one."""
    s = drs.Session("dilated_grsl", 4, 6, precision=prec)
    rs = np.random.RandomState(17)
    n = 0
    for C in (1, 3, 4, 5, 8):
        for co in (32, 64):
            for B, crop in ((1, 7), (3, 11), (2, 3), (4, 5), (1, 25), (40, 25)):
                x = rs.randn(B, crop, crop, C).astype(np.float32)
                w = (rs.randn(5, 5, C, co) / np.sqrt(25 * C)).astype(np.float32)
                scale = (0.5 + rs.rand(co)).astype(np.float32)
                shift = (rs.randn(co) * 0.1).astype(np.float32)
                act = n % 3
                n += 1
                xr, wr = rounded(x, prec), rounded(w, prec)
                z = torch_conv(xr, wr, 1)
                sab = torch_conv(np.abs(xr), np.abs(wr), 1)
                ref = act_np(z * scale + shift, act)
                y = s.debug_conv(x, w, scale, shift, 1, act, prec)
                assert np.abs(y - ref).max() < {"f16": 4e-3, "bf16": 3e-2}[prec], (C, co, B, crop, act)
                bound = U[prec] * np.abs(ref) + (1 + U[prec]) * gamma(25 * C) * (sab * scale + np.abs(shift)) + TINY[prec]
                assert ratio(("conv1 C%d Co%d" % (C, co), prec, "B%d crop%d" % (B, crop)), y, ref, bound) <= 1.0, (C, co, B, crop, act)
    s.close()
    _print_report("conv1_tc", 0.0)


# ------------------------------------------------------------------------------------------------ training forward
def check_train_forward(drs, monkeypatch, net, C, K, prec, B, crop, use_mask, sampled, tag):
    """One train_step with bn_decay = 0 under DRS_DEBUG_KEEP=1: per layer Z against conv(previous GPU output) + bias, the
    moving statistics (= the batch statistics) against float64 statistics of the GPU's own Z, and the layer output
    against normalise + activation + post-op of the GPU's Z."""
    from oracle import nets_torch
    monkeypatch.setenv("DRS_DEBUG_KEEP", "1")
    layers, _, act = net_layers(net, C)
    p = nets_torch.init_params(net, C, K, seed=5)          # biases 0.1: non-zero rows beyond M in a partial last tile
    rs = np.random.RandomState(6)
    x = rs.randn(B, crop * crop * C).astype(np.float32)
    y = rs.randint(0, K, size=(B, crop * crop)).astype(np.float32)
    mask = (rs.rand(B, crop * crop) > 0.3) if use_mask else None
    s = drs.Session(net, C, K, precision=prec, bn_decay=0.0)
    s.load_variables(p)
    s.train_step(x, y, crop, mask=mask)
    taps = {"x": rounded(x.reshape(B, crop, crop, C), prec)}
    M = B * crop * crop
    idx = sample_pixels(B, crop, rs) if sampled else np.arange(M)
    u, tiny = U[prec], TINY[prec]
    res = {}
    for L in layers:
        sc, co = L["scope"], L["co"]
        Z = s.debug_activation("z:" + sc, B, crop, co)
        taps[sc] = s.debug_activation(sc, B, crop, co)
        mm, mv = s.get_variable(sc + "/moving_mean"), s.get_variable(sc + "/moving_variance")
        # Z = conv + bias, stored in the session precision
        w = rounded(np.asarray(p[sc + "/weights"], np.float32), prec)
        b = np.asarray(p[sc + "/biases"], np.float64)
        z, sab = conv_at([taps[n] for n in L["inputs"]], w, L["rate"], idx, crop)
        z = z + b
        zb = u * np.abs(z) + (1 + u) * gamma(L["k"] ** 2 * L["ci"]) * (sab + np.abs(b)) + tiny
        res["Z " + sc] = ratio((tag, prec, "Z " + sc), Z.reshape(-1, co)[idx], z, zb)
        # batch statistics: fp32 sums of <= M terms per CTA, one 2^-20 fixed-point rounding per CTA (<= ceil(M/128) CTAs),
        # the fp32 result; mean and variance finished in double, stored in fp32
        Z64 = Z.reshape(-1, co).astype(np.float64)
        mean, var = Z64.mean(0), Z64.var(0)
        q = -(-M // 128) * 2.0 ** -21
        d1 = M * E24 * np.abs(Z64).sum(0) + q + E24 * np.abs(Z64.sum(0))
        d2 = (M + 1) * E24 * (Z64 ** 2).sum(0) + q
        dmean = d1 / M + 2 * E24 * np.abs(mean)
        dvar = d2 / M + 2 * np.abs(mean) * dmean + dmean ** 2
        var_ema = var * M / (M - 1)
        res["mean " + sc] = ratio((tag, prec, "mean " + sc), mm, mean, dmean + 1e-30)
        res["var " + sc] = ratio((tag, prec, "var " + sc), mv, var_ema, dvar * M / (M - 1) + 2 * E24 * var_ema + 1e-30)
        # layer output from the GPU's Z and the GPU's statistics (the moving ones, bn_decay = 0)
        need, win = post_needs(L, idx, B, crop, {})
        zn = Z.reshape(-1, co)[need].astype(np.float64)
        mg = mm.astype(np.float64)
        istd = 1.0 / np.sqrt(mv.astype(np.float64) * (M - 1) / M + EPS)
        a = act_np((zn - mg) * istd, act)
        ba = u * np.abs(a) + 8 * E24 * (np.abs(zn) + np.abs(mg)) * istd + tiny
        ref, bound = apply_post(L, a, ba, need, win, idx, B, crop, p, prec)
        res["out " + sc] = ratio((tag, prec, "out " + sc), taps[sc].reshape(-1, co)[idx], ref, bound)
    s.close()
    _assert_within(res, (tag, prec, B, crop))


@pytest.mark.parametrize("net,C,K,use_mask", TRAIN_NETS)
def test_train_forward_layers(drs, monkeypatch, net, C, K, use_mask):
    """Training forward of every training net, bf16 and fp32, whole tensors; M = 676 leaves a partial last tile."""
    t0 = time.time()
    for prec in ("bf16", "fp32"):
        check_train_forward(drs, monkeypatch, net, C, K, prec, 4, 13, use_mask, False, net)
    _print_report(net + " train", time.time() - t0)


def test_train_forward_layers_full_size(drs, monkeypatch):
    """The full-size training shape of dilated_grsl (B = 64, crop 49, M = 153 664), sampled pixels; statistics over all."""
    t0 = time.time()
    check_train_forward(drs, monkeypatch, "dilated_grsl", 4, 6, "bf16", 64, 49, False, True, "dilated_grsl B64 crop49")
    _print_report("full-size train", time.time() - t0)
