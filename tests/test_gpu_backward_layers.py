"""Teacher-forced per-layer checks of the training backward against a float64 reference.

One train_step per case under DRS_DEBUG_KEEP=1, with bn_decay = 0 (the moving mean after the step IS the batch mean the
backward used, and the batch inverse std follows from the moving variance as in check_train_forward) and weight_decay = 0
(get_gradient returns the total gradient).  Every stage's reference is computed in float64 from the GPU's own inputs to that
stage -- the exact stored values, fetched with debug_activation -- so errors cannot pile up across stages:

  loss, dlogits   from the `logits` tap, the labels and the mask / ignore label;
  classifier      dW = x^T dlogits, db = sum dlogits from the last layers' output taps;
  dout:<l>        the classifier's data gradient plus every consumer's data gradient dz:<j> (*) w_j^T -- taps flipped,
                  Ci/Co transposed, before/after pads swapped, weights rounded like the session's packers -- accumulated in step
                  order (dense nets: classifier, then the later layers in descending order; squeeze nets: _s2_2, then _s2_1);
  da:<l>          max pool: dout routed to the FIRST maximum, in row-major order, of the GPU's own z:<l> window; average pool:
                  every window's dout divided by that window's in-image count; SE gate: from pre:<l> and dout:<l>;
  dz:<l>          BN backward istd (g - mean g - xh mean(g xh)), g = da act'(xh), from z:<l>, the batch statistics and da:<l>
                  (fused bf16 pool + BN backward: dout:<l> routed as above, unrounded);
  filter grads    sum_m input tap (x) dz:<l>; conv1 reads the input as its path does (the bf16 im2col matrix on the tensor
                  cores, the fp32 input on the CUDA cores); conv biases: exactly 0 (BN without beta).

Bounds, derived from the arithmetic, none fitted:  |gpu - ref| <= u |ref| + (1 + u) e + tiny, u the storage rounding
(2^-8 bf16, 2^-24 fp32), E = 2^-24, gamma(n) = (n + 4) 2^-23 for an n-deep fp32 summation tree (adds that truncate), and e:
  * data gradient: gamma(k^2 Co) sum |dz| |w| per convolution (classifier: gamma(K) sum |dl| |w|), one rounding of each
    contribution and one of every partial sum it is added to (add_slice);
  * max / average pool routing: gamma(9) resp. (gamma(k^2) + E) times sum |terms|; the SE chain carries (value, bound)
    pairs through every product (|x| dy + |y| dx + dx dy + E |xy|) and fp32 dot product (gamma(n) sum |terms|), with the gate's
    forward bound of test_gpu_forward_layers and the hidden ReLU's kink counted as |value| where it is within its bound;
  * BN backward: sums S0 = sum g, S1 = sum g xh of depth h = ceil(rows / lanes) + lanes (bn_partial_kernel) give
    gamma(h) sum |terms| + 2^-40 per block (the fixed-point quantum) + E |S|, plus E_xh sum |g xh| on S1 with E_xh = 4E the
    error of the GPU's xh (its istd is within 2E of the one from the moving variance); the fused kernel's MODE 2 takes xh
    from the bf16 pooled activation (x10 for LeakyReLU): u |xh| more per term of S1; per element
    istd (dg + dm0 + |xh| dm1 + E_xh |xh| |m1| + 3E (|g| + |m0| + |xh m1|)) + 2E |ref|, dg the routing sum gamma(9)
    sum |terms| of the fused path and 2E |g| of the 0.1 slope;
  * filter gradient: gamma(h) sum |x| |dz| with h the summation depth of its path: pixels per split + splits on the tensor
    cores (launch_wgrad_tc mirrored below), 2M elsewhere (any tree of M terms plus at most M split partials);
  * loss and dlogits: every fp32 operation one ulp (2^-23, which also covers second-order terms), expf two.
The test prints the largest err / bound per (case, precision, quantity).
"""
import os
import time
from math import ceil

import numpy as np
import pytest

from test_gpu_forward_layers import E24, EPS, REPORT, U, _print_report, conv_at, gamma, net_layers, ratio, sample_pixels
from test_gpu_parity import TRAIN_NETS, rounded

ULP = 2.0 ** -23
TINY = 1e-30
OFFS9 = [(dy, dx) for dy in (-1, 0, 1) for dx in (-1, 0, 1)]     # the 3x3 window in row-major order
SLOPE = {0: 1.0, 1: 0.0, 2: 0.1}                                 # act'(x) for x <= 0 (identity, ReLU, LeakyReLU)


# ------------------------------------------------------------------------------------------------ float64 references
def ce_ref(lg, y, on, count=None):
    """Mean softmax cross entropy over the pixels `on` (labels outside [0, K) add no loss) and its gradient; also the per-pixel
    bound of the loss term and of the fp32 lse (every operation one ulp, expf two).  count: the pixels of the mean (None: the
    pixels `on`; data parallel: those of every rank)."""
    lg = lg.astype(np.float64)
    M, K = lg.shape
    yi = y.astype(np.int64)
    mx = lg.max(1, keepdims=True)
    se = np.exp(lg - mx).sum(1, keepdims=True)
    lse = mx + np.log(se)
    p = np.exp(lg - lse)
    onehot = (np.arange(K)[None, :] == yi[:, None]).astype(np.float64)
    valid = on & (yi >= 0) & (yi < K)
    count = float(on.sum()) if count is None else float(count)
    loss_px = np.where(valid, lse[:, 0] - lg[np.arange(M), np.clip(yi, 0, K - 1)], 0.0)
    dl = np.where(on[:, None], (p - onehot) / max(count, 1.0), 0.0)
    dlse = ULP * (2 + K + np.abs(lg - mx).max(1, keepdims=True) + 2 * np.abs(np.log(se)) + np.abs(lse))
    return dict(loss=loss_px.sum() / max(count, 1.0), loss_px=loss_px, dl=dl, p=p, lse=lse, dlse=dlse, count=count, valid=valid,
                onehot=onehot)


def flip_t(w):
    """The data-gradient filter of w [k, k, Ci, Co]: taps flipped, Ci / Co transposed -> [k, k, Co, Ci]."""
    return np.ascontiguousarray(w[::-1, ::-1].transpose(0, 1, 3, 2))


def dgrad_at(dz, w, rate, idx, crop, swap=True):
    """Data gradient of a SAME convolution at flat pixels idx: (value, sum |dz| |w|) [len(idx), Ci].  swap=False keeps the
    forward's pads (a wrong reference)."""
    total = (w.shape[0] - 1) * rate
    return conv_at([dz], flip_t(w), rate, idx, crop, pad_before=total - total // 2 if swap else total // 2)


def wgrad_ref(Xs, dz, k, rate, cols=None):
    """dW[ky, kx, c, o] = sum_m X[m + tap offset, c] dz[m, o] over the channel concatenation of Xs ([B, crop, crop, *] each) and
    the matching sum |X| |dz|, float64 [k, k, Ci, len(cols)]."""
    X = np.concatenate(Xs, -1)                            # (taps are fp32: the padded copy stays fp32)
    B, crop, ci = X.shape[0], X.shape[1], X.shape[-1]
    pad = (k - 1) * rate
    pb = pad // 2
    D = dz.reshape(-1, dz.shape[-1])
    D = (D if cols is None else D[:, cols]).astype(np.float64)
    Da = np.abs(D)
    Xp = np.zeros((B, crop + pad, crop + pad, ci), X.dtype)
    Xp[:, pb:pb + crop, pb:pb + crop] = X
    out = np.empty((k, k, ci, D.shape[1]))
    sab = np.empty_like(out)
    for ky in range(k):
        for kx in range(k):
            S = Xp[:, ky * rate:ky * rate + crop, kx * rate:kx * rate + crop].reshape(-1, ci).astype(np.float64)
            out[ky, kx] = S.T @ D
            sab[ky, kx] = np.abs(S).T @ Da
    return out, sab


def pool_route(Z, G, last=False, chunk=32):
    """3x3 SAME max-pool backward: G [B, crop, crop, C] (gradient of the pooled output) routed to the first (last=True: the
    last) maximum in row-major order of each window of Z.  Returns (dIn, sum |terms|, windows with a tie, winner's Z)."""
    B, crop, _, C = Z.shape
    da = np.zeros(Z.shape)
    sab = np.zeros(Z.shape)
    zmax = np.empty(Z.shape)
    ties = 0
    for c0 in range(0, C, chunk):
        cs = slice(c0, c0 + chunk)
        Zp = np.pad(Z[..., cs].astype(np.float32), ((0, 0), (1, 1), (1, 1), (0, 0)), constant_values=-np.inf)
        st = np.stack([Zp[:, 1 + dy:1 + dy + crop, 1 + dx:1 + dx + crop] for dy, dx in OFFS9])
        win = 8 - np.argmax(st[::-1], 0) if last else np.argmax(st, 0)
        mx = st.max(0)
        ties += int(((st == mx[None]).sum(0) > 1).sum())
        zmax[..., cs] = mx
        g = G[..., cs].astype(np.float64)
        for d, (dy, dx) in enumerate(OFFS9):
            sel = np.where(win == d, g, 0.0)
            dst = (slice(None), slice(max(0, dy), crop + min(0, dy)), slice(max(0, dx), crop + min(0, dx)), cs)
            src = sel[:, max(0, -dy):crop - max(0, dy), max(0, -dx):crop - max(0, dx)]
            da[dst] += src
            sab[dst] += np.abs(src)
    return da, sab, ties, zmax


def window_counts(crop, k):
    """In-image element count of every k x k SAME window, [crop, crop]."""
    pad = (k - 1) // 2
    i = np.arange(crop)
    n = np.minimum(crop - 1, i + pad) - np.maximum(0, i - pad) + 1
    return (n[:, None] * n[None, :]).astype(np.float64)


def avg_route(G, k, by_receiver=False):
    """k x k SAME average-pool backward: every window's gradient divided by that window's in-image count (by_receiver: by the
    receiving pixel's count, a wrong reference).  Returns (dIn, sum |terms|)."""
    B, crop, _, C = G.shape
    pad = (k - 1) // 2
    cnt = window_counts(crop, k)[None, :, :, None]
    g = G.astype(np.float64) / (1.0 if by_receiver else cnt)
    da = np.zeros(G.shape)
    sab = np.zeros(G.shape)
    for dy in range(-pad, pad + 1):
        for dx in range(-pad, pad + 1):
            dst = (slice(None), slice(max(0, dy), crop + min(0, dy)), slice(max(0, dx), crop + min(0, dx)))
            src = g[:, max(0, -dy):crop - max(0, dy), max(0, -dx):crop - max(0, dx)]
            da[dst] += src
            sab[dst] += np.abs(src)
    if by_receiver:
        da, sab = da / cnt, sab / cnt
    return da, sab


def bn_backward(Z, gin, mean, istd, act):
    """Train-mode BN (no beta / gamma) + activation backward from the gradient gin at the activation's output: rows [M, C].
    Returns xh, the gated g, and the two batch means of the formula dZ = istd (g - m0 - xh m1)."""
    Z = Z.astype(np.float64)
    xh = (Z - mean) * istd
    f = np.where(Z > mean, 1.0, SLOPE[act])            # fl(z - mean) > 0 iff z > mean: the GPU's gate, exactly
    g = gin * f
    M = Z.shape[0]
    return xh, g, g.sum(0) / M, (g * xh).sum(0) / M


def se_gate(A, p, name, px):
    """Forward SE gate with bounds (as apply_post of the forward test) from the exact pre-gate activations A [B, px, C]:
    (m, dm, h_pre, dh, h, e, de)."""
    w1, b1 = [np.asarray(p[name + "_fc1/" + n], np.float64) for n in ("weights", "biases")]
    w2, b2 = [np.asarray(p[name + "_fc2/" + n], np.float64) for n in ("weights", "biases")]
    m = A.mean(1)
    dm = gamma(ceil(px / 32) + 32) * np.abs(A).mean(1) + 2 * E24 * np.abs(m)
    hp = m @ w1 + b1
    dh = dm @ np.abs(w1) + gamma(w1.shape[0]) * (np.abs(m) @ np.abs(w1) + np.abs(b1))
    h = np.maximum(hp, 0)
    a2 = h @ w2 + b2
    e = 1.0 / (1.0 + np.exp(-a2))
    de = 0.25 * (dh @ np.abs(w2) + gamma(w2.shape[0]) * (np.abs(h) @ np.abs(w2) + np.abs(b2))) + 4 * E24
    return dict(m=m, dm=dm, hp=hp, dh=dh, h=h, e=e, de=de, w1=w1, w2=w2)


def _mul(x, y):
    """(value, bound) of a product of two (value, bound) pairs, one fp32 rounding."""
    v = x[0] * y[0]
    return v, np.abs(x[0]) * y[1] + np.abs(y[0]) * x[1] + x[1] * y[1] + E24 * np.abs(v)


def _dot(x, W, n):
    """(value, bound) of x @ W as an n-term fp32 fma chain, x a (value, bound) pair, W exact."""
    v = x[0] @ W
    return v, x[1] @ np.abs(W) + gamma(n) * (np.abs(x[0]) @ np.abs(W))


def se_backward(A, G, p, name, px):
    """SE gate backward (se_sum_kernel MODE 1, se_fc_bwd_kernel, reduce over images, se_scale_bwd_kernel) from the exact
    pre-gate activations A and output gradient G [B, px, C]: {quantity: (value, bound)} for da [B, px, C] and the four
    parameter gradients."""
    f = se_gate(A, p, name, px)
    B, _, C = A.shape
    R = f["w1"].shape[1]
    hs = ceil(px / 32) + 32
    dsum = ((G * A).sum(1), gamma(hs) * np.abs(G * A).sum(1))
    e = (f["e"], f["de"])
    q = (1.0 - f["e"], f["de"] + E24 * np.abs(1.0 - f["e"]))
    dz2 = _mul(_mul(dsum, e), q)
    a1 = _dot(dz2, f["w2"].T, C)
    amb = np.abs(f["hp"]) <= f["dh"]                     # the hidden ReLU's gate is not decided by the reference
    on = f["hp"] > 0
    dz1 = (np.where(on, a1[0], 0.0), np.where(on | amb, a1[1], 0.0) + np.where(amb, np.abs(a1[0]), 0.0))
    hv = (f["h"], f["dh"])
    sv = (f["m"], f["dm"])
    out = {}

    def over_images(x):                                  # fixed-order fp32 sum over the B images (reduce_partials_kernel)
        return x[0].sum(0), x[1].sum(0) + gamma(B) * np.abs(x[0]).sum(0)
    out["fc2/biases"] = over_images(dz2)
    out["fc1/biases"] = over_images(dz1)
    out["fc2/weights"] = over_images(_mul((hv[0][:, :, None], hv[1][:, :, None]), (dz2[0][:, None, :], dz2[1][:, None, :])))
    out["fc1/weights"] = over_images(_mul((sv[0][:, :, None], sv[1][:, :, None]), (dz1[0][:, None, :], dz1[1][:, None, :])))
    ds = _dot(dz1, f["w1"].T, R)
    ds = (ds[0] / px, ds[1] / px + 2 * E24 * np.abs(ds[0] / px))
    v = G * f["e"][:, None, :] + ds[0][:, None, :]
    out["da"] = (v, np.abs(G) * f["de"][:, None, :] + ds[1][:, None, :] + E24 * np.abs(v))
    return out


# ------------------------------------------------------------------------------------------------ summation depths
def bn_depth(M, C, sm):
    """(depth of a per-block BN sum, blocks) of bn_partial_kernel (bn_blocks, drs_train.cuh)."""
    nb = min(ceil(M / 128), sm * 2)
    lanes = 256 // (C // 8)
    return ceil(ceil(M / nb) / lanes) + lanes, nb


def cls_wgrad_depth(M, ci, sm):
    """Depth of the classifier filter gradient: per-thread rows, row lanes, block partials (classifier_bwd_weight_kernel)."""
    nb = min(ceil(M / 128), sm * 2)
    lanes = 256 // (ci // 8)
    return ceil(ceil(M / nb) / lanes) + lanes + nb


def rank_sum(parts):
    """Sum over ranks of per-rank (reference, bound) pairs, plus the exchange: one fixed-order fp32 sum of W terms,
    gamma(W - 1) sum_r |v_r| with |v_r| <= |ref_r| + bound_r (nothing for one rank)."""
    ref = sum(p[0] for p in parts)
    bound = sum(p[1] for p in parts)
    if len(parts) > 1:
        bound = bound + gamma(len(parts) - 1) * sum(np.abs(p[0]) + p[1] for p in parts)
    return ref, bound


def wgrad_tc_supported(ci, co):
    return (ci % 64 == 0 or ci == 32) and (co % 64 == 0 or co == 32) and co <= 256


def wgrad_tc_depth(M, k, ci, co, sm, part_cap):
    """Pixels per split + splits of launch_wgrad_tc (wgrad_tc.cuh)."""
    ci_pad, co_pad = -(-ci // 64) * 64, -(-co // 64) * 64
    n_tiles = (k * k * (ci_pad // 64) + 1) // 2
    acc = 64 if co_pad <= 64 else (128 if co_pad <= 128 else 256)
    T = 512 // acc
    while T > 1 and 3 * (T * 2 * 8192 + (co_pad // 64) * 8192) > 227 * 1024 - 2048:
        T -= 1
    T = min(T, n_tiles)
    n_groups = -(-n_tiles // T)
    n_chunks = -(-M // 64)
    splits = min(max(1, sm // n_groups), max(1, n_chunks // 8), part_cap // (k * k * ci_pad * co_pad))
    cps = -(-n_chunks // splits)
    return cps * 64 + -(-n_chunks // cps)


def conv1_uses_im2col(L0, prec):
    """conv1's filter gradient runs on the tensor cores from the bf16 im2col matrix (TrainWs::layout): its input is rounded."""
    return (prec == "bf16" and L0["k"] == 5 and L0["rate"] == 1 and L0["ci"] <= 5 and L0["co"] in (32, 64)
            and not os.environ.get("DRS_NO_WGRAD_CONV1_TC"))


def pool_nseg(B, crop, C, sm):
    """(nseg, seg, regime) of launch_maxpool3_bwd_apply (ops.cuh); regime: which limit chose nseg."""
    base = B * crop * (C // 8)
    fill, cap = max(1, -(-sm * 2048 // base)), max(1, crop // 4)
    n0 = min(fill, cap)
    seg = -(-crop // n0)
    return -(-crop // seg), seg, ("crop/4" if fill >= cap > 1 else ("1" if n0 == 1 else "intermediate"))


# ------------------------------------------------------------------------------------------------ one training step
class TrainRun:
    """One train_step (bn_decay = 0, DRS_DEBUG_KEEP=1) and every tap and gradient the checks read."""

    def __init__(self, drs, monkeypatch, net, C, K, prec, B, crop, use_mask=False, ignore=False, env=(), seed=5, x=None,
                 session_kw=None, y=None, mask=None, step=True):
        """x, y, mask: the feeds (None: drawn from the seed); step=False: create the session only (a data-parallel rank:
        its exchange is attached, then train() and collect() run)."""
        from oracle import nets_torch
        monkeypatch.setenv("DRS_DEBUG_KEEP", "1")
        for k in env:
            monkeypatch.setenv(k, "1")
        self.drs = drs
        self.layers, self.cls_inputs, self.act = net_layers(net, C)
        self.net, self.C, self.K, self.prec, self.B, self.crop = net, C, K, prec, B, crop
        self.M = B * crop * crop
        self.p = p = nets_torch.init_params(net, C, K, seed=seed)
        rs = np.random.RandomState(seed + 1)
        self.x = rs.randn(B, crop * crop * C).astype(np.float32) if x is None else x
        if y is None:
            y = rs.randint(0, K, size=(B, crop * crop)).astype(np.float32)
            if ignore:                                   # about 20 % of the labels are the ignored label K
                y = np.where(rs.rand(B, crop * crop) < 0.2, K, y).astype(np.float32)
            mask = (rs.rand(B, crop * crop) > 0.3) if use_mask else None
        self.y, self.ignore, self.mask = y, ignore, mask
        kw = dict(precision=prec, bn_decay=0.0, weight_decay=0.0)
        kw.update(session_kw or {})
        s = drs.Session(net, C, K, **kw)
        s.load_variables(p)
        if ignore:
            s.set_ignore_label(K)
        self.s = s
        import torch
        self.sm = torch.cuda.get_device_properties(0).multi_processor_count
        if step:
            self.train()
            self.collect()

    def train(self):
        """The training step: loss, pred and the confusion counts it returns."""
        loss, self.pred, self.cm, self.n_correct = self.s.train_step(self.x, self.y, self.crop, mask=self.mask, want_cm=True)
        self.loss = float(loss)

    def collect(self, bn_count=None):
        """Every tap and gradient the checks read.  bn_count: the pixels behind the batch statistics (None: this run's M;
        SyncBN: those of every rank), which the inverse std recovered from the unbiased moving variance needs."""
        s, B, crop, K, M = self.s, self.B, self.crop, self.K, self.M
        n = M if bn_count is None else bn_count
        self.taps = {}
        for L in self.layers:
            sc, co = L["scope"], L["co"]
            for t in ("z:", "", "dout:", "dz:", "da:", "pre:"):
                try:
                    self.taps[t + sc] = s.debug_activation(t + sc, B, crop, co)
                except self.drs.lib.DrsError:
                    assert t in ("da:", "pre:"), (t, sc)
        self.logits = s.debug_activation("logits", B, crop, K).reshape(M, K)
        self.dlogits = s.debug_activation("dlogits", B, crop, K).reshape(M, K)
        self.mean = {L["scope"]: s.get_variable(L["scope"] + "/moving_mean").astype(np.float64) for L in self.layers}
        self.istd = {L["scope"]: 1.0 / np.sqrt(s.get_variable(L["scope"] + "/moving_variance").astype(np.float64) * (n - 1) / n + EPS)
                     for L in self.layers}
        self.grad = {n: s.get_gradient(n) for n, _ in s.variable_names() if n.endswith(("/weights", "/biases")) and "/Momentum" not in n}

    def close(self):
        self.s.close()

    def loss_on(self):
        """The pixels in the mean of the loss: the mask, else every label but the ignored one."""
        if self.mask is not None:
            return self.mask.reshape(-1)
        return self.y.reshape(-1).astype(np.int64) != (self.K if self.ignore else -1)

    def w(self, scope):
        return rounded(np.asarray(self.p[scope + "/weights"], np.float32), self.prec).astype(np.float64)

    def wgrad_inputs(self, L):
        """The layer's input as its filter gradient reads it."""
        if L["inputs"] != ["x"]:
            return [self.taps[n] for n in L["inputs"]]
        x = self.x.reshape(self.B, self.crop, self.crop, self.C)
        return [rounded(x, "bf16") if conv1_uses_im2col(L, self.prec) else x]

    # ---------------------------------------------------------------- checks
    def check(self, tag, idx=None, wcols=None, mut=None):
        """{quantity: largest err / bound} over every stage of the backward; idx: pixels of the data-gradient check (None:
        all), wcols: output-channel subset of the filter-gradient check (None: all)."""
        return check_step([self], tag, idx, wcols, mut)

    def part_cap(self):
        """Floats of the filter gradients' split partials (TrainWs::layout): the largest filter x 48."""
        return max(L["k"] ** 2 * L["ci"] * L["co"] for L in self.layers) * 48


def check_step(runs, tag, idx=None, wcols=None, mut=None, sync_bn=False):
    """{quantity: largest err / bound over the ranks} over every stage of the backward of one step.  runs: the ranks of a
    data-parallel step, each with its own batch and taps (one run: the single-process step).  The per-pixel stages (dlogits,
    dout, routing, dz) are checked per rank from its own taps; the global quantities come from every rank: the loss count,
    the BN-backward sums with SyncBN (sync_bn), and the loss and parameter gradients (sums over ranks, rank_sum)."""
    mut = mut or {}
    r0 = runs[0]
    W = len(runs)
    B, crop, K, M, prec = r0.B, r0.crop, r0.K, r0.M, r0.prec
    u = U[prec]
    res = {}

    def rec(name, got, ref, bound):
        res[name] = max(res.get(name, 0.0), ratio((tag, prec, name), got, ref, bound))

    by_scope = {L["scope"]: (j, L) for j, L in enumerate(r0.layers)}
    # ---- loss and dlogits: every rank divides by the pixel count of all ranks
    ons = [r.loss_on() for r in runs]
    total = float(sum(on.sum() for on in ons))
    parts = []
    for r, on in zip(runs, ons):
        count = float(on.sum()) if mut.get("local_count") else (float(r.M) if mut.get("count_is_m") else total)
        ce = ce_ref(r.logits, r.y.reshape(-1), on, count)
        cnt = max(count, 1.0)
        d = (ce["p"] * (2 * ULP + ULP * np.abs(r.logits - ce["lse"]) + ce["dlse"]) + ULP * np.abs(ce["p"] - ce["onehot"])) / cnt
        rec("dlogits", r.dlogits, ce["dl"], np.where(on[:, None], d + 2 * ULP * np.abs(ce["dl"]), 0.0) + TINY)
        lb = ((ce["dlse"][:, 0] + ULP * ce["loss_px"]) * ce["valid"]).sum() / cnt + 8 * ULP * ce["loss_px"].sum() / cnt + 3 * ULP * abs(ce["loss"])
        parts.append((ce["loss"], lb))
    loss, lb = rank_sum(parts)
    for r in runs:
        rec("loss", np.array([r.loss]), np.array([loss]), np.array([lb + TINY]))
    dls = [r.dlogits.astype(np.float64) for r in runs]
    # ---- classifier filter gradient (fp32 weights as stored)
    xcs = [np.concatenate([r.taps[n].reshape(M, -1) for n in r.cls_inputs], 1).astype(np.float64) for r in runs]
    h = cls_wgrad_depth(M, xcs[0].shape[1], r0.sm)
    v, b = rank_sum([(xc.T @ dl, gamma(h) * (np.abs(xc).T @ np.abs(dl))) for xc, dl in zip(xcs, dls)])
    for r in runs:
        rec("classifier dW", r.grad["conv_classifier/weights"].reshape(-1, K), v, b + TINY)
    v, b = rank_sum([(dl.sum(0), gamma(h) * np.abs(dl).sum(0)) for dl in dls])
    for r in runs:
        rec("classifier db", r.grad["conv_classifier/biases"], v, b + TINY)
    # ---- data gradients: dout:<l> from the classifier and every consumer, in step order (per rank)
    idx_all = np.arange(M) if idx is None else idx
    wc = np.asarray(r0.p["conv_classifier/weights"], np.float64).reshape(-1, K)
    consumers = {L["scope"]: [] for L in r0.layers}
    off = 0
    for n in r0.cls_inputs:
        consumers[n].append(("classifier", off))
        off += by_scope[n][1]["co"]
    for j in range(len(r0.layers) - 1, -1, -1):
        Lj, off = r0.layers[j], 0
        for n in Lj["inputs"]:
            if n != "x":
                consumers[n].append((j, off))
                off += by_scope[n][1]["co"]
    for r, dl in zip(runs, dls):
        for L in r0.layers:
            sc, co = L["scope"], L["co"]
            S, Bd = None, None
            for ci, (j, o) in enumerate(consumers[sc]):
                if mut.get("drop_consumer") == sc and ci == 1:
                    continue
                if j == "classifier":
                    c = dl[idx_all] @ wc[o:o + co].T
                    cb = gamma(K) * (np.abs(dl[idx_all]) @ np.abs(wc[o:o + co]).T)
                else:
                    Lj = r0.layers[j]
                    v, sab = dgrad_at(r.taps["dz:" + Lj["scope"]], r0.w(Lj["scope"]), Lj["rate"], idx_all, crop,
                                      swap=mut.get("unswapped_pads") != Lj["scope"])
                    c, cb = v[:, o:o + co], gamma(Lj["k"] ** 2 * Lj["co"]) * sab[:, o:o + co]
                cb = u * np.abs(c) + (1 + u) * cb                   # its own rounding (direct write or the add_slice scratch)
                if S is None:
                    S, Bd = c, cb
                else:
                    S = S + c
                    Bd = Bd + cb + u * (np.abs(S) + Bd + cb)      # the add_slice rounding
            rec("dout " + sc, r.taps["dout:" + sc].reshape(M, co)[idx_all], S, Bd + TINY)
    # ---- per layer: post-op backward (per rank), BN backward (its sums over every rank with SyncBN), filter gradient
    Mbn = M * W if sync_bn else M
    exh = 4 * E24
    for L in r0.layers:
        sc, co, post = L["scope"], L["co"], L["post"]
        per, se_parts = [], {}
        for r in runs:
            Z = r.taps["z:" + sc]
            G = r.taps["dout:" + sc]
            mean, istd = r.mean[sc], r.istd[sc]
            eg = np.zeros((M, co))
            fused = None
            if post is None:
                gin = r.taps["da:" + sc].reshape(M, co).astype(np.float64)
                assert np.array_equal(r.taps["da:" + sc], G), sc       # no post-op: the BN reads dout itself
            elif post[0] == "max":
                ref, sab, _, zmax = pool_route(Z, G, last=mut.get("last_tie", False))
                if "da:" + sc in r.taps:
                    rec("pool " + sc, r.taps["da:" + sc], ref, u * np.abs(ref) + (1 + u) * gamma(9) * sab + TINY)
                    gin = r.taps["da:" + sc].reshape(M, co).astype(np.float64)
                else:                                          # fused pool + BN backward: the routed sum in fp32
                    assert prec == "bf16" and not mut.get("last_tie"), sc
                    gin, eg = ref.reshape(M, co), gamma(9) * sab.reshape(M, co)
                    zw = zmax.reshape(M, co).astype(np.float64)
                    f = np.where(zw > mean, 1.0, SLOPE[r.act])
                    t0 = np.abs(G.reshape(M, co) * f)
                    fused = (t0.sum(0), (t0 * np.abs(zw - mean) * istd).sum(0))
            elif post[0] == "avg":
                ref, sab = avg_route(G, post[1], by_receiver=mut.get("avg_by_receiver", False))
                rec("avgpool " + sc, r.taps["da:" + sc], ref, u * np.abs(ref) + (1 + u) * (gamma(post[1] ** 2) + E24) * sab + TINY)
                gin = r.taps["da:" + sc].reshape(M, co).astype(np.float64)
            else:
                px = crop * crop
                A = r.taps["pre:" + sc].reshape(B, px, co).astype(np.float64)
                out = se_backward(A, G.reshape(B, px, co).astype(np.float64), r.p, post[2], px)
                v, e = out.pop("da")
                rec("se da " + sc, r.taps["da:" + sc].reshape(B, px, co), v, u * np.abs(v) + (1 + u) * e + TINY)
                for q, ve in out.items():
                    se_parts.setdefault(q, []).append(ve)
                gin = r.taps["da:" + sc].reshape(M, co).astype(np.float64)
            # BN-backward sums of this rank: S0 = sum g, S1 = sum g xh
            Zr = Z.reshape(M, co)
            xh, g, _, _ = bn_backward(Zr, gin, mean, istd, r.act)
            neg = (Zr <= mean) & (r.act == 2)
            eg = eg * np.where(Zr > mean, 1.0, SLOPE[r.act]) + np.where(neg, 2 * E24 * np.abs(g), 0.0)
            h, nb = bn_depth(M, co, r0.sm)
            A0, A1 = (np.abs(g).sum(0), np.abs(g * xh).sum(0)) if fused is None else fused
            S0, S1 = g.sum(0), (g * xh).sum(0)
            dS0 = (gamma(h) + 2 * E24) * A0 + nb * 2.0 ** -40 + E24 * np.abs(S0)
            dS1 = (gamma(h) + 2 * E24 + exh + (u + 4 * E24 if fused is not None else 0.0)) * A1 + nb * 2.0 ** -40 + E24 * np.abs(S1)
            per.append(dict(xh=xh, g=g, eg=eg, istd=istd, s0=(S0, dS0), s1=(S1, dS1)))
        for q, parts in se_parts.items():
            v, e = rank_sum(parts)
            for r in runs:
                rec("se %s %s" % (q, sc), r.grad[post[2] + "_" + q].reshape(v.shape), v, e + TINY)
        if sync_bn and not mut.get("bn_sums_one_rank"):          # the all-reduced sums
            s0, s1 = rank_sum([q["s0"] for q in per]), rank_sum([q["s1"] for q in per])
            for q in per:
                q["s0"], q["s1"] = s0, s1
        # BN backward dZ = istd (g - m0 - xh m1), m0 / m1 the sums over the pixels behind the statistics
        for r, q in zip(runs, per):
            xh, g, eg, istd = q["xh"], q["g"], q["eg"], q["istd"]
            (S0, dS0), (S1, dS1) = q["s0"], q["s1"]
            m0, m1 = S0 / Mbn, S1 / Mbn
            dm0, dm1 = dS0 / Mbn + E24 * np.abs(m0), dS1 / Mbn + E24 * np.abs(m1)
            ref = istd * (g - m0 - (0.0 if mut.get("bn_drop_s1") else xh * m1))
            err = istd * (eg + dm0 + np.abs(xh) * dm1 + exh * np.abs(xh) * np.abs(m1) + 3 * E24 * (np.abs(g) + np.abs(m0) + np.abs(xh * m1)))
            err = err + 2 * E24 * np.abs(ref)
            rec("dz " + sc, r.taps["dz:" + sc].reshape(M, co), ref, u * np.abs(ref) + (1 + u) * err + TINY)
        # filter gradient (summed over ranks) and the (absent) bias gradient
        cols = np.arange(co) if wcols is None else wcols(co)
        if L["inputs"] == ["x"]:
            tc = conv1_uses_im2col(L, prec)
            depth = wgrad_tc_depth(M, 1, 128, co, r0.sm, r0.part_cap()) if tc else 2 * M
        else:
            tc = prec == "bf16" and wgrad_tc_supported(L["ci"], co)
            depth = wgrad_tc_depth(M, L["k"], L["ci"], co, r0.sm, r0.part_cap()) if tc else 2 * M
        parts = []
        for i, r in enumerate(runs):
            if mut.get("drop_rank_share") == sc and i == W - 1:
                continue
            v, sab = wgrad_ref(r.wgrad_inputs(L), r.taps["dz:" + sc], L["k"], L["rate"], cols)
            if mut.get("transpose_taps"):
                v = v.transpose(1, 0, 2, 3)
            parts.append((v, gamma(depth) * sab))
        v, b = rank_sum(parts)
        for r in runs:
            gw = r.grad[sc + "/weights"].reshape(L["k"], L["k"], L["ci"], co)[..., cols]
            rec("dW " + sc, gw, v, b + TINY)
            assert not r.grad[sc + "/biases"].any(), sc
    return res


def _assert_within(res, what):
    bad = {k: v for k, v in res.items() if not v <= 1.0}
    assert not bad, (what, bad)


def _subset_cols(rs, n_random=8):
    """Output channels of the filter-gradient check at large sizes: the first and last of every 64-wide tile, plus random."""
    def pick(co):
        t = np.arange(0, co, 64)
        return np.unique(np.concatenate([t, np.minimum(t + 63, co - 1), rs.randint(0, co, n_random)]))
    return pick


def _run(drs, monkeypatch, net, C, K, prec, B, crop, tag, idx_fn=None, wcols=None, **kw):
    r = TrainRun(drs, monkeypatch, net, C, K, prec, B, crop, **kw)
    try:
        idx = idx_fn(r) if idx_fn else None
        res = r.check(tag, idx=idx, wcols=wcols)
    finally:
        r.close()
    _assert_within(res, (tag, prec, B, crop))
    return r


# ------------------------------------------------------------------------------------------------ GPU cases
@pytest.mark.gpu
@pytest.mark.parametrize("net,C,K,use_mask", TRAIN_NETS)
def test_backward_layers(drs, monkeypatch, net, C, K, use_mask):
    """Every stage of the backward of every training net, bf16 and fp32, whole tensors; M = 676 leaves a partial last tile.
    The masked nets use a mask."""
    t0 = time.time()
    for prec in ("bf16", "fp32"):
        _run(drs, monkeypatch, net, C, K, prec, 4, 13, net, use_mask=use_mask)
    _print_report(net + " backward", time.time() - t0)


@pytest.mark.gpu
def test_backward_with_ignore_label(drs, monkeypatch):
    """set_ignore_label(K), no mask: about 20 % of the labels are K; the loss count comes from mask_count_kernel."""
    t0 = time.time()
    for prec in ("bf16", "fp32"):
        _run(drs, monkeypatch, "dilated_grsl", 4, 6, prec, 4, 13, "dilated_grsl ignore", ignore=True)
    _print_report("ignore label", time.time() - t0)


@pytest.mark.gpu
@pytest.mark.parametrize("net,C,K", [("dilated_icpr_rate6_avgpool", 3, 2), ("dilated_icpr_rate6_SE", 4, 6)])
def test_backward_tiny_crop(drs, monkeypatch, net, C, K):
    """B = 3, crop 5: the 7x7 average-pool window is wider than the image and the SE gate averages over 25 pixels."""
    t0 = time.time()
    for prec in ("bf16", "fp32"):
        _run(drs, monkeypatch, net, C, K, prec, 3, 5, net + " crop5")
    _print_report(net + " crop 5", time.time() - t0)


@pytest.mark.gpu
@pytest.mark.parametrize("net,C,K,use_mask", [n for n in TRAIN_NETS if "grsl" in n[0]])
def test_backward_separate_pool_kernels(drs, monkeypatch, net, C, K, use_mask):
    """The separate pool and BN backward kernels of the bf16 pooling nets (DRS_NO_FUSED_POOL_APPLY=1): the path that stores
    the pool's input gradient da:<l>."""
    t0 = time.time()
    _run(drs, monkeypatch, net, C, K, "bf16", 4, 13, net + " unfused", use_mask=use_mask, env=("DRS_NO_FUSED_POOL_APPLY",))
    _print_report(net + " unfused pool", time.time() - t0)


POOL_SWEEP = ((2, 3), (1, 17), (4, 13), (150, 27), (730, 13))


@pytest.mark.gpu
def test_fused_pool_backward_row_segments(drs, monkeypatch):
    """pool_lean::bwd_apply_kernel at every row-segment regime of launch_maxpool3_bwd_apply -- nseg = crop/4, an intermediate
    value and 1 --, segment lengths = 0, 1 and 2 (mod 3) (the row loop is unrolled by three), a last segment shorter than
    the others, and crop 3.  Large cases check the data gradient at sampled pixels, BN and routing on whole tensors."""
    import torch
    sm = torch.cuda.get_device_properties(0).multi_processor_count
    layers, _, _ = net_layers("dilated_grsl", 4)
    seen = {"regime": set(), "seg mod 3": set(), "short last": False, "crop 3": False}
    rs = np.random.RandomState(19)
    t0 = time.time()
    for B, crop in POOL_SWEEP:
        for L in layers:
            nseg, seg, regime = pool_nseg(B, crop, L["co"], sm)
            seen["regime"].add(regime)
            seen["seg mod 3"].add(seg % 3)
            seen["short last"] |= crop - (nseg - 1) * seg < seg
        seen["crop 3"] |= crop == 3
        large = B * crop * crop > 4096
        _run(drs, monkeypatch, "dilated_grsl", 4, 6, "bf16", B, crop, "grsl B%d crop%d" % (B, crop),
             idx_fn=(lambda r: sample_pixels(r.B, r.crop, rs)) if large else None, wcols=_subset_cols(rs) if large else None)
    print("pool backward row segments covered:", seen)
    assert seen == {"regime": {"crop/4", "intermediate", "1"}, "seg mod 3": {0, 1, 2}, "short last": True, "crop 3": True}, seen
    _print_report("pool row segments", time.time() - t0)


@pytest.mark.gpu
def test_backward_full_size(drs, monkeypatch):
    """The product training shape: dilated_grsl in bf16 at B = 64, crop 49 (M = 153 664).  dout at sampled pixels, BN and
    pool on whole tensors, filter gradients on all rows and the first / last output channel of every 64-wide tile plus
    random ones."""
    rs = np.random.RandomState(23)
    t0 = time.time()
    _run(drs, monkeypatch, "dilated_grsl", 4, 6, "bf16", 64, 49, "grsl B64 crop49", idx_fn=lambda r: sample_pixels(r.B, r.crop, rs),
         wcols=_subset_cols(rs))
    _print_report("full-size backward", time.time() - t0)


@pytest.mark.gpu
def test_momentum_update(drs, monkeypatch):
    """One step with weight_decay > 0, non-zero momentum slots and a global step past a decay_steps boundary: every slot is
    mom a + g_total and every variable w - lr a' (either rounding of the product) to within one ulp, g_total is the CE
    gradient of the same step without weight decay plus wd w, and the loss is CE + wd/2 sum w^2 over the pre-step weights."""
    net, C, K, B, crop = "dilated_grsl", 4, 6, 4, 13
    wd, lr0, mom, decay_steps, step = 0.005, 0.01, 0.9, 3, 7
    kw = dict(weight_decay=wd, lr_initial=lr0, momentum=mom, decay_steps=decay_steps, decay_rate=0.5)
    from oracle import nets_torch
    monkeypatch.setenv("DRS_DEBUG_KEEP", "1")
    p = nets_torch.init_params(net, C, K, seed=5)
    rs = np.random.RandomState(29)
    slots = None
    runs = []
    for w in (wd, 0.0):
        s = drs.Session(net, C, K, precision="bf16", bn_decay=0.0, **dict(kw, weight_decay=w))
        s.load_variables(p)
        names = [n for n, _ in s.variable_names() if n.endswith("/Momentum")]
        if slots is None:
            slots = {n: (rs.randn(dict(s.variable_names())[n]) * 0.01).astype(np.float32) for n in names}
        for n, v in slots.items():
            s.set_variable(n, v)
        s.set_variable("global_step", np.array([step], np.float32))
        x = np.random.RandomState(31).randn(B, crop * crop * C).astype(np.float32)
        y = np.random.RandomState(37).randint(0, K, size=(B, crop * crop)).astype(np.float32)
        loss = float(s.train_step(x, y, crop)[0])
        logits = s.debug_activation("logits", B, crop, K).reshape(-1, K)
        out = {n[:-len("/Momentum")]: (s.get_gradient(n[:-len("/Momentum")]), s.get_variable(n), s.get_variable(n[:-len("/Momentum")]))
               for n in names}
        runs.append((loss, logits, out, y))
        s.close()
    (loss, logits, out, y), (_, _, out0, _) = runs
    lr = float(np.float32(lr0) * np.float32(0.5) ** (step // decay_steps))
    momf, wdf = float(np.float32(mom)), float(np.float32(wd))
    worst = {}
    l2 = 0.0

    def ulp(v):
        return np.spacing(np.abs(v).astype(np.float32)).astype(np.float64)
    for n, (g, a, wv) in out.items():
        w0 = np.asarray(p[n], np.float64).reshape(-1)
        a0 = slots[n + "/Momentum"].astype(np.float64)
        g0 = out0[n][0].astype(np.float64)
        gref = g0 + wdf * w0 if n.endswith("/weights") else g0
        if n.endswith("/weights"):
            l2 += (w0 ** 2).sum()
        worst[n] = max(float((np.abs(g - gref) / ulp(g)).max()),
                       float((np.abs(a - (momf * a0 + g.astype(np.float64))) / ulp(a)).max()),
                       float((np.abs(wv - (w0 - lr * a.astype(np.float64))) / (ulp(wv) + 0.5 * ulp(lr * a.astype(np.float64)))).max()))
    print("momentum update, largest error in ulps per variable:", {k: round(v, 3) for k, v in worst.items()})
    assert max(worst.values()) <= 1.0, worst
    ce = ce_ref(logits, y.reshape(-1), np.ones(y.size, bool))
    ref = ce["loss"] + 0.5 * wdf * l2
    bound = (ce["dlse"][:, 0] + ULP * ce["loss_px"]).sum() / y.size + 8 * ULP * ce["loss"] + 0.5 * wdf * 10 * ULP * l2 + 4 * ULP * abs(ref)
    assert abs(loss - ref) <= bound, (loss, ref, bound)


@pytest.mark.gpu
def test_wrong_backward_references_break_the_bounds(drs, monkeypatch):
    """The bounds tell a right answer from a wrong one: on the GPU's own taps each of these wrong references exceeds its bound
    at least 10x -- the data gradient of the k=4, rate-3 layer with the forward's pads, the max-pool gradient routed to the
    LAST tied maximum (on an input with many bf16 ties), the average-pool gradient divided by the receiving pixel's count, the
    BN backward without its xh mean(g xh) term, the filter gradient with its taps transposed, and the squeeze _s1 gradient
    with one consumer dropped."""
    got = {}
    t0 = time.time()
    r = TrainRun(drs, monkeypatch, "dilated_grsl", 4, 6, "bf16", 3, 25, env=("DRS_NO_FUSED_POOL_APPLY",))
    try:
        _assert_within(r.check("sensitivity"), "right reference")
        got["unswapped pads"] = r.check("wrong", mut={"unswapped_pads": "conv3"})["dout conv2"]
        got["bn without s1"] = max(v for k, v in r.check("wrong", mut={"bn_drop_s1": True}).items() if k.startswith("dz "))
        got["transposed taps"] = max(v for k, v in r.check("wrong", mut={"transpose_taps": True}).items() if k.startswith("dW "))
    finally:
        r.close()
    # piecewise-constant input (12 x 12 blocks): the conv outputs are equal across the blocks' interiors -> bf16 ties
    x = np.repeat(np.repeat(np.random.RandomState(41).randn(3, 2, 2, 4), 12, 1), 12, 2).astype(np.float32).reshape(3, -1)
    r = TrainRun(drs, monkeypatch, "dilated_grsl", 4, 6, "bf16", 3, 24, env=("DRS_NO_FUSED_POOL_APPLY",), x=x)
    try:
        _assert_within(r.check("sensitivity ties"), "right reference, ties")
        _, _, ties, _ = pool_route(r.taps["z:conv1"], r.taps["dout:conv1"])
        assert ties > r.M * r.layers[0]["co"] // 10, ties          # many windows with a tied maximum
        got["last tied maximum"] = r.check("wrong", mut={"last_tie": True})["pool conv1"]
    finally:
        r.close()
    r = TrainRun(drs, monkeypatch, "dilated_icpr_rate6_avgpool", 3, 2, "bf16", 3, 5)
    try:
        got["avg count of receiver"] = max(v for k, v in r.check("wrong", mut={"avg_by_receiver": True}).items() if k.startswith("avgpool "))
    finally:
        r.close()
    r = TrainRun(drs, monkeypatch, "dilated_icpr_rate6_squeeze", 4, 6, "bf16", 4, 13)
    try:
        got["squeeze consumer dropped"] = r.check("wrong", mut={"drop_consumer": "conv4_s1"})["dout conv4_s1"]
    finally:
        r.close()
    REPORT.clear()
    print("wrong backward references, largest err / bound:", got, "%.1f s" % (time.time() - t0))
    assert all(v >= 10.0 for v in got.values()), got


# ------------------------------------------------------------------------------------------------ CPU: references vs autograd
def _t(a):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a)).double()


def _conv_t(x, w, rate):
    import torch.nn.functional as F
    k = w.shape[0]
    total = (k - 1) * rate
    xt = x.permute(0, 3, 1, 2)
    y = F.conv2d(F.pad(xt, (total // 2, total - total // 2, total // 2, total - total // 2)), w.permute(3, 2, 0, 1), dilation=rate)
    return y.permute(0, 2, 3, 1)


def test_float64_references_match_autograd():
    """The reference functions above against torch.autograd in float64: data and filter gradients of every (k, rate) of the
    nets, first-maximum routing on quantised inputs with ties, average pooling at crop 5 with k = 7, BN + activation, the SE
    gate and masked / ignore-label cross entropy."""
    import torch
    import torch.nn.functional as F
    from oracle import nets_torch as nt
    rs = np.random.RandomState(3)
    kr = sorted({(k, r) for spec in nt.NET_SPECS.values() for (k, r, _) in spec["convs"]} |
                {(k, r) for spec in nt.NET_SPECS.values() for (_, _, _, _, k, r) in spec.get("squeeze", ())} | {(1, 1)})
    for (k, rate) in kr:
        B, crop, ci, co = 2, 9, 3, 5
        x = _t(rs.randn(B, crop, crop, ci)).requires_grad_(True)
        w = _t(rs.randn(k, k, ci, co)).requires_grad_(True)
        dy = rs.randn(B, crop, crop, co)
        (_conv_t(x, w, rate) * _t(dy)).sum().backward()
        dx, _ = dgrad_at(dy, w.detach().numpy(), rate, np.arange(B * crop * crop), crop)
        assert np.allclose(dx, x.grad.numpy().reshape(-1, ci), rtol=1e-12, atol=1e-12), (k, rate)
        dw, sab = wgrad_ref([x.detach().numpy()], dy, k, rate)
        assert np.allclose(dw, w.grad.numpy(), rtol=1e-12, atol=1e-11), (k, rate)
        assert np.all(sab >= np.abs(dw) - 1e-12)
        if (k - 1) * rate % 2:                                  # asymmetric pads: the unswapped reference differs
            wrong, _ = dgrad_at(dy, w.detach().numpy(), rate, np.arange(B * crop * crop), crop, swap=False)
            assert not np.allclose(wrong, dx)
    # max pool, first maximum on ties (PyTorch's CPU kernel keeps the first strictly greater element in row-major order)
    for crop, C in ((7, 8), (3, 4), (6, 16)):
        z = np.round(rs.randn(2, crop, crop, C) * 2) / 2
        g = rs.randn(2, crop, crop, C)
        zt = _t(z).requires_grad_(True)
        pooled = F.max_pool2d(F.pad(zt.permute(0, 3, 1, 2), (1, 1, 1, 1), value=-np.inf), 3, 1)
        (pooled.permute(0, 2, 3, 1) * _t(g)).sum().backward()
        da, sab, ties, zmax = pool_route(z, g)
        assert ties > 0 and np.allclose(da, zt.grad.numpy(), atol=1e-12), crop
        assert np.array_equal(zmax, pooled.detach().permute(0, 2, 3, 1).numpy())
        last, _, _, _ = pool_route(z, g, last=True)
        assert not np.allclose(last, da)
    # average pool (TF SAME: divide by the in-image count), 7x7 at crop 5 and 5x5 at crop 9
    for crop, k in ((5, 7), (9, 5), (5, 5)):
        a = _t(rs.randn(2, crop, crop, 8)).requires_grad_(True)
        g = rs.randn(2, crop, crop, 8)
        pooled = F.avg_pool2d(a.permute(0, 3, 1, 2), k, 1, k // 2, count_include_pad=False)
        (pooled.permute(0, 2, 3, 1) * _t(g)).sum().backward()
        da, _ = avg_route(g, k)
        assert np.allclose(da, a.grad.numpy(), atol=1e-12), (crop, k)
        assert not np.allclose(avg_route(g, k, by_receiver=True)[0], da)
    # BN (batch statistics, no beta / gamma) + ReLU / LeakyReLU / identity
    for act in (0, 1, 2):
        z = rs.randn(300, 16) * 1.5 + 0.3
        g = rs.randn(300, 16)
        zt = _t(z).requires_grad_(True)
        mean, var = zt.mean(0), zt.var(0, unbiased=False)
        xh = (zt - mean) / torch.sqrt(var + EPS)
        a = torch.relu(xh) if act == 1 else (torch.maximum(0.1 * xh, xh) if act == 2 else xh)
        (a * _t(g)).sum().backward()
        zm = z.mean(0)
        xh_, gg, m0, m1 = bn_backward(z, g, zm, 1.0 / np.sqrt(z.var(0) + EPS), act)
        assert np.allclose((1.0 / np.sqrt(z.var(0) + EPS)) * (gg - m0 - xh_ * m1), zt.grad.numpy(), atol=1e-12), act
    # SE gate: mean -> FC -> ReLU -> FC -> sigmoid -> scale, every gradient
    B, px, C, R = 3, 25, 16, 4
    p = {"se_fc1/weights": rs.randn(C, R) * 0.3, "se_fc1/biases": rs.randn(R) * 0.1,
         "se_fc2/weights": rs.randn(R, C) * 0.3, "se_fc2/biases": rs.randn(C) * 0.1}
    A = np.abs(rs.randn(B, px, C))
    G = rs.randn(B, px, C)
    pt = {k: _t(v).requires_grad_(True) for k, v in p.items()}
    At = _t(A).requires_grad_(True)
    hid = torch.relu(At.mean(1) @ pt["se_fc1/weights"] + pt["se_fc1/biases"])
    e = torch.sigmoid(hid @ pt["se_fc2/weights"] + pt["se_fc2/biases"])
    (At * e[:, None, :] * _t(G)).sum().backward()
    out = se_backward(A, G, p, "se", px)
    assert np.allclose(out["da"][0], At.grad.numpy(), atol=1e-12)
    for q in ("fc1/weights", "fc1/biases", "fc2/weights", "fc2/biases"):
        assert np.allclose(out[q][0], pt["se_" + q].grad.numpy(), atol=1e-12), q
        assert np.all(out[q][1] >= 0), q
    # cross entropy over masked pixels and with an ignored label (labels outside [0, K) add nothing)
    M, K = 200, 6
    lg = rs.randn(M, K) * 3
    y = rs.randint(0, K + 1, size=M).astype(np.float64)
    for on in (rs.rand(M) > 0.3, y != K):
        lt = _t(lg).requires_grad_(True)
        valid = torch.from_numpy(on & (y < K))
        lp = torch.log_softmax(lt, 1)
        loss = -(lp[torch.arange(M), torch.from_numpy(np.minimum(y, K - 1).astype(np.int64))] * valid).sum() / float(on.sum())
        loss.backward()
        ce = ce_ref(lg, y, on)
        assert abs(ce["loss"] - loss.item()) < 1e-12
        dl_t = np.where(on[:, None], lt.grad.numpy(), 0.0)
        assert np.allclose(ce["dl"][on & (y < K)], dl_t[on & (y < K)], atol=1e-12)
        assert not ce["dl"][~on].any()
