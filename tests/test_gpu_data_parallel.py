"""The data-parallel training step, layer by layer, on one GPU: W sessions on one device are the ranks, each stepping in its
own Python thread, and they exchange through the allreduce callback (Session.set_allreduce, the path of DRS_COMM=torch).
That runs every line of the library's data-parallel code except the NCCL call itself: the SyncBN reductions, the global
pixel count, the two gradient buckets and the extras (loss numerator and confusion counts) packed behind the gradients.

The exchange model (Exchange below): a rank's callback synchronises the stream it was handed and waits at a barrier; once
all W have arrived, one thread sums the W buffers in fixed order ((b0 + b1) + b2) + ... in fp32 on a private stream and
writes the sum into every rank's buffer; every rank then logs (pointer, count, stream).  The result is deterministic and
the same on every rank, and its error is one fp32 sum of W terms: gamma(W - 1) sum_r |v_r| (rank_sum).  Any rank that
fails aborts the barrier, so a schedule on which the ranks disagree fails the test instead of hanging it.

Checks, per step (W ranks, B_r patches each, bn_decay = 0, weight_decay = 0, DRS_DEBUG_KEEP=1, as in TrainRun):
  * the exchange schedule, exactly, on every rank: with SyncBN one reduction of 2 co floats per layer in step order, then
    one per layer in backward order; one float (the pixel count) with a mask or the ignore label; with L >= 4 layers the
    bucket [w_off(L-3), n_trainable + K^2 + 2) right after layer L-3's backward reduction, on a stream other than the
    front range's; the front range [0, w_off(L-3)) last, at the buffer base; DRS_NO_BUCKETS=1 or L < 4: one reduction of
    the whole buffer.  The offsets come from the variable order of build_net (trainable_offsets);
  * the forward statistics: every rank's moving mean and variance against float64 statistics of the concatenated z: taps
    of all ranks (SyncBN, unbiased with Mg = W M_r) or of its own (no SyncBN; they then differ between ranks).  Bound of
    test_gpu_forward_layers per rank, plus the fp32 rounding of each rank's sums and the exchange;
  * every stage of the backward, check_step of test_gpu_backward_layers: per-pixel stages per rank from its own taps;
    dlogits and the loss divided by the count of all ranks; with SyncBN the BN-backward sums S0, S1 of all ranks over
    Mg, in the separate and the fused pool + BN backward; the loss, the classifier, filter and SE-parameter gradients
    as sums over ranks of the per-rank float64 references, bound: the per-rank bounds summed plus the exchange term;
    conv biases exactly 0;
  * the confusion counts: exactly the sum of the ranks' host bincounts of (label, pred) over the counted pixels;
  * after the step every rank holds bit-identical variables and momentum slots (and moving statistics with SyncBN); a
    second run, DRS_NO_BUCKETS=1 and DRS_NO_OVERLAP=1 change no bit.
The test prints the largest err / bound per (case, precision, quantity).
"""
import os
import threading
import time

import numpy as np
import pytest

from test_gpu_backward_layers import TrainRun, _assert_within, _subset_cols, check_step
from test_gpu_forward_layers import E24, REPORT, _print_report, gamma, net_layers, ratio, sample_pixels
from test_gpu_parity import TRAIN_NETS

TIMEOUT = 120.0                                  # seconds a rank may wait for the others at one exchange


# ------------------------------------------------------------------------------------------------ the exchange
class Exchange:
    """The in-process allreduce of W ranks (module docstring); fn(r) is rank r's callback, log[r] what it was called with."""

    def __init__(self, W):
        import torch
        self.W = W
        self.bufs = [None] * W
        self.log = [[] for _ in range(W)]
        self.errors = []
        self.stream = torch.cuda.Stream()
        self.barrier = threading.Barrier(W, action=self._sum, timeout=TIMEOUT)

    def _sum(self):
        """Run by one thread once every rank has arrived: the fixed-order fp32 sum, written back to every buffer."""
        import torch
        counts = [t.numel() for t in self.bufs]
        if len(set(counts)) != 1:
            raise AssertionError("ranks exchange different counts at the same point: %s" % counts)
        with torch.cuda.stream(self.stream):
            acc = self.bufs[0].clone()
            for t in self.bufs[1:]:
                acc += t
            for t in self.bufs:
                t.copy_(acc)
        self.stream.synchronize()

    def fn(self, r):
        import torch
        from drs_b200 import dist

        def allreduce(ptr, count, stream):
            try:
                (torch.cuda.ExternalStream(stream) if stream else torch.cuda.default_stream()).synchronize()
                self.bufs[r] = torch.as_tensor(dist._DevBuf(ptr, count), device="cuda")
                self.barrier.wait()
                self.log[r].append((ptr, count, stream))
            except Exception as e:
                self.errors.append((r, e))
                self.barrier.abort()
                raise
        return allreduce


def step_ranks(runs, ex):
    """train() of every rank in its own thread; re-raises the first failure (a hang past the timeouts fails too)."""
    errs = [None] * len(runs)

    def work(r):
        try:
            runs[r].train()
        except BaseException as e:
            errs[r] = e
            ex.barrier.abort()
    threads = [threading.Thread(target=work, args=(r,), daemon=True) for r in range(len(runs))]
    for t in threads:
        t.start()
    for t in threads:
        t.join(4 * TIMEOUT)
    if any(t.is_alive() for t in threads):
        ex.barrier.abort()
        raise AssertionError("a data-parallel rank did not finish its step")
    root = [e for _, e in ex.errors if not isinstance(e, threading.BrokenBarrierError)]
    if root:
        raise root[0]
    for e in errs:
        if e is not None:
            raise e


# ------------------------------------------------------------------------------------------------ schedule
def trainable_offsets(layers, cls_inputs, K):
    """({scope: offset of its weights in the flat parameter buffer}, n_trainable) in build_net's variable order: per
    convolution its weights, its biases and any SE gate parameters, then the classifier."""
    off, w_off, co = 0, {}, {}
    for L in layers:
        w_off[L["scope"]] = off
        co[L["scope"]] = L["co"]
        off += L["k"] ** 2 * L["ci"] * L["co"] + L["co"]
        if L["post"] is not None and L["post"][0] == "se":
            c, r = L["co"], L["co"] // L["post"][1]
            off += 2 * c * r + r + c
    cls_in = sum(co[n] for n in cls_inputs)
    return w_off, off + cls_in * K + K


def expected_schedule(layers, cls_inputs, K, W, sync_bn, counted, buckets):
    """[(stage, count)] of the exchanges of one step, in order, from the net description."""
    w_off, n_tr = trainable_offsets(layers, cls_inputs, K)
    total = n_tr + K * K + 2
    L = len(layers)
    split = L - 3 if (W > 1 and buckets and L >= 4) else -1
    out = [("bn forward " + l["scope"], 2 * l["co"]) for l in layers] if sync_bn else []
    if counted:
        out.append(("pixel count", 1))
    for l in range(L - 1, -1, -1):
        if sync_bn:
            out.append(("bn backward " + layers[l]["scope"], 2 * layers[l]["co"]))
        if l == split:
            out.append(("bucket", total - w_off[layers[l]["scope"]]))
    out.append(("front range", w_off[layers[split]["scope"]]) if split >= 0 else ("whole buffer", total))
    return out, (w_off[layers[split]["scope"]] if split >= 0 else None), total


def check_schedule(run0, log, W, sync_bn, counted, buckets, tag):
    """Every rank's log against the schedule; the bucket and the front range cover the gradient buffer exactly once."""
    exp, split_off, total = expected_schedule(run0.layers, run0.cls_inputs, run0.K, W, sync_bn, counted, buckets)
    sizes = dict(run0.s.variable_names())
    assert total == sum(c for n, c in sizes.items() if n.endswith(("/weights", "/biases")) and "/Momentum" not in n) + run0.K ** 2 + 2, tag
    for r, lg in enumerate(log):
        got = [c for _, c, _ in lg]
        for i, (stage, c) in enumerate(exp):
            assert i < len(got) and got[i] == c, (tag, "rank %d: exchange %d should be %s of %d floats" % (r, i, stage, c),
                                                  got[i] if i < len(got) else "missing", [e[0] for e in exp])
        assert len(got) == len(exp), (tag, "rank %d: %d exchanges after the %s" % (r, len(got) - len(exp), exp[-1][0]))
        assert [c for _, c, _ in lg] == [c for _, c, _ in log[0]], (tag, "ranks exchange different schedules")
        base, _, s_front = lg[-1]
        if split_off is not None:
            b_ptr, b_cnt, s_bucket = [e for e, (stage, _) in zip(lg, exp) if stage == "bucket"][0]
            assert b_ptr - base == 4 * split_off, (tag, "bucket at byte %d of the gradient buffer, expected %d" % (b_ptr - base, 4 * split_off))
            assert split_off + b_cnt == total, (tag, "front range + bucket do not cover the buffer")
            assert s_bucket != s_front, (tag, "the bucket is exchanged on the front range's stream")
        # the BN sums and the pixel count go on the handle's stream, which is the front range's
        assert all(s == s_front for (_, _, s), (stage, _) in zip(lg, exp) if stage != "bucket"), tag


# ------------------------------------------------------------------------------------------------ forward statistics
def check_stats(runs, sync_bn, tag, mut=None):
    """Moving mean / variance (bn_decay = 0: the batch statistics, unbiased) of every rank against float64 statistics of
    the z: taps of every rank (SyncBN) or of its own.  Bound of check_train_forward per rank sum (depth M_r, one 2^-20
    fixed-point rounding per CTA), one fp32 rounding of each rank's sum, the exchange of W terms, then Mg = W M_r."""
    mut = mut or {}
    W, M, prec = len(runs), runs[0].M, runs[0].prec
    res = {}
    glob = sync_bn and not mut.get("local_stats")
    for L in runs[0].layers:
        sc, co = L["scope"], L["co"]
        Zs = [r.taps["z:" + sc].reshape(-1, co).astype(np.float64) for r in runs]
        for i, r in enumerate(runs):
            group = Zs if glob else [Zs[i]]
            n = len(group)
            Zg = np.concatenate(group)
            Mg = Zg.shape[0]
            mean, var = Zg.mean(0), Zg.var(0)
            A, Q = np.abs(Zg).sum(0), (Zg ** 2).sum(0)
            xg = gamma(n - 1) if n > 1 else 0.0
            q = n * -(-M // 128) * 2.0 ** -21
            d1 = M * E24 * A + q + E24 * sum(np.abs(z.sum(0)) for z in group) + xg * A
            d2 = (M + 1) * E24 * Q + q + xg * Q
            dmean = d1 / Mg + 2 * E24 * np.abs(mean)
            dvar = d2 / Mg + 2 * np.abs(mean) * dmean + dmean ** 2
            var_ema = var * Mg / (Mg - 1)
            mm, mv = r.s.get_variable(sc + "/moving_mean"), r.s.get_variable(sc + "/moving_variance")
            for name, got, ref, b in (("mean " + sc, mm, mean, dmean), ("var " + sc, mv, var_ema, dvar * Mg / (Mg - 1) + 2 * E24 * var_ema)):
                res[name] = max(res.get(name, 0.0), ratio((tag, prec, name), got, ref, b + 1e-30))
    return res


# ------------------------------------------------------------------------------------------------ one data-parallel step
def global_batch(net, C, K, W, B_r, crop, use_mask, ignore, seed):
    """Feeds of the global batch, rank r's share rows [r B_r, (r+1) B_r).  With a mask or the ignore label the ranks' valid
    pixel counts are far apart: rank 0 keeps about 80 % of its pixels, the last rank about 15 %."""
    rs = np.random.RandomState(seed)
    B, P = W * B_r, crop * crop
    x = rs.randn(B, P * C).astype(np.float32)
    y = rs.randint(0, K, size=(B, P)).astype(np.float32)
    keep = np.repeat(np.linspace(0.8, 0.15, W), B_r)[:, None]
    mask = None
    if ignore:
        y = np.where(rs.rand(B, P) < keep, y, K).astype(np.float32)
    if use_mask:
        mask = rs.rand(B, P) < keep
    return x, y, mask


class DPRun:
    """One data-parallel step of W ranks over a global batch (Exchange), its schedule checked, every tap collected."""

    def __init__(self, drs, monkeypatch, net, C, K, prec, W, B_r, crop, sync_bn, use_mask=False, ignore=False, env=(), seed=5):
        import torch
        torch.cuda.init()
        self.W, self.sync_bn, self.tag = W, sync_bn, "%s W%d B%d crop%d%s" % (net, W, B_r, crop, " syncbn" if sync_bn else "")
        x, y, mask = global_batch(net, C, K, W, B_r, crop, use_mask, ignore, seed + 1)
        sl = [slice(r * B_r, (r + 1) * B_r) for r in range(W)]
        self.runs = []
        try:
            for r in range(W):
                self.runs.append(TrainRun(drs, monkeypatch, net, C, K, prec, B_r, crop, ignore=ignore, env=env, seed=seed, x=x[sl[r]],
                                          y=y[sl[r]], mask=None if mask is None else mask[sl[r]], step=False))
            self.ex = Exchange(W)
            for r, run in enumerate(self.runs):
                run.s.set_allreduce(self.ex.fn(r), W, sync_bn)
            step_ranks(self.runs, self.ex)
            for run in self.runs:
                run.collect(W * run.M if sync_bn else None)
            self.state = [{n: run.s.get_variable(n) for n, _ in run.s.variable_names()} for run in self.runs]
            check_schedule(self.runs[0], self.ex.log, W, sync_bn, use_mask or ignore, not os.environ.get("DRS_NO_BUCKETS"), self.tag)
        except BaseException:
            self.close()
            raise

    def close(self):
        for run in self.runs:
            run.close()

    def check(self, idx=None, wcols=None, mut=None):
        """{quantity: largest err / bound}: forward statistics, every backward stage; confusion counts and bit-identity of
        the ranks asserted on the way."""
        runs, tag = self.runs, self.tag
        res = check_stats(runs, self.sync_bn, tag, mut)
        res.update(check_step(runs, tag, idx, wcols, mut, self.sync_bn))
        if mut:
            return res
        # confusion counts: the sum of every rank's bincount of (label, pred) over the counted pixels, exactly
        K = runs[0].K
        ref = np.zeros(K * K, np.int64)
        for r in runs:
            y = r.y.reshape(-1).astype(np.int64)
            ok = (r.mask.reshape(-1) if r.mask is not None else np.ones(y.size, bool)) & (y < K)
            ref += np.bincount(y[ok] * K + r.pred.reshape(-1)[ok], minlength=K * K)
        for r in runs:
            assert np.array_equal(r.cm.reshape(-1).astype(np.int64), ref), (tag, "confusion counts")
            assert r.n_correct == int(np.trace(ref.reshape(K, K))), (tag, "correct pixels")
        # every rank holds the same variables, slots and (SyncBN) moving statistics; without SyncBN those differ
        for name in self.state[0]:
            same = all(np.array_equal(st[name], self.state[0][name]) for st in self.state[1:])
            if "moving_" not in name or self.sync_bn:
                assert same, (tag, "ranks differ after the step in", name)
            elif name.endswith("moving_mean"):
                assert not same, (tag, "every rank has the same batch statistics without SyncBN", name)
        return res


def _dp(drs, monkeypatch, net, C, K, prec, W, B_r, crop, sync_bn, idx_fn=None, wcols=None, **kw):
    d = DPRun(drs, monkeypatch, net, C, K, prec, W, B_r, crop, sync_bn, **kw)
    try:
        res = d.check(idx=idx_fn(d.runs[0]) if idx_fn else None, wcols=wcols)
    finally:
        d.close()
    _assert_within(res, (d.tag, prec))
    return d


# ------------------------------------------------------------------------------------------------ GPU cases
@pytest.mark.gpu
@pytest.mark.parametrize("net,C,K,use_mask", TRAIN_NETS)
def test_data_parallel_layers(drs, monkeypatch, net, C, K, use_mask):
    """W = 2, global B = 4, crop 13: every training net in bf16 and fp32, SyncBN on and off; the masked nets with uneven
    valid counts."""
    t0 = time.time()
    for prec in ("bf16", "fp32"):
        for sync_bn in (True, False):
            _dp(drs, monkeypatch, net, C, K, prec, 2, 2, 13, sync_bn, use_mask=use_mask)
    _print_report(net + " data parallel", time.time() - t0)


@pytest.mark.gpu
@pytest.mark.parametrize("W,B_r", [(3, 2), (4, 2), (4, 1)])
def test_data_parallel_world_sizes(drs, monkeypatch, W, B_r):
    """dilated_grsl bf16 at W = 3 (a global count that is not a power of two) and W = 4, and one patch per rank."""
    t0 = time.time()
    for sync_bn in (True, False):
        _dp(drs, monkeypatch, "dilated_grsl", 4, 6, "bf16", W, B_r, 13, sync_bn)
    _print_report("data parallel W%d B%d" % (W, B_r), time.time() - t0)


@pytest.mark.gpu
def test_data_parallel_ignore_label(drs, monkeypatch):
    """dilated_grsl with the ignore label K: the ranks count their valid pixels and exchange the count; rank 0 keeps about
    80 % of its pixels, rank 1 about 15 %."""
    t0 = time.time()
    for prec in ("bf16", "fp32"):
        for sync_bn in (True, False):
            _dp(drs, monkeypatch, "dilated_grsl", 4, 6, prec, 2, 2, 13, sync_bn, ignore=True)
    _print_report("data parallel ignore label", time.time() - t0)


@pytest.mark.gpu
@pytest.mark.parametrize("net,C,K,use_mask", [n for n in TRAIN_NETS if "grsl" in n[0]])
def test_data_parallel_separate_pool_kernels(drs, monkeypatch, net, C, K, use_mask):
    """The separate pool and BN backward kernels of the bf16 pooling nets (DRS_NO_FUSED_POOL_APPLY=1) under SyncBN."""
    t0 = time.time()
    _dp(drs, monkeypatch, net, C, K, "bf16", 2, 2, 13, True, use_mask=use_mask, env=("DRS_NO_FUSED_POOL_APPLY",))
    _print_report(net + " data parallel unfused pool", time.time() - t0)


@pytest.mark.gpu
def test_data_parallel_full_size(drs, monkeypatch):
    """The product shape: W = 2, B_r = 32, crop 49, dilated_grsl bf16, SyncBN.  dout at sampled pixels, filter gradients on
    the first / last output channel of every 64-wide tile plus random ones, everything else on whole tensors."""
    rs = np.random.RandomState(23)
    t0 = time.time()
    _dp(drs, monkeypatch, "dilated_grsl", 4, 6, "bf16", 2, 32, 49, True, idx_fn=lambda r: sample_pixels(r.B, r.crop, rs),
        wcols=_subset_cols(rs))
    _print_report("data parallel full size", time.time() - t0)


@pytest.mark.gpu
def test_data_parallel_switches_keep_every_bit(drs, monkeypatch):
    """The same step twice, under DRS_NO_BUCKETS=1 (one exchange of the whole buffer, checked by the schedule) and under
    DRS_NO_OVERLAP=1: the variables, slots and moving statistics after it are the same bits.  Either switch only changes
    when the same fp32 sums are made."""
    args = ("dilated_icpr_rate6_SE", 4, 6, "bf16", 2, 2, 13, True)
    states = {}
    for sw in ("", "", "DRS_NO_BUCKETS", "DRS_NO_OVERLAP"):
        with monkeypatch.context() as m:
            d = DPRun(drs, m, *args, ignore=True, env=(sw,) if sw else ())
            d.close()
        assert all(len(lg) == len(d.ex.log[0]) for lg in d.ex.log)
        states.setdefault(sw or "default", []).append(d.state[0])
    base = states["default"][0]
    for sw, sts in states.items():
        for st in sts:
            diff = [n for n in base if not np.array_equal(base[n], st[n])]
            assert not diff, (sw, "changes", diff)


@pytest.mark.gpu
def test_wrong_data_parallel_references_break_the_bounds(drs, monkeypatch):
    """On one SyncBN step with the ignore label and uneven valid counts, each wrong reference exceeds its bound at least
    10x: SyncBN statistics from the rank's own batch, dlogits divided by the rank's own count, the BN-backward sums of one
    rank only, a front-range filter gradient (conv1) missing one rank's share, and the count taken as M_r."""
    t0 = time.time()
    d = DPRun(drs, monkeypatch, "dilated_grsl", 4, 6, "bf16", 2, 2, 13, True, ignore=True)
    try:
        _assert_within(d.check(), "right reference")
        got = {"local statistics": max(v for k, v in d.check(mut={"local_stats": True}).items() if k.startswith(("mean ", "var "))),
               "local count": d.check(mut={"local_count": True})["dlogits"],
               "bn sums of one rank": max(v for k, v in d.check(mut={"bn_sums_one_rank": True}).items() if k.startswith("dz ")),
               "rank share dropped": d.check(mut={"drop_rank_share": "conv1"})["dW conv1"],
               "count is M_r": d.check(mut={"count_is_m": True})["dlogits"]}
    finally:
        d.close()
    REPORT.clear()
    print("wrong data-parallel references, largest err / bound:", got, "%.1f s" % (time.time() - t0))
    assert all(v >= 10.0 for v in got.values()), got


# ------------------------------------------------------------------------------------------------ CPU: the schedule model
def test_schedule_model_covers_the_gradient_buffer():
    """For every training net: the offsets of trainable_offsets add up to the trainable variables of nets.variable_shapes;
    the bucket follows layer L-3's backward reduction and, with the front range, covers [0, n_trainable + K^2 + 2) once;
    without buckets (or with fewer than four layers) one exchange covers it."""
    from drs_b200 import nets
    for net, C, K, _ in TRAIN_NETS:
        layers, cls_inputs, _ = net_layers(net, C)
        shapes = nets.variable_shapes(net, C, K)
        n_tr = sum(int(np.prod(s)) for n, s in shapes.items() if n.endswith(("/weights", "/biases")))
        w_off, total = trainable_offsets(layers, cls_inputs, K)
        assert total == n_tr, net
        for sync_bn in (True, False):
            exp, split_off, total = expected_schedule(layers, cls_inputs, K, 2, sync_bn, True, True)
            stages = [s for s, _ in exp]
            assert stages[:len(layers) * sync_bn + 1] == ["bn forward " + l["scope"] for l in layers] * sync_bn + ["pixel count"]
            if len(layers) < 4:
                assert split_off is None and exp[-1] == ("whole buffer", n_tr + K * K + 2), net
                continue
            i = stages.index("bucket")
            if sync_bn:
                assert stages[i - 1] == "bn backward " + layers[-3]["scope"] and stages[i + 1] == "bn backward " + layers[-4]["scope"], net
            assert exp[i][1] + exp[-1][1] == n_tr + K * K + 2 and exp[-1] == ("front range", split_off), net
            assert split_off == w_off[layers[-3]["scope"]] > 0, net
            one, _, _ = expected_schedule(layers, cls_inputs, K, 2, sync_bn, True, False)
            assert one[-1] == ("whole buffer", n_tr + K * K + 2) and "bucket" not in [s for s, _ in one], net
