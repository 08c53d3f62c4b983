"""``Session`` -- the drop-in for the reference's ``tf.Session`` on the hot path.

The reference's only compute seam is ``sess.run(fetches, feed_dict)`` (SURVEY.md section 8b):

    train : sess.run([optimizer, loss, pred_up], {x, y, crop, keep_prob, is_training=True[, mask]})
            isprs:1750-1752, contest:1083-1086, coffee:1295-1297
    infer : sess.run([pred_up, logits], {x, y, crop, keep_prob=1, is_training=False})
            isprs:1274-1275, contest:929-931, coffee:1058-1059

``Session.train_step`` / ``Session.infer`` take the same NumPy feeds (flattened NHWC ``x``, float class ids
``y``) and return the same fetches (fp32 scalar loss incl. the L2 terms, int64 ``pred_up`` [B,crop,crop],
fp32 ``logits`` [B,crop,crop,K]).  Everything is computed by libdrs.so on the GPU; nothing here falls back
to NumPy or PyTorch.
"""
import ctypes as C

import numpy as np

from . import lib as L
from . import nets


class Session:
    def __init__(self, net_type, channels, num_classes, weight_decay=0.005, lr_initial=0.01, decay_steps=50000,
                 decay_rate=0.5, momentum=0.9, precision="bf16", device=0, isprs_scopes=True, bn_unbiased_ema=True,
                 seed=None, bn_decay=0.999):
        """bn_decay: decay of the BN moving averages (tf.contrib.layers.batch_norm's 0.999 by default); 0 makes the moving
        statistics after a step that step's batch statistics."""
        if net_type not in L.NET_TYPES:
            # same message the reference prints before returning (isprs:1679)
            raise ValueError("Error! Net type not identified: " + str(net_type))
        self._lib = L.load()
        self.net_type, self.channels, self.num_classes = net_type, int(channels), int(num_classes)
        self.precision = precision
        self.isprs_scopes = bool(isprs_scopes)
        cfg = L.Config(L.NET_TYPES[net_type], channels, num_classes, L.PREC[precision], weight_decay, lr_initial,
                       decay_steps, decay_rate, momentum, float(bn_decay), 0.001, int(bool(bn_unbiased_ema)), device,
                       int(self.isprs_scopes))
        self._h = C.c_void_p()
        L.check(self._lib.drs_create(C.byref(self._h), C.byref(cfg)))
        self._cb = None
        self._keep = []
        self.has_nccl = False
        if seed is not None:
            self.init_variables(seed)

    # ---------------------------------------------------------------- life cycle
    def close(self):
        if getattr(self, "_h", None) is not None and self._h:
            self._lib.drs_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def set_stream(self, cuda_stream):
        """Enqueue on this cudaStream_t (0 = the legacy default stream torch uses by default); None = the handle's own stream."""
        v = C.c_void_p(-1) if cuda_stream is None else C.c_void_p(int(cuda_stream))
        L.check(self._lib.drs_set_stream(self._h, v))

    def synchronize(self):
        L.check(self._lib.drs_synchronize(self._h))

    @property
    def launch_count(self):
        return int(self._lib.drs_launch_count(self._h))

    # ---------------------------------------------------------------- variables (tf.train.Saver / init)
    def variable_names(self):
        n = self._lib.drs_num_variables(self._h)
        out = []
        buf = C.create_string_buffer(256)
        cnt = C.c_int64()
        for i in range(n):
            L.check(self._lib.drs_variable_name(self._h, i, buf, 256, C.byref(cnt)))
            out.append((buf.value.decode(), int(cnt.value)))
        return out

    def set_variable(self, name, value):
        a = np.ascontiguousarray(np.asarray(value, dtype=np.float32))
        L.check(self._lib.drs_set_variable(self._h, name.encode(), L.ptr(a), a.size))

    def get_variable(self, name, shape=None):
        cnt = dict(self.variable_names())[name]
        a = np.empty(cnt, dtype=np.float32)
        L.check(self._lib.drs_get_variable(self._h, name.encode(), L.ptr(a), cnt))
        return a.reshape(shape) if shape is not None else a

    def get_gradient(self, name, shape=None):
        cnt = dict(self.variable_names())[name]
        a = np.empty(cnt, dtype=np.float32)
        L.check(self._lib.drs_get_gradient(self._h, name.encode(), L.ptr(a), cnt))
        return a.reshape(shape) if shape is not None else a

    def init_variables(self, seed):
        """sess.run(init) (isprs:1717) with a seeded xavier-uniform draw."""
        self.load_variables(nets.initial_variables(self.net_type, self.channels, self.num_classes, seed,
                                                   self.isprs_scopes))

    def load_variables(self, variables):
        for k, v in variables.items():
            self.set_variable(k, v)

    def variables(self):
        shapes = nets.variable_shapes(self.net_type, self.channels, self.num_classes, self.isprs_scopes)
        out = {}
        for name, cnt in self.variable_names():
            base = name[:-len("/Momentum")] if name.endswith("/Momentum") else name
            out[name] = self.get_variable(name, shapes.get(base))
        return out

    def save(self, path):
        """saver.save(sess, output_path + 'model', global_step=step) (isprs:1798): one uncompressed .npz keyed by the TF
        variable names, written by the library (drs_save: temp file + rename).  Returns the file name."""
        path = str(path)
        if not path.endswith(".npz"):
            path += ".npz"                    # what numpy.savez would have appended
        L.check(self._lib.drs_save(self._h, path.encode()))
        return path

    def restore(self, path):
        """saver.restore(sess, model_path) (isprs:1715): every array of the .npz is validated against the model, then applied
        (drs_load).  Files written by numpy.savez load as well."""
        path = str(path)
        L.check(self._lib.drs_load(self._h, (path if path.endswith(".npz") else path + ".npz").encode()))

    @property
    def global_step(self):
        return int(self.get_variable("global_step")[0])

    # ---------------------------------------------------------------- sess.run
    def infer(self, x, crop, want_logits=True):
        """(pred_up int64 [B,crop,crop], logits fp32 [B,crop,crop,K])  -- isprs:1274-1275."""
        x = np.ascontiguousarray(np.asarray(x, dtype=np.float32))
        B = x.shape[0]
        if x.size != B * crop * crop * self.channels:
            raise ValueError("x has %d elements, expected B*crop*crop*C = %d" % (x.size, B * crop * crop * self.channels))
        pred = np.empty((B, crop, crop), dtype=np.int64)
        logits = np.empty((B, crop, crop, self.num_classes), dtype=np.float32) if want_logits else None
        L.check(self._lib.drs_forward_host(self._h, L.ptr(x), B, crop, L.ptr(logits), L.ptr(pred)))
        return pred, logits

    def train_step(self, x, y, crop, mask=None, want_cm=False, acc_mask=None):
        """(loss fp32, pred_up int64 [B,crop,crop][, cm uint32 [K,K], n_correct])  -- isprs:1750-1752."""
        x = np.ascontiguousarray(np.asarray(x, dtype=np.float32))
        y = np.ascontiguousarray(np.asarray(y, dtype=np.float32))
        B = x.shape[0]
        if x.size != B * crop * crop * self.channels or y.size != B * crop * crop:
            raise ValueError("feed shapes do not match B=%d crop=%d C=%d" % (B, crop, self.channels))
        m = None
        if mask is not None:
            m = np.ascontiguousarray(np.asarray(mask).astype(np.uint8))
        am = None
        if acc_mask is not None:
            am = np.ascontiguousarray(np.asarray(acc_mask).astype(np.uint8))
        pred = np.empty((B, crop, crop), dtype=np.int64)
        K = self.num_classes
        cm = np.zeros(K * K + 1, dtype=np.uint32)
        loss = C.c_float()
        L.check(self._lib.drs_train_step_host(self._h, L.ptr(x), L.ptr(y), L.ptr(m), L.ptr(am), B, crop, C.byref(loss),
                                              L.ptr(pred), L.ptr(cm)))
        if want_cm:
            return np.float32(loss.value), pred, cm[:K * K].reshape(K, K).copy(), int(cm[K * K])
        return np.float32(loss.value), pred

    # device-pointer variants (inputs already resident in HBM; torch tensors or raw addresses)
    def infer_dev(self, x_dev, B, crop, logits_dev=None, pred_dev=None):
        L.check(self._lib.drs_forward_dev(self._h, L.ptr(x_dev), B, crop, L.ptr(logits_dev), L.ptr(pred_dev)))

    def train_step_dev(self, x_dev, y_dev, B, crop, mask_dev=None, pred_dev=None, cm_dev=None, want_loss=True,
                       acc_mask_dev=None):
        loss = C.c_float()
        L.check(self._lib.drs_train_step_dev(self._h, L.ptr(x_dev), L.ptr(y_dev), L.ptr(mask_dev), L.ptr(acc_mask_dev), B, crop,
                                             C.byref(loss) if want_loss else None, L.ptr(pred_dev), L.ptr(cm_dev)))
        return np.float32(loss.value) if want_loss else None

    def train_step_async(self, x_dev, y_dev, B, crop, mask_dev=None, pred_dev=None, acc_mask_dev=None):
        """The train step without a host round trip -> ticket for train_result (at most 8 outstanding)."""
        t = C.c_int64()
        L.check(self._lib.drs_train_step_async(self._h, L.ptr(x_dev), L.ptr(y_dev), L.ptr(mask_dev), L.ptr(acc_mask_dev), B, crop,
                                               L.ptr(pred_dev), C.byref(t)))
        return int(t.value)

    def train_result(self, ticket):
        """(loss fp32, cm uint32 [K,K], n_correct) of the step behind ``ticket``; waits for that step only."""
        K = self.num_classes
        cm = np.empty(K * K + 1, dtype=np.uint32)
        loss = C.c_float()
        L.check(self._lib.drs_train_result(self._h, int(ticket), C.byref(loss), L.ptr(cm)))
        return np.float32(loss.value), cm[:K * K].reshape(K, K).copy(), int(cm[K * K])

    def set_ignore_label(self, label):
        """contest: label 7 = unlabelled pixels, excluded from loss / gradient / confusion (contest:236-239, 886-897)."""
        L.check(self._lib.drs_set_ignore_label(self._h, -1 if label is None else int(label)))

    def reserve(self, B, crop_max, training=True):
        """Allocate the workspace for the largest (batch, patch size) of the run up front."""
        L.check(self._lib.drs_reserve_workspace(self._h, int(B), int(crop_max), int(bool(training))))

    def prepare_training(self, x_dev, y_dev, B, crops, mask_dev=None, pred_dev=None, cm_dev=None, acc_mask_dev=None):
        """Capture the training-step graphs for the given patch sizes up front (nothing executes, no variable changes)."""
        for crop in crops:
            L.check(self._lib.drs_train_prepare(self._h, L.ptr(x_dev), L.ptr(y_dev), L.ptr(mask_dev), L.ptr(acc_mask_dev), B,
                                                int(crop), L.ptr(pred_dev), L.ptr(cm_dev)))

    # ---------------------------------------------------------------- data-parallel hook
    def set_allreduce(self, fn, world_size, sync_bn=False):
        """fn(buf_ptr:int, count:int, stream:int) must sum ``count`` floats at ``buf_ptr`` over ranks in place."""
        if fn is None:
            L.check(self._lib.drs_set_allreduce(self._h, L.ALLREDUCE_FN(0), None, 1, 0))
            self._cb = None
            return

        def _cb(user, buf, count, stream):
            try:
                fn(int(buf), int(count), int(stream or 0))
                return 0
            except Exception as e:  # surfaced as a DrsError by the library
                import traceback
                traceback.print_exc()
                return 1

        self._cb = L.ALLREDUCE_FN(_cb)
        L.check(self._lib.drs_set_allreduce(self._h, self._cb, None, int(world_size), int(bool(sync_bn))))

    def comm_init(self, id128, rank, world, sync_bn=False):
        """In-library NCCL communicator (drs_comm_init); ``id128`` from comm_unique_id() on rank 0, distributed by the host."""
        buf = (C.c_uint8 * 128).from_buffer_copy(bytes(id128))
        L.check(self._lib.drs_comm_init(self._h, buf, int(rank), int(world), int(bool(sync_bn))))
        self.has_nccl = True

    def comm_destroy(self):
        L.check(self._lib.drs_comm_destroy(self._h))

    def scene_gather_labels(self, H, W, row_cuts, rank, all_ranks=False):
        """Label stripes of the last scene_infer -> [H, W] on rank 0 (None elsewhere unless all_ranks), device to device over
        NCCL."""
        cuts = np.ascontiguousarray(np.asarray(row_cuts, dtype=np.int32))
        out = np.empty((H, W), dtype=np.uint8) if (rank == 0 or all_ranks) else None
        L.check(self._lib.drs_scene_gather_labels(self._h, int(H), int(W), L.ptr(cuts), int(bool(all_ranks)), L.ptr(out)))
        return out

    # ---------------------------------------------------------------- scene path
    def upload_scene(self, scene_id, scene, labels=None, row_begin=None, row_end=None):
        """Keep a scene resident in HBM.  With row_begin/row_end only those rows are uploaded (a rank's stripe + halo,
        see dist.stripe_rows_needed); coordinates stay those of the whole scene."""
        if row_begin is not None:
            H, W, Cc = scene.shape
            sub = np.ascontiguousarray(scene[row_begin:row_end])
            dt = L.SCENE_F64 if sub.dtype == np.float64 else L.SCENE_F32
            if sub.dtype not in (np.float64, np.float32):
                raise ValueError("scene dtype must be float64 or float32, got %s" % sub.dtype)
            lab = None if labels is None else np.ascontiguousarray(np.asarray(labels, dtype=np.uint8).reshape(H, W)[row_begin:row_end])
            L.check(self._lib.drs_scene_upload_rows(self._h, scene_id, L.ptr(sub), H, W, Cc, dt, L.ptr(lab), row_begin,
                                                    row_end - row_begin))
            return
        scene = np.ascontiguousarray(scene)
        if scene.dtype == np.float64:
            dt = L.SCENE_F64
        elif scene.dtype == np.float32:
            dt = L.SCENE_F32
        else:
            raise ValueError("scene dtype must be float64 (isprs) or float32 (contest/coffee), got %s" % scene.dtype)
        H, W, Cc = scene.shape
        lab = None if labels is None else np.ascontiguousarray(np.asarray(labels, dtype=np.uint8).reshape(H, W))
        L.check(self._lib.drs_scene_upload(self._h, scene_id, L.ptr(scene), H, W, Cc, dt, L.ptr(lab)))

    def free_scene(self, scene_id):
        L.check(self._lib.drs_scene_free(self._h, scene_id))

    def set_normalization(self, mean_full, std_full):
        m = np.ascontiguousarray(np.asarray(mean_full, dtype=np.float64)[:3])
        s = np.ascontiguousarray(np.asarray(std_full, dtype=np.float64)[:3])
        L.check(self._lib.drs_set_normalization(self._h, L.ptr(m), L.ptr(s)))

    def set_gather_fp16(self, on):
        """coffee: training patches are float16 before normalisation (coffee:293, SURVEY F12)."""
        L.check(self._lib.drs_set_gather_fp16(self._h, int(bool(on))))

    def gather_dev(self, inst, flips, crop, x_out_dev, y_out_dev=None, noise=None, noise_on=None, over_x=None,
                   over_y=None, over_on=None):
        inst = np.ascontiguousarray(np.asarray(inst, dtype=np.int32).reshape(-1, 3))
        B = inst.shape[0]
        f = None if flips is None else np.ascontiguousarray(np.asarray(flips, dtype=np.uint8))
        nz = None if noise is None else np.ascontiguousarray(np.asarray(noise, dtype=np.float64))
        nzo = None if noise_on is None else np.ascontiguousarray(np.asarray(noise_on, dtype=np.uint8))
        ox = None if over_x is None else np.ascontiguousarray(np.asarray(over_x, dtype=np.float64))
        oy = None if over_y is None else np.ascontiguousarray(np.asarray(over_y, dtype=np.uint8))
        oo = None if over_on is None else np.ascontiguousarray(np.asarray(over_on, dtype=np.uint8))
        L.check(self._lib.drs_gather_dev(self._h, L.ptr(inst), L.ptr(f), B, crop, L.ptr(nz), L.ptr(nzo), L.ptr(ox),
                                         L.ptr(oy), L.ptr(oo), L.ptr(x_out_dev), L.ptr(y_out_dev)))

    def gather_rot_dev(self, inst, flips, crop, x_out_dev, y_out_dev=None, noise=None, noise_on=None, rot=None, rot_on=None,
                       amask_out_dev=None):
        """gather_dev with the nearest-neighbour rotation of isprs:287-296 done by the kernel (host.rotate_affine gives
        the per-patch affine map); amask_out_dev receives the accuracy mask (rotate(np.ones) then flip)."""
        inst = np.ascontiguousarray(np.asarray(inst, dtype=np.int32).reshape(-1, 3))
        B = inst.shape[0]
        f = None if flips is None else np.ascontiguousarray(np.asarray(flips, dtype=np.uint8))
        nz = None if noise is None else np.ascontiguousarray(np.asarray(noise, dtype=np.float64))
        nzo = None if noise_on is None else np.ascontiguousarray(np.asarray(noise_on, dtype=np.uint8))
        r = None if rot is None else np.ascontiguousarray(np.asarray(rot, dtype=np.float64).reshape(B, 6))
        ro = None if rot_on is None else np.ascontiguousarray(np.asarray(rot_on, dtype=np.uint8))
        L.check(self._lib.drs_gather_rot_dev(self._h, L.ptr(inst), L.ptr(f), B, crop, L.ptr(nz), L.ptr(nzo), L.ptr(r), L.ptr(ro),
                                             L.ptr(x_out_dev), L.ptr(y_out_dev), L.ptr(amask_out_dev)))

    def gather_plan_dev(self, plan, x_out_dev, y_out_dev=None, amask_out_dev=None):
        """Gather of a natively planned batch (host.NativePlanner): asynchronous uploads from the plan's pinned buffers."""
        B = plan.inst.shape[0]
        nz = plan.noise
        L.check(self._lib.drs_gather_plan_dev(self._h, L.ptr(plan.inst), L.ptr(plan.flips), B, plan.crop, L.ptr(plan.rot_on),
                                              L.ptr(plan.rot), L.ptr(plan.noise_on), L.ptr(plan.noise_slot), L.ptr(nz),
                                              0 if nz is None else int(nz.size), L.ptr(x_out_dev), L.ptr(y_out_dev),
                                              L.ptr(amask_out_dev)))

    def accumulate_argmax(self, logits_dev, positions, crop, H, W, want_mean=False):
        pos = np.ascontiguousarray(np.asarray(positions, dtype=np.int32).reshape(-1, 2))
        K = self.num_classes
        labels = np.empty((H, W), dtype=np.uint8)
        mean = np.empty((H, W, K), dtype=np.float64) if want_mean else None
        L.check(self._lib.drs_accumulate_argmax(self._h, L.ptr(logits_dev), L.ptr(pos), pos.shape[0], crop, K, H, W,
                                                L.ptr(labels), L.ptr(mean)))
        return (labels, mean) if want_mean else labels

    def scene_infer(self, scene_id, crop, batch, H, W, variant="isprs", row_begin=0, row_end=None, want_mean=False,
                    keep_on_device=False):
        """The inner loop of validate_test / test / generate_final_maps (isprs:1249-1284) for one scene (stripe).
        keep_on_device: do not copy the label stripe back (scene_gather_labels / scene_confusion read it on the device)."""
        row_end = H if row_end is None else row_end
        rows = row_end - row_begin
        labels = None if keep_on_device else np.empty((rows, W), dtype=np.uint8)
        mean = np.empty((rows, W, self.num_classes), dtype=np.float64) if want_mean else None
        L.check(self._lib.drs_scene_infer(self._h, scene_id, crop, batch, L.GRID[variant], row_begin, row_end,
                                          L.ptr(labels), L.ptr(mean)))
        return (labels, mean) if want_mean else labels

    def scene_infer_multiscale(self, scene_id, crops, batch, H, W, variant="isprs", row_begin=0, row_end=None, want_sum=False,
                               keep_on_device=False):
        """validate_test_multiscale (isprs:1347-1474) for one scene (stripe): a scene pass per crop, in the order given, each
        mean map softmax-ed with NumPy's float32 arithmetic and added to a float32 sum; the labels are its argmax.
        want_sum: also return the sum ([rows, W, K] float32, ``np.sum(mean_prob, axis=0)``).  keep_on_device: as scene_infer."""
        c = np.ascontiguousarray(np.asarray(crops, dtype=np.int32).reshape(-1))
        row_end = H if row_end is None else row_end
        rows = row_end - row_begin
        labels = None if keep_on_device else np.empty((rows, W), dtype=np.uint8)
        psum = np.empty((rows, W, self.num_classes), dtype=np.float32) if want_sum else None
        L.check(self._lib.drs_scene_infer_multiscale(self._h, scene_id, int(c.size), L.ptr(c), batch, L.GRID[variant], row_begin,
                                                     row_end, L.ptr(labels), L.ptr(psum)))
        return (labels, psum) if want_sum else labels

    def scene_infer_host(self, scene_id, scene, crop, batch, variant="isprs", want_mean=False):
        """scene_infer for a scene that is still a host array (a fresh tile): the upload is streamed just ahead of the
        chunks that read it and overlaps the convolutions.  The scene stays resident as scene_id."""
        scene = np.ascontiguousarray(scene)
        if scene.dtype == np.float64:
            dt = L.SCENE_F64
        elif scene.dtype == np.float32:
            dt = L.SCENE_F32
        else:
            raise ValueError("scene dtype must be float64 (isprs) or float32 (contest/coffee), got %s" % scene.dtype)
        H, W, Cc = scene.shape
        labels = np.empty((H, W), dtype=np.uint8)
        mean = np.empty((H, W, self.num_classes), dtype=np.float64) if want_mean else None
        L.check(self._lib.drs_scene_infer_host(self._h, scene_id, L.ptr(scene), H, W, Cc, dt, crop, batch, L.GRID[variant],
                                               L.ptr(labels), L.ptr(mean)))
        return (labels, mean) if want_mean else labels

    def scene_confusion(self, scene_id, num_classes, ignore_label=-1):
        """K x K confusion counts [truth, pred] of the last scene_infer pass over scene_id against the labels uploaded with
        the scene, computed on the device (isprs:1289-1296); also returns the number of correct pixels."""
        cm = np.zeros(num_classes * num_classes + 1, dtype=np.uint32)
        L.check(self._lib.drs_scene_confusion(self._h, int(scene_id), int(num_classes), -1 if ignore_label is None else int(ignore_label),
                                              L.ptr(cm)))
        return cm[:-1].reshape(num_classes, num_classes).astype(np.int64), int(cm[-1])

    def confusion_dev(self, truth_dev, pred_dev, n, mask_dev=None, ignore_label=-1):
        K = self.num_classes
        cm = np.zeros(K * K + 1, dtype=np.uint32)
        L.check(self._lib.drs_confusion_dev(self._h, L.ptr(truth_dev), L.ptr(pred_dev), L.ptr(mask_dev), n, K,
                                            ignore_label, L.ptr(cm)))
        return cm[:K * K].reshape(K, K).copy(), int(cm[K * K])

    # ---------------------------------------------------------------- profiling / debug
    def set_profiling(self, on=True):
        L.check(self._lib.drs_set_profiling(self._h, int(bool(on))))

    def profile_read(self):
        ms, n, fl = C.c_float(), C.c_int64(), C.c_double()
        L.check(self._lib.drs_profile_read(self._h, C.byref(ms), C.byref(n), C.byref(fl)))
        return float(ms.value), int(n.value), float(fl.value)

    def debug_activation(self, scope, B, crop, co):
        a = np.empty((B, crop, crop, co), dtype=np.float32)
        L.check(self._lib.drs_debug_activation(self._h, scope.encode(), L.ptr(a), a.size))
        return a

    def debug_conv(self, x, w, scale, shift, rate, act=0, precision="f16"):
        x = np.ascontiguousarray(x, dtype=np.float32)
        w = np.ascontiguousarray(w, dtype=np.float32)
        B, crop, _, ci = x.shape
        k, _, _, co = w.shape
        sc = np.ascontiguousarray(scale, dtype=np.float32)
        sh = np.ascontiguousarray(shift, dtype=np.float32)
        y = np.empty((B, crop, crop, co), dtype=np.float32)
        L.check(self._lib.drs_debug_conv(self._h, L.ptr(x), L.ptr(w), L.ptr(sc), L.ptr(sh), B, crop, k, rate, ci, co, act,
                                         L.PREC[precision], L.ptr(y)))
        return y

    def debug_dgrad(self, dy, w, rate, precision="bf16"):
        dy = np.ascontiguousarray(dy, dtype=np.float32)
        w = np.ascontiguousarray(w, dtype=np.float32)
        B, crop, _, co = dy.shape
        k, _, ci, _ = w.shape
        dx = np.empty((B, crop, crop, ci), dtype=np.float32)
        L.check(self._lib.drs_debug_dgrad(self._h, L.ptr(dy), L.ptr(w), B, crop, k, rate, ci, co, L.PREC[precision], L.ptr(dx)))
        return dx

    def debug_layer(self, z, dout, pool, act, precision="bf16"):
        """(out, dz, batch mean, batch inverse std) of one train-mode BN + activation (+ max-pool) layer."""
        z = np.ascontiguousarray(z, dtype=np.float32)
        dout = np.ascontiguousarray(dout, dtype=np.float32)
        B, crop, _, c = z.shape
        out, dz = np.empty_like(z), np.empty_like(z)
        mean, istd = np.empty(c, dtype=np.float32), np.empty(c, dtype=np.float32)
        L.check(self._lib.drs_debug_layer(self._h, L.ptr(z), L.ptr(dout), B, crop, c, int(bool(pool)), int(act), L.PREC[precision],
                                          L.ptr(out), L.ptr(dz), L.ptr(mean), L.ptr(istd)))
        return out, dz, mean, istd

    def debug_multiscale_softmax_add(self, prob, occur, acc=None, want_labels=True):
        """One launch of the multi-scale kernel: (acc + softmax(float32(prob / occur)), first argmax of it or None).
        prob [N, K] float32 score sums, occur [N] visit counts, acc [N, K] float32 or None (the first scale)."""
        p = np.ascontiguousarray(np.asarray(prob, dtype=np.float32))
        o = np.ascontiguousarray(np.asarray(occur, dtype=np.uint32))
        n = o.size
        if p.shape != (n, self.num_classes):
            raise ValueError("prob must be [N, K] = [%d, %d]" % (n, self.num_classes))
        out = np.zeros_like(p) if acc is None else np.array(acc, dtype=np.float32, order="C", copy=True)
        labels = np.empty(n, dtype=np.uint8) if want_labels else None
        L.check(self._lib.drs_debug_multiscale_softmax_add(self._h, L.ptr(p), L.ptr(o), n, int(acc is None), L.ptr(out),
                                                           L.ptr(labels)))
        return out, labels

    def debug_wgrad(self, x, dy, k, rate, precision="bf16"):
        x = np.ascontiguousarray(x, dtype=np.float32)
        dy = np.ascontiguousarray(dy, dtype=np.float32)
        B, crop, _, ci = x.shape
        co = dy.shape[-1]
        dw = np.empty((k, k, ci, co), dtype=np.float32)
        L.check(self._lib.drs_debug_wgrad(self._h, L.ptr(x), L.ptr(dy), B, crop, k, rate, ci, co, L.PREC[precision], L.ptr(dw)))
        return dw


def npz_write(path, arrays):
    """The library's checkpoint container without a session (drs_npz_write): ``arrays`` maps member names to arrays of
    up to four dimensions; stored as float32.  numpy.load reads the result."""
    lib = L.load()
    names = [k.encode() for k in arrays]
    vals = [np.asarray(v, dtype=np.float32, order="C") for v in arrays.values()]
    n = len(names)
    dims = np.zeros((max(n, 1), 4), dtype=np.int64)
    ndim = np.zeros(max(n, 1), dtype=np.int32)
    for i, v in enumerate(vals):
        if v.ndim > 4:
            raise ValueError("at most four dimensions")
        ndim[i] = v.ndim
        dims[i, :v.ndim] = v.shape
    L.check(lib.drs_npz_write(str(path).encode(), n, (C.c_char_p * max(n, 1))(*names),
                              (C.c_void_p * max(n, 1))(*[v.ctypes.data for v in vals]),
                              ndim.ctypes.data_as(C.POINTER(C.c_int32)), dims.ctypes.data_as(C.POINTER(C.c_int64))))


def npz_read(path):
    """Every array of a stored .npz as float32, in archive order (drs_npz_entry / drs_npz_read)."""
    lib = L.load()
    total = C.c_int32()
    L.check(lib.drs_npz_entry(str(path).encode(), -1, None, 0, None, None, None, C.byref(total)))
    out = {}
    buf = C.create_string_buffer(512)
    nd, cnt = C.c_int32(), C.c_int64()
    dims = (C.c_int64 * 4)()
    for i in range(total.value):
        L.check(lib.drs_npz_entry(str(path).encode(), i, buf, 512, C.byref(nd), dims, C.byref(cnt), None))
        a = np.empty(cnt.value, dtype=np.float32)
        L.check(lib.drs_npz_read(str(path).encode(), buf.value, L.ptr(a), cnt.value))
        out[buf.value.decode("utf-8", "replace")] = a.reshape([dims[j] for j in range(nd.value)])
    return out


def np_softmax(values):
    """The multi-scale kernel's per-pixel softmax over the last axis, compiled for the host (drs_debug_np_softmax, no GPU):
    equal bit for bit to ``loops.reference_softmax`` of a float32 array."""
    a = np.ascontiguousarray(np.asarray(values, dtype=np.float32))
    K = a.shape[-1]
    out = np.empty_like(a)
    L.check(L.load().drs_debug_np_softmax(L.ptr(a), a.size // K, K, L.ptr(out)))
    return out


def np_expf(values):
    """The exp of that softmax (NumPy's float32 exp restated), compiled for the host (drs_debug_np_expf, no GPU)."""
    a = np.ascontiguousarray(np.asarray(values, dtype=np.float32))
    out = np.empty_like(a)
    L.check(L.load().drs_debug_np_expf(L.ptr(a), a.size, L.ptr(out)))
    return out


def grid_positions(H, W, crop, batch, variant="isprs"):
    """Visiting order of create_patches_per_map over a whole scene (host code inside libdrs, no GPU)."""
    lib = L.load()
    n = C.c_int64()
    L.check(lib.drs_grid_positions(H, W, crop, batch, L.GRID[variant], None, 0, C.byref(n)))
    pos = np.empty((n.value, 2), dtype=np.int32)
    L.check(lib.drs_grid_positions(H, W, crop, batch, L.GRID[variant], L.ptr(pos), n.value, C.byref(n)))
    return pos
