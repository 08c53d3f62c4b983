"""GPU backend of the drop-in scripts: executes a host ``BatchPlan`` (host.py) on the device.

The scripts' loops call a backend with these operations; ``GpuBackend`` is the product implementation
(libdrs.so through ``Session``, torch only for device buffers).  Tests drive the same loops with a
closed-form stand-in to pin the host logic against reference-generated traces without a GPU.

    submit_train(plan, loss_mask=None)   -> ticket   gather + normalise + sess.run(train) + confusion, nothing waited for
    train_result(ticket)                 -> (loss, cm[K,K] uint32, n_correct)
    train_on_plan(plan, loss_mask=None)  == train_result(submit_train(...))
    eval_on_plan(plan, scene_offset=0)   -> (pred int64 [B,c,c], labels [B,c,c]) gather + normalise + sess.run(pred_up)
    scene_labels(scene_id, crop, batch, variant) -> uint8 [H,W]   whole sliding-window inference
    scene_multiscale_labels(scene_id, crops, batch, variant) -> uint8 [H,W]   multi-scale evaluation, one pass per crop
    save(path) / restore(path)                                    tf.train.Saver stand-in (one .npz keyed by TF names)
"""
import numpy as np


class GpuBackend:
    def __init__(self, session, scenes, label_maps, mean_full, std_full, device=0, rank=0, world=1, train_fp16_patches=False):
        import torch
        self.train_fp16_patches = train_fp16_patches      # coffee:293
        self.rank, self.world = rank, world
        self.torch = torch
        self.s = session
        self.dev = torch.device("cuda", device)
        self.K = session.num_classes
        self.C = session.channels
        self.shapes = []
        self.has_labels = label_maps is not None
        for i, sc in enumerate(scenes):
            lab = None if label_maps is None else label_maps[i]
            session.upload_scene(i, np.ascontiguousarray(sc), lab)
            self.shapes.append(sc.shape[:2])
        session.set_normalization(mean_full, std_full)
        self._x = self._y = self._pred = self._mask = None
        self._amask_on_dev = False
        self.rotate_on_device = True      # isprs rotation augmentation in the gather kernel (plan_isprs_batch flag)
        self.pinned_plans = True          # plan slots are page-locked (asynchronous uploads, host.PlanSlot)
        import os
        self._dp_debug = os.environ.get("DRS_DP_DEBUG", "0") != "0"
        self._cm = torch.zeros(self.K * self.K + 1, dtype=torch.int32, device=self.dev)
        session.set_stream(torch.cuda.current_stream(self.dev).cuda_stream)

    def _buffers(self, B, crop):
        t = self.torch
        n = B * crop * crop
        if self._x is None or self._x.numel() < n * self.C:
            self._x = t.empty(n * self.C, dtype=t.float32, device=self.dev)
            self._y = t.empty(n, dtype=t.float32, device=self.dev)
            self._pred = t.empty(n, dtype=t.uint8, device=self.dev)
            self._mask = t.empty(n, dtype=t.uint8, device=self.dev)
            self._amask = t.empty(n, dtype=t.uint8, device=self.dev)
        return self._x, self._y, self._pred

    def _rank_rows(self, n):
        """Data parallel: this rank's contiguous share of a global batch (SURVEY.md section 8e)."""
        if self.world <= 1:
            return slice(0, n)
        if n % self.world != 0:
            raise ValueError("data-parallel training needs batch_size %% world_size == 0 (batch %d over %d ranks): the reference's "
                             "batch would otherwise lose its remainder every step" % (n, self.world))
        per = n // self.world
        return slice(self.rank * per, (self.rank + 1) * per)

    def own_rows(self, n):
        sl = self._rank_rows(n)
        return sl.start, sl.stop

    def prepare_training(self, batch_size, crops, isprs=True, loss_mask=None):
        """Before the loop, like TF building its graph (isprs:1652-1693): size every buffer for the largest patch size of the
        interval and capture the step's CUDA graph for each size (nothing executes)."""
        crops = sorted(set(int(c) for c in crops))
        per = batch_size // max(self.world, 1)
        x, y, pred = self._buffers(per, crops[-1])
        self.s.reserve(per, crops[-1], training=True)
        if isinstance(loss_mask, str):
            self.s.set_ignore_label(int(loss_mask.split("!=")[1]))
        if self.world > 1 and not self.s.has_nccl:
            return          # the exchange goes through a host callback: not capturable
        self.s.prepare_training(x, y, per, crops, pred_dev=pred, acc_mask_dev=self._amask if isprs else None)

    def _gather(self, plan, scene_offset=0, shard=False):
        if shard and self.world > 1 and not getattr(plan, "local", False):
            sl = self._rank_rows(plan.inst.shape[0])
            sub = type(plan)()
            for k in plan.__slots__:
                v = getattr(plan, k)
                setattr(sub, k, v[sl] if isinstance(v, np.ndarray) and k not in ("noise",) else v)
            if plan.noise_slot is None and plan.noise is not None:
                sub.noise = plan.noise[sl]               # dense per-patch noise (Python planner)
            elif plan.noise_slot is not None and plan.noise is not None:
                # compact noise (native planner): upload only the blocks of this rank's patches
                own = sub.noise_slot[sub.noise_slot >= 0]
                if own.size:
                    per = plan.crop * plan.crop * self.C
                    s0, s1 = int(own.min()), int(own.max()) + 1
                    sub.noise = plan.noise[s0 * per:s1 * per]
                    sub.noise_slot = np.where(sub.noise_slot >= 0, sub.noise_slot - s0, -1).astype(np.int32)
                else:
                    sub.noise = None
            plan = sub
        self._plan = plan
        B, crop = plan.inst.shape[0], plan.crop
        x, y, pred = self._buffers(B, crop)
        inst = plan.inst
        if scene_offset:
            inst = inst.copy()
            inst[:, 0] += scene_offset
        self._amask_on_dev = False
        if getattr(plan, "noise_slot", None) is not None:
            # natively planned batch: asynchronous uploads from the plan's pinned buffers, rotation on the device
            self.s.gather_plan_dev(plan, x, y, self._amask)
            self._amask_on_dev = True
        elif getattr(plan, "rot", None) is not None:
            # rotation on the device (SURVEY 8f N1): the kernel also writes the accuracy mask
            self.s.gather_rot_dev(inst, plan.flips, crop, x, y, noise=plan.noise, noise_on=plan.noise_on, rot=plan.rot,
                                  rot_on=plan.rot_on, amask_out_dev=self._amask)
            self._amask_on_dev = True
        else:
            self.s.gather_dev(inst, plan.flips, crop, x, y, noise=plan.noise, noise_on=plan.noise_on,
                              over_x=plan.over_x, over_y=plan.over_y, over_on=plan.over_on)
        return x, y, pred, B, crop

    def sync_host_rng(self):
        """Data parallel: same host policy streams on every rank (dist.sync_host_rng); no-op for one process."""
        if self.world > 1:
            from . import dist as ddist
            ddist.sync_host_rng()

    def rank0_first(self, fn):
        """Cache files in the working directory: rank 0 creates them, the others wait and load (dist.rank0_first)."""
        if self.world <= 1:
            return fn()
        from . import dist as ddist
        return ddist.rank0_first(fn)

    def _check_same_plan(self, plan):
        """DRS_DP_DEBUG=1: assert that patch size and batch are identical on every rank before the step is enqueued."""
        import zlib
        from . import dist as ddist
        h = 0 if getattr(plan, "local", False) else \
            zlib.crc32(np.ascontiguousarray(plan.inst).tobytes() + np.ascontiguousarray(plan.flips).tobytes())
        ddist.check_same_plan(int(plan.crop), int(h))

    def submit_train(self, plan, loss_mask=None):
        t = self.torch
        if self.world > 1 and self._dp_debug:
            self._check_same_plan(plan)
        if self.train_fp16_patches:
            self.s.set_gather_fp16(True)
        x, y, pred, B, crop = self._gather(plan, shard=True)
        if self.train_fp16_patches:
            self.s.set_gather_fp16(False)
        sl = slice(0, plan.inst.shape[0]) if getattr(plan, "local", False) else self._rank_rows(plan.inst.shape[0])
        plan = self._plan
        n = B * crop * crop
        mask_dev = None
        if isinstance(loss_mask, str):
            # "label!=K": the session derives the mask on the device from the gathered labels (Session.set_ignore_label)
            self.s.set_ignore_label(int(loss_mask.split("!=")[1]))
        elif loss_mask is not None:
            m = np.ascontiguousarray(loss_mask, dtype=np.uint8).reshape(-1, crop * crop)[sl]
            self._mask[:n].copy_(t.from_numpy(np.ascontiguousarray(m).reshape(-1)))
            mask_dev = self._mask
        amask_dev = self._amask if self._amask_on_dev else None
        if plan.acc_mask is not None:
            self._amask[:n].copy_(t.from_numpy(np.ascontiguousarray(plan.acc_mask, dtype=np.uint8).reshape(-1)))
            amask_dev = self._amask
        return self.s.train_step_async(x, y, B, crop, mask_dev=mask_dev, pred_dev=pred, acc_mask_dev=amask_dev)

    def train_result(self, ticket):
        loss, cm, acc = self.s.train_result(ticket)
        return loss, cm, acc

    def train_on_plan(self, plan, loss_mask=None):
        return self.train_result(self.submit_train(plan, loss_mask))

    def eval_on_plan(self, plan, scene_offset=0):
        x, y, pred, B, crop = self._gather(plan, scene_offset)
        self.s.infer_dev(x, B, crop, None, pred)
        self.s.synchronize()
        n = B * crop * crop
        return (pred[:n].cpu().numpy().astype(np.int64).reshape(B, crop, crop),
                y[:n].cpu().numpy().astype(np.int64).reshape(B, crop, crop))

    def sync_bn_stats(self):
        """Data parallel without SyncBN: every rank has normalised with its own batch statistics, so the moving averages
        differ across ranks.  Average them (one small allreduce) before anything evaluates or saves the model, so that every
        rank -- and every stripe of a sharded scene pass -- uses the same statistics."""
        if self.world <= 1:
            return
        import torch.distributed as dist
        t = self.torch
        names = [n for n, _ in self.s.variable_names() if n.endswith("/moving_mean") or n.endswith("/moving_variance")]
        flat = np.concatenate([self.s.get_variable(n) for n in names]).astype(np.float32)
        buf = t.from_numpy(flat).to(self.dev)
        dist.all_reduce(buf, op=dist.ReduceOp.SUM)
        flat = (buf / self.world).cpu().numpy()
        off = 0
        for n in names:
            cnt = self.s.get_variable(n).size
            self.s.set_variable(n, flat[off:off + cnt])
            off += cnt

    def scene_labels(self, scene_id, crop, batch, variant="isprs"):
        H, W = self.shapes[scene_id]
        if self.world == 1:
            return self.s.scene_infer(scene_id, crop, batch, H, W, variant=variant)
        from . import dist as ddist
        r0, r1 = ddist.stripe_bounds(H, self.world, self.rank)
        if self.s.has_nccl:
            # stripes stay on the device: NCCL send/recv to rank 0, broadcast of the assembled map (every rank prints metrics)
            self.s.scene_infer(scene_id, crop, batch, H, W, variant=variant, row_begin=r0, row_end=r1, keep_on_device=True)
            return self.s.scene_gather_labels(H, W, ddist.stripe_bounds(H, self.world), self.rank, all_ranks=True)
        stripe = self.s.scene_infer(scene_id, crop, batch, H, W, variant=variant, row_begin=r0, row_end=r1)
        return ddist.gather_label_stripes(stripe, H, W, self.rank, self.world, device=self.dev, all_ranks=True)

    def scene_multiscale_labels(self, scene_id, crops, batch, variant="isprs"):
        """Label map of the multi-scale evaluation (isprs:1380-1411) over ``crops`` in order, computed on the device: the
        argmax of the summed softmax of every scale's mean map, bit for bit the host composition.  Striped over the ranks
        like scene_labels."""
        H, W = self.shapes[scene_id]
        crops = [int(c) for c in crops]
        if self.world == 1:
            return self.s.scene_infer_multiscale(scene_id, crops, batch, H, W, variant=variant)
        from . import dist as ddist
        r0, r1 = ddist.stripe_bounds(H, self.world, self.rank)
        if self.s.has_nccl:
            self.s.scene_infer_multiscale(scene_id, crops, batch, H, W, variant=variant, row_begin=r0, row_end=r1,
                                          keep_on_device=True)
            return self.s.scene_gather_labels(H, W, ddist.stripe_bounds(H, self.world), self.rank, all_ranks=True)
        stripe = self.s.scene_infer_multiscale(scene_id, crops, batch, H, W, variant=variant, row_begin=r0, row_end=r1)
        return ddist.gather_label_stripes(stripe, H, W, self.rank, self.world, device=self.dev, all_ranks=True)

    def scene_mean_logits(self, scene_id, crop, batch, variant="isprs"):
        """``prob_im / occur_im`` (float64 [H,W,K]) of one sliding-window pass: the per-scale map of the multi-scale
        evaluation (isprs:1380-1411)."""
        H, W = self.shapes[scene_id]
        if self.world != 1:
            raise NotImplementedError("multi-scale evaluation runs on one rank")
        _, mean = self.s.scene_infer(scene_id, crop, batch, H, W, variant=variant, want_mean=True)
        return mean

    def scene_confusion(self, scene_id, num_classes, ignore_label=None):
        """Confusion counts of the label map scene_labels() just produced against the resident ground truth, on the device
        (isprs:1289-1296).  None when the ground truth is not resident or the map is striped over ranks (host path then)."""
        if not self.has_labels or self.world != 1:
            return None
        cm, _ = self.s.scene_confusion(scene_id, num_classes, ignore_label)
        return cm.astype(np.uint32)

    def save(self, path):
        self.s.save(path)

    def restore(self, path):
        self.s.restore(path)
