"""Training / evaluation engine of the unsupervised-homography path on one GPU (one process per GPU).

Owns the flat fp32 parameter / gradient / Adam buffers and the activation workspace, and strings the libudh calls
into the reference's step (code/homography_CNN_synthetic.py:229-278,333-353):
    regressor fwd -> h4p losses -> DLT -> fused warp + photometric reductions -> backward of the selected loss
    -> gradient mean over ranks (one NCCL allreduce of the flat buffer) -> TF-1 Adam with staircase decay.
All arithmetic is in libudh's CUDA kernels; torch provides memory, streams and torch.distributed.
"""
import ctypes
import math
import os
from collections import OrderedDict

import numpy as np
import torch

from . import _lib, ops, params as P
from ._lib import check, lib

LOSS_TYPES = ("h_loss", "rec_loss", "ssim_loss", "l1_loss", "l1_smooth_loss", "ncc_loss")
_PHOTO_BWD = {"l1_loss": _lib.LOSS_L1, "rec_loss": _lib.LOSS_REC, "l1_smooth_loss": _lib.LOSS_L1_SMOOTH, "ncc_loss": _lib.LOSS_NCC,
              "ssim_loss": _lib.LOSS_CUSTOM}
NUMERIC = {"fp32": _lib.NUMERIC_FP32, "bf16": _lib.NUMERIC_BF16, "bf16x3": _lib.NUMERIC_BF16X3}


def decay_steps(lr, min_lr, num_total_steps=150000, decay_rate=0.96):
    """homography_CNN_synthetic.py:161-169."""
    return int((math.log(decay_rate) * num_total_steps) / math.log(min_lr * 1.0 / lr))


def learning_rate(step, lr, min_lr, num_total_steps=150000, decay_rate=0.96):
    """tf.train.exponential_decay(lr, step, decay_steps, 0.96, staircase=True)."""
    return lr * decay_rate ** (step // decay_steps(lr, min_lr, num_total_steps, decay_rate))


def dp_slices(specs):
    """Row G (utils/utils.py:380-403) as two slices of the flat gradient buffer: (head, convs).  `head` = fc1 w/b + fc2 w/b
    (98 % of the bytes, complete after the head phase of the backward, reduced under the conv backward); `convs` = the eight
    conv layers (complete at the end of the backward).  Together they cover the whole buffer exactly once."""
    off = specs["model/fc1/fc1/weights"].offset
    return slice(off, None), slice(0, off)


def dp_shard_range(begin, count, rank, world):
    """Rank `rank`'s contiguous shard [lo, hi) of the float range [begin, begin + count) for the sharded optimiser of the
    multicast path (csrc/dp_update.cu): 4-float aligned (the kernel moves float4), equal sizes except a shorter / empty tail,
    together the shards cover the range exactly once.  Returns (lo, hi, per) with `per` the full shard size."""
    per = -(-count // (4 * world)) * 4
    lo = min(begin + rank * per, begin + count)
    hi = min(lo + per, begin + count)
    return lo, hi, per


def allreduce_two_phase(flat, specs, group=None, between=None):
    """sum-allreduce of the flat gradient in the engine's two phases (head slice first, `between()` — the conv backward in
    the engine — then the conv slice).  Device-agnostic: the gloo CPU test drives exactly this function."""
    head, convs = dp_slices(specs)
    torch.distributed.all_reduce(flat[head], group=group)
    if between is not None:
        between()
    torch.distributed.all_reduce(flat[convs], group=group)
    return flat


class HomographyEngine(object):
    def __init__(self, batch_size, patch_size=128, img_h=240, img_w=320, numeric="fp32", seed=0, device=None,
                 lr=1e-4, min_lr=0.9e-4, loss_type="l1_loss", process_group=None, world_size=1):
        _lib.require_device()
        if loss_type not in LOSS_TYPES:
            raise ValueError("unknown loss_type %r" % (loss_type,))
        self.device = torch.device(device if device is not None else "cuda")
        self.B, self.Pz, self.img_h, self.img_w = int(batch_size), int(patch_size), int(img_h), int(img_w)
        self.numeric = NUMERIC[numeric]
        self.numeric_name = numeric
        self.loss_type = loss_type
        self.lr, self.min_lr = lr, min_lr
        self.specs = P.param_specs(patch_size)
        n = P.total_floats(self.specs)
        assert n == lib.udh_param_total_floats(patch_size), "python / C parameter layouts disagree"
        self.pg = process_group
        self.world_size = world_size
        # N > 1: parameters, gradients and the workspace (it holds fc1's weight mirror) are symmetric-memory allocations bound
        # to an NVSwitch multicast object when the box offers one (_dp_setup_multicast) — plain device memory otherwise
        self._symm = self._dp_want_multicast()
        self.params = self._alloc(n, torch.float32).zero_()
        self.grads = self._alloc(n, torch.float32).zero_()
        self.adam_m = torch.zeros_like(self.params)
        self.adam_v = torch.zeros_like(self.params)
        if seed is not None:
            self.load_flat(P.init_flat(seed, patch_size))
        self.ws_bytes = lib.udh_cnn_workspace_bytes(self.B, self.Pz, self.numeric)
        if self.ws_bytes == 0:
            raise _lib.UdhError("unsupported batch / patch size (%d, %d)" % (self.B, self.Pz))
        self.ws = self._alloc(self.ws_bytes, torch.uint8)
        check(lib.udh_cnn_workspace_init(self._p(self.ws), self.ws_bytes, self.B, self.Pz, self.numeric, ops._stream()),
              "udh_cnn_workspace_init")
        # bf16 mode: Adam refreshes the bf16 copy of fc1's weights in the same pass, the next forward skips its conversion
        mp, mb, mc, st = ctypes.c_void_p(), ctypes.c_size_t(), ctypes.c_size_t(), ctypes.c_int()
        check(lib.udh_cnn_fc1_mirror(self._p(self.ws), self.ws_bytes, self.B, self.Pz, self.numeric, ctypes.byref(mp), ctypes.byref(mb),
                                     ctypes.byref(mc), ctypes.byref(st)), "udh_cnn_fc1_mirror")
        self._mirror = (mp.value, mb.value, mc.value, st.value) if mp.value else None
        self._mirror_current = False
        self._mirror_version = -1          # torch version counter of self.params when the mirror was written
        self.global_step = 0
        self._mv_sharded = False
        self._mc = self._dp_setup_multicast() if self._symm else None
        # second stream: Row G of the fully connected slice under the conv backward
        self._comm_stream = torch.cuda.Stream(device=self.device) if world_size > 1 else None
        # SM policy of this engine's steps (library-global knobs, applied at the start of every step).  A conv CTA with 200+ KB
        # of shared memory shares its SM with nothing, so a second stream's kernel and the persistent conv kernels take turns
        # on an SM rather than overlap:
        #   top: the SMs NCCL's allreduce kernel (NCCL_MAX_CTAS) takes next to conv4_x's backward on the NCCL path — those four
        #     launches have <= 2 items per CTA and lose nothing on 116 CTAs;
        #   marker layer: where in the conv backward the multicast kernel starts (it queues for SMs like any other kernel).
        self._sm_policy = dict(top=int(os.environ.get("NCCL_MAX_CTAS", "32")) if (world_size > 1 and self._mc is None) else 0,
                               marker=3 if self._mc is not None else -1)
        # static per-step outputs of the one-call step (udh_step_forward_backward): reused every step
        B, Pz, dev = self.B, self.Pz, self.device
        self._sb = dict(h4p=torch.zeros(B, 8, device=dev), H=torch.zeros(B, 3, 3, device=dev), pred=torch.zeros(B, Pz, Pz, 1, device=dev),
                        dh4p=torch.zeros(B, 8, device=dev), dH=torch.zeros(B, 3, 3, device=dev), scratch=torch.zeros(B * 9, device=dev),
                        sums=torch.zeros(_lib.NSUMS, device=dev, dtype=torch.float64), photo=torch.zeros(_lib.NLOSSES, device=dev),
                        metrics=torch.zeros(_lib.NMETRICS, device=dev), per=torch.zeros(B, device=dev))
        self._args = _lib.StepArgs()
        # dropout masks are keep_bit(seed + global_step, salt, LOCAL element index): every data-parallel rank needs its own
        # stream (the reference's towers draw independent masks), parameter init stays rank-independent
        rank = torch.distributed.get_rank(process_group) if world_size > 1 else 0
        self.rank = rank
        self.dropout_seed = (0x5EED0000 + (seed or 0) + rank * 0x9E3779B97F4A7C15) & 0xFFFFFFFFFFFFFFFF

    # ------------------------------------------------------------------ parameters
    def _mirror_is_current(self):
        """The bf16 copy of fc1's weights (written by udh_adam_step_mirror) still matches self.params: libudh's kernels
        write through raw pointers and leave torch's version counter alone, any torch in-place write to self.params
        (copy_, add_, optimizers, checkpoint loads) bumps it and so invalidates the mirror without further bookkeeping."""
        return self._mirror_current and self.params._version == self._mirror_version

    def load_flat(self, flat_np):
        self.params.copy_(torch.as_tensor(flat_np, dtype=torch.float32))
        self._mirror_current = False          # any write to self.params outside update() must clear this

    def named_parameters(self):
        return P.unflatten(self.params, self.specs)

    def named_gradients(self):
        return P.unflatten(self.grads, self.specs)

    def export_named(self, path):
        """Parameters under the reference's TF-Slim variable names / shapes (+ global_step)."""
        import numpy as np
        P.save_named_npz(path, self.params.cpu().numpy(), extra={"global_step": np.array(self.global_step)}, patch_size=self.Pz)

    def import_named(self, path):
        self.load_flat(P.load_named_npz(path, self.Pz))

    def save_tf_checkpoint(self, prefix, with_optimizer=True):
        """TensorFlow checkpoint V2 bundle (<prefix>.index / .data-00000-of-00001) with the reference graph's variable names,
        Adam slots and global_step — what tf.train.Saver writes at code/homography_CNN_synthetic.py:360 (tf_checkpoint.py)."""
        from . import tf_checkpoint as tfc
        tfc.write_checkpoint(prefix, self.snapshot_tf_variables(with_optimizer))

    def snapshot_tf_variables(self, with_optimizer=True):
        """Host copy of the state as the name -> array table tf_checkpoint.write_checkpoint takes (the D2H copies happen here;
        the table can then be written by another thread while training goes on)."""
        from . import tf_checkpoint as tfc
        m = self.adam_m.cpu().numpy() if with_optimizer else None
        v = self.adam_v.cpu().numpy() if with_optimizer else None
        return tfc.engine_state_to_variables(self.params.cpu().numpy(), m, v, self.global_step, self.specs)

    def load_tf_checkpoint(self, prefix, reset_step=False):
        """Restore from a TensorFlow checkpoint V2 bundle (e.g. the reference's published models): parameters, and Adam slots /
        global_step when present (train_saver.restore, code/homography_CNN_synthetic.py:314-317)."""
        from . import tf_checkpoint as tfc
        flat, m, v, step = tfc.variables_to_engine_state(tfc.read_checkpoint(prefix), self.specs, self.params.numel())
        self.load_flat(flat)
        if m is not None:
            self.adam_m.copy_(torch.as_tensor(m)); self.adam_v.copy_(torch.as_tensor(v))
        if step is not None and not reset_step:
            self.global_step = step
        elif reset_step:
            self.global_step = 0

    def state_dict(self):
        return OrderedDict(params=self.params.cpu(), adam_m=self.adam_m.cpu(), adam_v=self.adam_v.cpu(),
                           global_step=self.global_step, patch_size=self.Pz)

    def load_state_dict(self, sd, reset_step=False):
        self.params.copy_(sd["params"]); self.adam_m.copy_(sd["adam_m"]); self.adam_v.copy_(sd["adam_v"])
        self.global_step = 0 if reset_step else int(sd["global_step"])
        self._mirror_current = False

    # ------------------------------------------------------------------ forward
    def _p(self, t):
        return ctypes.c_void_p(t.data_ptr()) if t is not None else None

    def forward(self, batch, train=False, want_pred=True, dropout_seed=None):
        """batch: dict of CUDA tensors — I1_aug, I2_aug [B,P,P,1]; I_aug [B,Hh,W,C]; pts1 [B,8]; gt [B,8] or None;
        patch_indices [B,P*P] int32.  Returns dict with the reference model's result attributes
        (pred_h4p, H_mat, pred_I2, the six losses; test metrics when gt is given)."""
        B, Pz = self.B, self.Pz
        I1, I2 = batch["I1_aug"], batch["I2_aug"]
        assert I1.shape[0] == B and I1.shape[1] == Pz, "batch shape does not match the engine"
        st = ops._stream()
        out = OrderedDict()
        h4p = torch.empty(B, 8, device=self.device, dtype=torch.float32)
        seed = (self.dropout_seed + self.global_step) & 0xFFFFFFFFFFFFFFFF if dropout_seed is None else dropout_seed
        check(lib.udh_cnn_fwd(self._p(self.params), self._p(I1), self._p(I2), self._p(h4p), self._p(self.ws), self.ws_bytes,
                              B, Pz, int(train), seed, self.numeric, st), "udh_cnn_fwd")
        out["pred_h4p"] = h4p
        gt = batch.get("gt")
        if gt is not None:
            metrics, per, dpred = ops.h4p_loss(h4p, gt, want_grad=train and self.loss_type == "h_loss", want_per_sample=not train)
            out["h4p_metrics"], out["batch_h_loss"], out["_dpred"] = metrics, per, dpred
        H = ops.dlt_forward(batch["pts1"], h4p)
        out["H_mat"] = H
        pred, sums = ops.warp_loss_forward(batch["I_aug"], H, I2, batch.get("patch_indices"), Pz, Pz, want_pred=True)
        out["pred_I2"] = pred
        out["_sums"] = sums
        out["photo_losses"] = ops.photo_losses(pred, I2, sums, Pz, Pz, B)
        return out

    @staticmethod
    def losses_dict(out):
        """Host-side view (one D2H sync) named like the reference's attributes."""
        pl = out["photo_losses"].tolist()
        d = OrderedDict(rec_loss=pl[_lib.L_REC], ssim_loss=pl[_lib.L_SSIM], l1_loss=pl[_lib.L_L1],
                        l1_smooth_loss=pl[_lib.L_L1_SMOOTH], ncc_loss=pl[_lib.L_NCC])
        if "h4p_metrics" in out:
            m = out["h4p_metrics"].tolist()
            d.update(h_loss=m[_lib.M_H_LOSS], bounded_h_loss=m[_lib.M_BOUNDED_H_LOSS], num_fail=m[_lib.M_NUM_FAIL],
                     ace=m[_lib.M_ACE])
        return d

    # ------------------------------------------------------------------ backward + update
    def backward(self, batch, out):
        """Gradient of the selected loss into self.grads (which must be zero on entry)."""
        self._apply_sm_policy()
        lt = self.loss_type
        if lt == "h_loss":
            dpred = out["_dpred"]
            if dpred is None:
                raise _lib.UdhError("h_loss needs gt")
        elif lt in _PHOTO_BWD:
            dpm = ops.ssim_backward(out["pred_I2"], batch["I2_aug"], self.Pz, self.Pz) if lt == "ssim_loss" else None
            dH = ops.warp_loss_backward(batch["I_aug"], out["H_mat"], batch["I2_aug"], batch.get("patch_indices"), self.Pz,
                                        self.Pz, _PHOTO_BWD[lt], out["_sums"], 1.0, dpred=dpm)
            dpred = ops.dlt_backward(batch["pts1"], out["pred_h4p"], out["H_mat"], dH)
        else:
            raise _lib.UdhError("unknown loss_type %s" % lt)
        out["_dh4p"] = dpred
        args = (self._p(self.params), self._p(batch["I1_aug"]), self._p(batch["I2_aug"]), self._p(dpred), self._p(self.grads),
                self._p(self.ws), self.ws_bytes, self.B, self.Pz, 1, self.numeric)
        if self.world_size == 1:
            check(lib.udh_cnn_bwd(*args, ops._stream()), "udh_cnn_bwd")
            return
        # Row G with overlap: the fully connected gradients (fc1 = 134 of the 137 MB) are complete after the head phase;
        # their allreduce runs on the communication stream underneath the convolution backward.
        cur = torch.cuda.current_stream()
        check(lib.udh_cnn_bwd_phase(*args, _lib.BWD_HEAD, ops._stream()), "udh_cnn_bwd_phase(head)")
        head, _ = dp_slices(self.specs)
        self._comm_stream.wait_stream(cur)
        with torch.cuda.stream(self._comm_stream):
            torch.distributed.all_reduce(self.grads[head], group=self.pg)                 # fc1 w, fc1 b, fc2 w, fc2 b
        check(lib.udh_cnn_bwd_phase(*args, _lib.BWD_CONVS, ops._stream()), "udh_cnn_bwd_phase(convs)")
        self._head_reduced = True

    def allreduce_grads(self):
        """Row G: utils/utils.py:380-403 get_average_grads == allreduce(sum) here, 1/N folded into Adam."""
        if self.world_size > 1:
            if getattr(self, "_head_reduced", False):
                _, convs = dp_slices(self.specs)
                torch.distributed.all_reduce(self.grads[convs], group=self.pg)            # the 8 conv layers (2.5 MB)
                torch.cuda.current_stream().wait_stream(self._comm_stream)
                self._head_reduced = False
            else:
                torch.distributed.all_reduce(self.grads, group=self.pg)

    # ------------------------------------------------------------------ Row G over NVSwitch multicast memory
    def _dp_want_multicast(self):
        """UDH_DP_MODE = nccl (default) | multicast.  `multicast` selects the fused switch-reduce / sharded-Adam / weight-multicast
        kernel (csrc/dp_update.cu) for fc1's weights; it is parity-tested but measured no faster than the NCCL path on B200
        (DESIGN.md section 6), hence opt-in."""
        mode = os.environ.get("UDH_DP_MODE", "nccl")
        if mode not in ("nccl", "multicast"):
            raise ValueError("UDH_DP_MODE must be nccl or multicast")
        if self.world_size <= 1 or mode == "nccl" or self.pg is None:
            return None
        import torch.distributed._symmetric_memory as symm
        return symm

    def _alloc(self, n, dtype):
        if self._symm is not None:
            return self._symm.empty(int(n), dtype=dtype, device=self.device)
        return torch.empty(int(n), device=self.device, dtype=dtype)

    def _dp_setup_multicast(self):
        """Rendezvous of the three symmetric buffers (collective, same order on every rank).  Returns the multicast addresses
        and this rank's shard of fc1's weights; fails loudly when the fabric has no multicast support."""
        symm = self._symm
        name = self.pg.group_name
        hp, hg, hw = (symm.rendezvous(t, group=name) for t in (self.params, self.grads, self.ws))
        mcs = [int(getattr(h, "multicast_ptr", 0) or 0) for h in (hp, hg, hw)]
        if not all(mcs):
            raise _lib.UdhError("UDH_DP_MODE=multicast: no NVSwitch multicast address for the symmetric buffers")
        w = self.specs["model/fc1/fc1/weights"]
        begin, count = w.offset, int(np.prod(w.shape))
        if self._mirror is not None:
            mp, mb, mc, stored = self._mirror
            assert (mb, mc) == (begin, count) and stored, "the sharded update assumes fc1's weight gradient is stored"
        rank, N = hp.rank, hp.world_size
        lo, hi, per = dp_shard_range(begin, count, rank, N)
        return dict(hp=hp, hg=hg, hw=hw, mc_params=mcs[0], mc_grads=mcs[1], mc_ws=mcs[2], begin=begin, count=count, shard=(lo, hi),
                    per=per, rank=rank, N=N)

    def _dp_sharded_update(self, alpha):
        """fc1's weights: udh_dp_shard_update (switch-side gradient sum, Adam on this rank's shard, new weights and limbs
        multicast to all replicas) -> barrier, on the current (communication) stream; the caller has enqueued the barrier that
        orders every rank's fc gradients before it."""
        mc = self._mc
        lo, hi = mc["shard"]
        mirror, limbs, mb, mcount = None, 0, 0, 0
        if self._mirror is not None:
            mp, mb, mcount, _ = self._mirror
            mirror = ctypes.c_void_p(mc["mc_ws"] + (mp - self.ws.data_ptr()))
            limbs = 2 if self.numeric == _lib.NUMERIC_BF16X3 else 1
        check(lib.udh_dp_shard_update(ctypes.c_void_p(mc["mc_grads"]), self._p(self.params), ctypes.c_void_p(mc["mc_params"]),
                                      self._p(self.adam_m), self._p(self.adam_v), mirror, lo, hi - lo, mb, mcount, limbs, alpha, 0.9, 0.999,
                                      1e-8, 1.0 / self.world_size, 0, ops._stream()), "udh_dp_shard_update")     # grid 0: the default
        mc["hg"].barrier(channel=1, timeout_ms=30000)                    # every owner's stores have landed in every replica
        self._mv_sharded = True

    def sync_optimizer_state(self):
        """COLLECTIVE (all ranks).  With the sharded update each rank holds Adam's m, v of fc1's weights for its own shard only;
        this gathers them so that every rank's adam_m / adam_v is complete (call it before a rank saves a checkpoint)."""
        if self._mc is None or not self._mv_sharded:
            return
        mc = self._mc
        for r in range(mc["N"]):
            lo, hi, _ = dp_shard_range(mc["begin"], mc["count"], r, mc["N"])
            if hi > lo:
                torch.distributed.broadcast(self.adam_m[lo:hi], group=self.pg, group_src=r)
                torch.distributed.broadcast(self.adam_v[lo:hi], group=self.pg, group_src=r)
        self._mv_sharded = False

    def _apply_sm_policy(self):
        pol = self._sm_policy
        check(lib.udh_set_sm_reserve_top(pol["top"]), "udh_set_sm_reserve_top")
        check(lib.udh_set_bwd_marker(pol["marker"]), "udh_set_bwd_marker")

    def _adam(self, lo, hi, alpha):
        """TF-1 Adam on the float range [lo, hi) of the flat buffers (4-float aligned), on the current stream; refreshes the
        part of fc1's tensor-core weight mirror that falls inside the range."""
        n = hi - lo
        off = lo * 4
        pp = lambda t: ctypes.c_void_p(t.data_ptr() + off)
        if self._mirror is not None:
            mp, mb, mc, stored = self._mirror
            limbs = 2 if self.numeric == _lib.NUMERIC_BF16X3 else 1
            inside = lo <= mb and mb + mc <= hi
            if not inside and not (mb + mc <= lo or hi <= mb):
                raise _lib.UdhError("Adam range splits the fc1 mirror")
            check(lib.udh_adam_step_mirror_ex(pp(self.params), pp(self.grads), pp(self.adam_m), pp(self.adam_v), n, alpha, 0.9, 0.999,
                                              1e-8, 1.0 / self.world_size, 1, ctypes.c_void_p(mp if inside else None),
                                              (mb - lo) if inside else 0, mc if inside else 0, stored, limbs, ops._stream()),
                  "udh_adam_step_mirror_ex")
        else:
            check(lib.udh_adam_step(pp(self.params), pp(self.grads), pp(self.adam_m), pp(self.adam_v), n, alpha, 0.9, 0.999, 1e-8,
                                    1.0 / self.world_size, 1, ops._stream()), "udh_adam_step")

    def _alpha(self):
        t = self.global_step + 1
        lr_t = learning_rate(self.global_step, self.lr, self.min_lr)
        return lr_t, lr_t * math.sqrt(1.0 - 0.999 ** t) / (1.0 - 0.9 ** t)

    def update(self):
        self.sync_optimizer_state()          # no-op unless sharded steps (train_step on the multicast path) came before
        lr_t, alpha = self._alpha()
        self._adam(0, self.params.numel(), alpha)
        if self._mirror is not None:
            self._mirror_current = True
            self._mirror_version = self.params._version
        self.global_step += 1
        return lr_t

    def _fill_args(self, batch, train):
        a, sb = self._args, self._sb
        I_aug = batch["I_aug"]
        a.B, a.P, a.img_h, a.img_w, a.C = self.B, self.Pz, I_aug.shape[1], I_aug.shape[2], I_aug.shape[3]
        a.numeric_mode, a.train = self.numeric, int(train)
        a.fwd_flags = _lib.FWD_FC1_MIRROR_CURRENT if self._mirror_is_current() else 0
        a.loss_type = _lib.STEP_LOSS.get(self.loss_type, -1)
        a.seed = (self.dropout_seed + self.global_step) & 0xFFFFFFFFFFFFFFFF
        dp = lambda t: t.data_ptr() if t is not None else None
        a.params, a.grads, a.ws, a.ws_bytes = dp(self.params), dp(self.grads), dp(self.ws), self.ws_bytes
        a.I1, a.I2, a.I_aug, a.pts1, a.gt = dp(batch["I1_aug"]), dp(batch["I2_aug"]), dp(I_aug), dp(batch["pts1"]), dp(batch.get("gt"))
        pi = batch.get("patch_indices")
        a.patch_indices = dp(pi)
        a.idx_stride = 0 if pi is None else (pi.stride(0) if pi.dim() > 1 else 1)
        a.h4p, a.H, a.pred_I2 = dp(sb["h4p"]), dp(sb["H"]), dp(sb["pred"])
        a.dh4p, a.dH, a.scratch, a.sums = dp(sb["dh4p"]), dp(sb["dH"]), dp(sb["scratch"]), dp(sb["sums"])
        if self.loss_type == "ssim_loss" and "dpm" not in sb:
            sb["dpm"] = torch.zeros(self.B, self.Pz, self.Pz, device=self.device)
        a.dpred_map = dp(sb.get("dpm"))
        a.photo_losses, a.h4p_metrics, a.per_sample = dp(sb["photo"]), dp(sb["metrics"]), dp(sb["per"])
        return a

    def _step_out(self, batch):
        sb = self._sb
        out = OrderedDict(pred_h4p=sb["h4p"], H_mat=sb["H"], pred_I2=sb["pred"], photo_losses=sb["photo"], _sums=sb["sums"])
        if batch.get("gt") is not None:
            out["h4p_metrics"], out["batch_h_loss"] = sb["metrics"], sb["per"]
        return out

    def train_step(self, batch):
        """One optimiser step.  The whole forward/backward is ONE C call (udh_step_forward_backward); result tensors are
        the engine's static buffers (valid until the next step)."""
        a = self._fill_args(batch, True)
        st = ops._stream()
        self._apply_sm_policy()
        if self.world_size == 1:
            check(lib.udh_step_forward_backward(ctypes.byref(a), _lib.STEP_ALL, st), "udh_step_forward_backward")
            out = self._step_out(batch)
            out["lr"] = self.update()
            return out
        # The fully connected gradients (fc1 = 134 of the 137 MB) are final after the head phase of the backward: Row G for them
        # runs on a second stream underneath the conv backward.
        cur = torch.cuda.current_stream()
        side = self._comm_stream
        lr_t, alpha = self._alpha()
        head, convs = dp_slices(self.specs)
        n = self.params.numel()
        check(lib.udh_step_forward_backward(ctypes.byref(a), _lib.STEP_FWD_HEAD, st), "udh_step_forward_backward(head)")
        side.wait_stream(cur)
        if self._mc is not None:
            # multicast path: fc1's weights (98 % of the bytes) are reduced, updated and redistributed by ONE kernel over
            # NVSwitch multicast memory (csrc/dp_update.cu); the rest (conv layers, biases, fc2: 2.6 MB) goes through NCCL.
            # The kernel starts at the backward marker (udh_set_bwd_marker): under the wide layers' backward, not conv4_x's.
            w0, w1 = self._mc["begin"], self._mc["begin"] + self._mc["count"]
            with torch.cuda.stream(side):
                torch.distributed.all_reduce(self.grads[w1:], group=self.pg)     # fc1 bias, fc2: final after the head phase too
                self._adam(w1, n, alpha)
                self._mc["hg"].barrier(channel=0, timeout_ms=30000)      # every rank's fc gradients are final (and its fc1 reads done)
            check(lib.udh_step_forward_backward(ctypes.byref(a), _lib.STEP_CONVS, st), "udh_step_forward_backward(convs)")
            with torch.cuda.stream(side):
                check(lib.udh_bwd_marker_wait(ops._stream()), "udh_bwd_marker_wait")
                self._dp_sharded_update(alpha)
            torch.distributed.all_reduce(self.grads[:w0], group=self.pg)
            self._adam(0, w0, alpha)
        else:
            with torch.cuda.stream(side):
                torch.distributed.all_reduce(self.grads[head], group=self.pg)
            check(lib.udh_step_forward_backward(ctypes.byref(a), _lib.STEP_CONVS, st), "udh_step_forward_backward(convs)")
            torch.distributed.all_reduce(self.grads[convs], group=self.pg)
        cur.wait_stream(side)
        if self._mc is None:
            self._adam(0, n, alpha)
        if self._mirror is not None:
            self._mirror_current = True
            self._mirror_version = self.params._version
        self.global_step += 1
        out = self._step_out(batch)
        out["lr"] = lr_t
        return out

    def eval_step(self, batch):
        """Forward + all losses / test metrics in one C call (static result buffers)."""
        a = self._fill_args(batch, False)
        check(lib.udh_step_forward_backward(ctypes.byref(a), _lib.STEP_FWD_ONLY, ops._stream()), "udh_step_forward_backward(eval)")
        return self._step_out(batch)

    # ------------------------------------------------------------------ test helpers
    def dropout_masks(self):
        m1, m2 = ctypes.c_void_p(), ctypes.c_void_p()
        check(lib.udh_cnn_dropout_masks(self._p(self.ws), self.ws_bytes, self.B, self.Pz, self.numeric, ctypes.byref(m1),
                                        ctypes.byref(m2)), "udh_cnn_dropout_masks")
        base = self.ws.data_ptr()
        s = self.Pz // 8
        n1, n2 = self.B * s * s * 128, self.B * 1024
        a = self.ws[m1.value - base: m1.value - base + n1].reshape(self.B, s, s, 128)
        b = self.ws[m2.value - base: m2.value - base + n2].reshape(self.B, 1024)
        return a, b

    def materialize_activations(self):
        """bf16x3 mode keeps activations as 16-bit limb streams; this writes their fp32 values (hi + lo) into the fp32 slots
        activation() reads.  Returns the size of the leading workspace region whose layout all numeric modes share."""
        n = ctypes.c_size_t()
        check(lib.udh_debug_x3_materialize(self._p(self.ws), self.ws_bytes, self.B, self.Pz, ctypes.byref(n), ops._stream()),
              "udh_debug_x3_materialize")
        return n.value

    def activation(self, layer):
        if self.numeric == _lib.NUMERIC_BF16X3 and layer < 11:
            self.materialize_activations()
        ptr, numel = ctypes.c_void_p(), ctypes.c_size_t()
        check(lib.udh_cnn_activation(self._p(self.ws), self.ws_bytes, self.B, self.Pz, self.numeric, layer, ctypes.byref(ptr),
                                     ctypes.byref(numel)), "udh_cnn_activation")
        off = ptr.value - self.ws.data_ptr()
        return self.ws[off: off + numel.value * 4].view(torch.float32)
