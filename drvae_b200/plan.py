"""Python handle on a C-ABI plan (include/drvae_b200.h): owns the torch tensors the kernels
borrow (parameters, Adam moments, gradients) and marshals batches / hyper-parameters.

PyTorch is used for device memory and streams only; every computation of the step happens in
the shared library.  CUDA-only: there is no CPU fallback.
"""
import ctypes
import math
import os
from collections import OrderedDict

import torch

from . import _lib
from ._lib import Arch, Batch, EpsLayout, HParams, InferOut, KIND, Noise

LOSS_KEYS = ("RECL", "KLD", "PERT", "YL", "MMD", "ELBO", "CMPL")


class _CudaView:
    def __init__(self, ptr, shape, typestr):
        self.__cuda_array_interface__ = {"shape": tuple(shape), "typestr": typestr, "data": (ptr, False), "version": 2}


def _ptr(t):
    return ctypes.c_void_p(t.data_ptr()) if t is not None else None


def anneal_coef(iter_num, iter_max=1000, iter_offset=0):
    """DGMMixin._compute_anneal_coef (reference src/DGMMixin.py:77-89), 'linear' only."""
    if iter_num - iter_offset > 0:
        return min(1., 0.01 + (iter_num - iter_offset) / (1. * iter_max))
    return 0.01


class Plan:
    def __init__(self, kind, dim_x, dim_y, dim_z1, dim_z3, enc_z1, dec_x, enc_z3=(), dec_z1=(), L=1, max_batch=200,
                 n_models=1, weight_norm=False, device=None, clf_hidden=()):
        """clf_hidden: widths of the classifier's hidden ELU layers (dim_h_clf, --class-y), DrVAE / VFAE only."""
        if not torch.cuda.is_available():
            raise RuntimeError("drvae_b200 needs a CUDA device (sm_100a); there is no CPU fallback")
        self.lib = _lib.load()
        self.kind = kind
        self.device = torch.device(device if device is not None else "cuda:%d" % torch.cuda.current_device())
        self.E = int(n_models)
        a = Arch()
        a.kind = KIND[kind]
        a.dim_x, a.dim_y, a.dim_z1, a.dim_z3 = int(dim_x), int(dim_y), int(dim_z1), int(dim_z3)
        for name, lst in (("enc_z1", enc_z1), ("dec_x", dec_x), ("enc_z3", enc_z3), ("dec_z1", dec_z1)):
            lst = [int(h) for h in lst]
            if len(lst) > _lib.MAX_HIDDEN:
                raise ValueError("at most %d hidden layers per block are supported" % _lib.MAX_HIDDEN)
            setattr(a, "n_" + name, len(lst))
            arr = getattr(a, name)
            for i, h in enumerate(lst):
                arr[i] = h
        clf_hidden = [int(h) for h in clf_hidden]
        if len(clf_hidden) > _lib.MAX_HIDDEN:
            raise ValueError("at most %d classifier hidden layers are supported" % _lib.MAX_HIDDEN)
        self.clf_hidden = tuple(clf_hidden)
        a.weight_norm = int(bool(weight_norm))
        a.L = int(L)
        a.max_batch = int(max_batch)
        self.arch = a
        self.L, self.Ncap = int(L), int(max_batch)
        self.dim_x, self.dim_y, self.dim_z1, self.dim_z3 = a.dim_x, a.dim_y, a.dim_z1, a.dim_z3
        h = ctypes.c_void_p()
        with torch.cuda.device(self.device):
            widths = (ctypes.c_int * max(1, len(clf_hidden)))(*clf_hidden)
            _lib.check(self.lib.drvae_plan_create_clf(ctypes.byref(a), len(clf_hidden), widths, self.E, ctypes.byref(h)),
                       "plan_create")
        self.h = h
        self.P = int(self.lib.drvae_plan_param_count(h))
        self.tensors = []
        nm = ctypes.create_string_buffer(256)
        for i in range(self.lib.drvae_plan_num_tensors(h)):
            r, c, off = ctypes.c_int(), ctypes.c_int(), ctypes.c_longlong()
            _lib.check(self.lib.drvae_plan_tensor_info(h, i, nm, 256, ctypes.byref(r), ctypes.byref(c), ctypes.byref(off)))
            self.tensors.append((nm.value.decode(), r.value, c.value, off.value))
        # floats between matrix rows (cols rounded up to 4: 16-byte aligned rows, see include/drvae_b200.h)
        self.tensor_ld = [int(self.lib.drvae_plan_tensor_ld(h, i)) for i in range(len(self.tensors))]
        el = EpsLayout()
        _lib.check(self.lib.drvae_plan_eps_layout(h, ctypes.byref(el)))
        self.eps_layout = el
        kw = dict(dtype=torch.float32, device=self.device)
        self.params = torch.zeros(self.E, self.P, **kw)
        self.adam_m = torch.zeros(self.E, self.P, **kw)
        self.adam_v = torch.zeros(self.E, self.P, **kw)
        self.grads = torch.zeros(self.E, self.P, **kw)
        self.losses = torch.zeros(self.E, 8, **kw)
        # CUDA graphs cannot be captured on the legacy default stream: calls made while torch's current stream is
        # the default one run on this stream instead, ordered after / before the caller's stream with events
        self._own_stream = torch.cuda.Stream(device=self.device)
        _lib.check(self.lib.drvae_plan_bind(h, _ptr(self.params), _ptr(self.adam_m), _ptr(self.adam_v), _ptr(self.grads)))
        if os.environ.get("DRVAE_B200_GRAPH", "1") == "0":  # measurement knob: launch kernel by kernel
            self.set_graph(False)

    def __del__(self):
        try:
            if getattr(self, "h", None):
                self.lib.drvae_plan_destroy(self.h)
                self.h = None
        except Exception:
            pass

    # ---- parameters -----------------------------------------------------------------------
    def tensor_views(self, buf, model=0):
        """name -> zero-copy view (reference shapes, SURVEY.md Appendix C) into buf[model].  Matrix rows are
        16-byte aligned in the flat vector, so a matrix whose width is not a multiple of 4 is a strided view."""
        out = OrderedDict()
        for (name, r, c, off), ld in zip(self.tensors, self.tensor_ld):
            if c > 0:
                out[name] = buf[model, off:off + r * ld].view(r, ld)[:, :c]
            else:
                out[name] = buf[model, off:off + r]
        return out

    def state_dict(self, model=0):
        return OrderedDict((k, v.detach().clone(memory_format=torch.contiguous_format)) for k, v in self.tensor_views(self.params, model).items())

    def load_state_dict(self, sd, model=0, strict=True):
        views = self.tensor_views(self.params, model)
        missing = [k for k in views if k not in sd]
        extra = [k for k in sd if k not in views]
        if strict and (missing or extra):
            raise KeyError("state_dict mismatch: missing %s unexpected %s" % (missing, extra))
        with torch.no_grad():
            for k, v in views.items():
                if k in sd:
                    src = sd[k]
                    if tuple(src.shape) != tuple(v.shape):
                        raise ValueError("shape mismatch for %s: %s vs %s" % (k, tuple(src.shape), tuple(v.shape)))
                    v.copy_(src.to(self.device, torch.float32))
        self.sync_shadows()

    def sync_shadows(self):
        _lib.check(self.lib.drvae_sync_shadows(self.h, self._stream()), "sync_shadows")

    def _stream(self):
        return ctypes.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    # ---- marshalling ----------------------------------------------------------------------
    def hparams(self, step, training=True, add_noise=True, noise_std=0.01, beta_pert=1.0, pertloss_rate=0.05,
                kl_qz2pz2_rate=1.0, yloss_rate=1.0, kl_min=2.0, lr=5e-4, beta1=0.9, beta2=0.999, adam_eps=1e-8,
                weight_decay=0.05, global_counts=None, prior_y=None, global_counts_ptr=None):
        hp = HParams()
        hp.step, hp.training, hp.add_noise = int(step), int(training), int(add_noise)
        hp.noise_std, hp.beta_pert, hp.pertloss_rate = noise_std, beta_pert, pertloss_rate
        hp.kl_qz2pz2_rate, hp.yloss_rate, hp.kl_min = kl_qz2pz2_rate, yloss_rate, kl_min
        hp.lr, hp.beta1, hp.beta2, hp.adam_eps, hp.weight_decay = lr, beta1, beta2, adam_eps, weight_decay
        if isinstance(global_counts, torch.Tensor) and global_counts.is_cuda:
            # device-resident [N, Np, Nlab] (int64), e.g. straight out of an all-reduce: no host round trip
            if global_counts.dtype != torch.int64 or global_counts.numel() != 3 or not global_counts.is_contiguous():
                raise ValueError("device global_counts must be a contiguous int64 tensor of 3 elements")
            hp.global_counts_dev = global_counts.data_ptr()
            hp._keep = global_counts
        elif global_counts is not None:
            hp.global_N, hp.global_Np, hp.global_Nlab = [int(c) for c in global_counts]
        if global_counts_ptr:  # raw device pointer to int64 {N, Np, Nlab} (drvae_dp_counts_ptr)
            hp.global_counts_dev = int(global_counts_ptr)
        ny = max(1, self.dim_y)
        for j in range(8):
            if prior_y is None:
                hp.log_prior_y[j] = math.log(1.0 / ny)
            else:
                hp.log_prior_y[j] = math.log(float(prior_y[j])) if j < len(prior_y) else 0.0
        return hp

    MEMBER_KEYS = ("yloss_rate", "pertloss_rate", "kl_qz2pz2_rate", "noise_std", "lr", "weight_decay", "prior_y")

    def set_member_hparams(self, members):
        """Per-member hyperparameters (drvae_set_member_hparams): `members` is a list of n_models dicts with the keys of
        MEMBER_KEYS (prior_y: class probabilities, as in hparams()); these values then replace the same fields of the
        hparams passed to every step, member by member.  None clears the table.  Takes effect from the next step
        enqueued on the current stream."""
        if members is None:
            with torch.cuda.device(self.device):
                _lib.check(self.lib.drvae_set_member_hparams(self.h, None, 0, self._stream()), "set_member_hparams")
            return
        members = list(members)
        if len(members) != self.E:
            raise ValueError("need one hyperparameter dict per member (%d), got %d" % (self.E, len(members)))
        table = (_lib.MemberHParams * self.E)()
        ny = max(1, self.dim_y)
        for m, (row, d) in enumerate(zip(table, members)):
            if set(d) != set(self.MEMBER_KEYS):
                raise ValueError("member %d: keys must be %s, got %s" % (m, sorted(self.MEMBER_KEYS), sorted(d)))
            for k in self.MEMBER_KEYS[:-1]:
                x = float(d[k])
                if not math.isfinite(x) or x < 0:
                    raise ValueError("member %d: %s must be finite and >= 0, got %r" % (m, k, d[k]))
                setattr(row, k, x)
            prior = [float(p) for p in d["prior_y"]]
            if len(prior) != ny or not all(math.isfinite(p) and p > 0 for p in prior):
                raise ValueError("member %d: prior_y must be %d positive probabilities, got %r" % (m, ny, d["prior_y"]))
            for j in range(8):
                row.log_prior_y[j] = math.log(prior[j]) if j < ny else 0.0
        with torch.cuda.device(self.device):
            _lib.check(self.lib.drvae_set_member_hparams(self.h, table, self.E, self._stream()), "set_member_hparams")

    def _batch(self, x1, x2=None, y=None, has_x2=None, has_y=None, row_index=None):
        """Marshal one minibatch per model.  With row_index ([n_models, N] or [N] int32) the other fields are whole
        device-resident datasets ([n_models, D, ...]) and the minibatch is rows row_index of them — the step reads the
        dataset through the indices (drvae_batch_t.row_index), nothing is gathered."""
        def f32(t):
            if t is None:
                return None
            t = t.to(self.device, torch.float32)
            return t.contiguous()

        def i32(t):
            if t is None:
                return None
            return t.to(self.device, torch.int32).contiguous()

        x1 = f32(x1)
        if x1.dim() == 2:
            if self.E != 1:
                raise ValueError("ensemble plans take batches shaped [n_models, N, dim_x]")
            rows = x1.shape[0]
        else:
            if x1.shape[0] != self.E:
                raise ValueError("first batch dimension must be n_models")
            rows = x1.shape[1]
        if x1.shape[-1] != self.dim_x:
            raise ValueError("x1 has %d features, the model has dim_x=%d" % (x1.shape[-1], self.dim_x))
        ridx = i32(row_index)
        N = rows
        if ridx is not None:
            if ridx.numel() % self.E != 0:
                raise ValueError("row_index must be shaped [n_models, N]")
            N = ridx.numel() // self.E
        keep = [x1, f32(x2), i32(y), i32(has_x2), i32(has_y), ridx]
        for t in keep[1:5]:
            if t is not None and t.numel() not in (self.E * rows, self.E * rows * self.dim_x):
                raise ValueError("batch field has an unexpected number of elements")
        b = Batch(_ptr(keep[0]), _ptr(keep[1]), _ptr(keep[2]), _ptr(keep[3]), _ptr(keep[4]), int(N), _ptr(ridx),
                  int(rows) if ridx is not None else 0)
        return b, keep

    def _noise(self, eps, seed, row_offset=0):
        if eps is not None:
            eps = eps.to(self.device, torch.float32).contiguous()
            if eps.numel() != self.E * self.eps_layout.total:
                raise ValueError("eps block must have n_models * %d floats" % self.eps_layout.total)
        return Noise(_ptr(eps), int(seed) & 0xFFFFFFFFFFFFFFFF, int(row_offset)), eps

    def _run(self, fn, what, batch, hp, eps=None, seed=0, row_offset=0, losses_out=None):
        b, keep = self._batch(**batch)
        nz, keep_eps = self._noise(eps, seed, row_offset)
        lo = _ptr(self.losses) if losses_out is None else _ptr(losses_out)
        with torch.cuda.device(self.device):
            cur = torch.cuda.current_stream(self.device)
            if cur.cuda_stream == 0:
                own = self._own_stream
                own.wait_stream(cur)
                _lib.check(fn(self.h, ctypes.byref(b), ctypes.byref(nz), ctypes.byref(hp), lo,
                              ctypes.c_void_p(own.cuda_stream)), what)
                cur.wait_stream(own)  # later work on the caller's stream (incl. reuse of freed batch memory) is ordered after the step
            else:
                _lib.check(fn(self.h, ctypes.byref(b), ctypes.byref(nz), ctypes.byref(hp), lo, self._stream()), what)
        del keep, keep_eps  # stream-ordered: torch's caching allocator keeps them alive for this stream
        return self.losses if losses_out is None else losses_out

    def train_step(self, batch, hp, eps=None, seed=0, row_offset=0):
        return self._run(self.lib.drvae_train_step, "train_step", batch, hp, eps, seed, row_offset)

    def grad_step(self, batch, hp, eps=None, seed=0, row_offset=0, losses_out=None):
        return self._run(self.lib.drvae_grad_step, "grad_step", batch, hp, eps, seed, row_offset, losses_out)

    def loss_forward(self, batch, hp, eps=None, seed=0, row_offset=0):
        return self._run(self.lib.drvae_loss_forward, "loss_forward", batch, hp, eps, seed, row_offset)

    def adam_step(self, hp):
        with torch.cuda.device(self.device):
            _lib.check(self.lib.drvae_adam_step(self.h, ctypes.byref(hp), self._stream()), "adam_step")

    # ---- data parallelism over NVLink peer memory (include/drvae_b200.h, drvae_dp_*) ----
    def dp_grad_floats(self):
        return int(self.lib.drvae_dp_grad_floats(self.h))

    def dp_attach(self, rank, world, grad_ptrs, ctl_ptrs, multicast_ptr=0):
        pe = _lib.DpPeers()
        pe.rank, pe.world = int(rank), int(world)
        ga = (ctypes.c_void_p * world)(*[int(p) for p in grad_ptrs])
        ca = (ctypes.c_void_p * world)(*[int(p) for p in ctl_ptrs])
        pe.grad_ptrs, pe.ctl_ptrs = ga, ca
        pe.grads_multicast = int(multicast_ptr) if multicast_ptr else None
        _lib.check(self.lib.drvae_dp_attach(self.h, ctypes.byref(pe)), "dp_attach")
        self.dp_counts_ptr = int(self.lib.drvae_dp_counts_ptr(self.h))

    def dp_exchange_counts(self, counts, tag):
        with torch.cuda.device(self.device):
            _lib.check(self.lib.drvae_dp_exchange_counts(self.h, int(counts[0]), int(counts[1]), int(counts[2]), int(tag), self._stream()),
                       "dp_exchange_counts")

    def dp_train_step(self, batch, hp, losses_out, eps=None, seed=0, row_offset=0):
        """One data-parallel optimisation step (drvae_dp_train_step): with peers attached gradient, NVLink reduction and
        Adam, the global losses written to losses_out (8 floats); without, this plan's rows alone ([n_models, 8])."""
        return self._run(self.lib.drvae_dp_train_step, "dp_train_step", batch, hp, eps, seed, row_offset, losses_out)

    def infer(self, x1):
        x1 = x1.to(self.device, torch.float32).contiguous()
        if x1.dim() == 2:
            x1 = x1.unsqueeze(0)
        E, N = x1.shape[0], x1.shape[1]
        if E != self.E:
            raise ValueError("first dimension must be n_models")
        kw = dict(dtype=torch.float32, device=self.device)
        Z, X, Y = self.dim_z1, self.dim_x, max(1, self.dim_y)
        res = OrderedDict()
        res["z1_mu"], res["z1_lv"] = torch.empty(E, N, Z, **kw), torch.empty(E, N, Z, **kw)
        res["px1_mu"], res["px1_sg"] = torch.empty(E, N, X, **kw), torch.empty(E, N, X, **kw)
        if self.kind in ("drvae", "pvae"):
            res["z2_mu"], res["z2_lv"] = torch.empty(E, N, Z, **kw), torch.empty(E, N, Z, **kw)
            res["px2_mu"], res["px2_sg"] = torch.empty(E, N, X, **kw), torch.empty(E, N, X, **kw)
        if self.kind in ("drvae", "vfae"):
            res["proba"] = torch.empty(E, N, Y, **kw)
            res["pred"] = torch.empty(E, N, dtype=torch.int32, device=self.device)
        out = InferOut()
        for k, v in res.items():
            setattr(out, k, v.data_ptr())
        with torch.cuda.device(self.device):
            _lib.check(self.lib.drvae_infer(self.h, _ptr(x1), int(N), ctypes.byref(out), self._stream()), "infer")
        return res

    def set_infer_precision(self, fp32=True):
        """fp32 (default): exact thresholded predictions; False: bf16 tensor-core inference."""
        _lib.check(self.lib.drvae_set_infer_precision(self.h, int(bool(fp32))), "set_infer_precision")

    def grad_buckets(self):
        """[(offset, count)] of the flat gradient in the order drvae_grad_step completes them."""
        out = []
        for i in range(self.lib.drvae_plan_num_buckets(self.h)):
            off, cnt = ctypes.c_longlong(), ctypes.c_longlong()
            _lib.check(self.lib.drvae_plan_bucket_info(self.h, i, ctypes.byref(off), ctypes.byref(cnt)), "bucket_info")
            out.append((off.value, cnt.value))
        return out

    def stream_wait_bucket(self, index, stream):
        _lib.check(self.lib.drvae_stream_wait_bucket(self.h, int(index), ctypes.c_void_p(stream.cuda_stream)), "wait_bucket")

    # ---- introspection --------------------------------------------------------------------
    def set_graph(self, enable):
        _lib.check(self.lib.drvae_set_graph(self.h, int(bool(enable))), "set_graph")

    def graph_replays(self):
        return int(self.lib.drvae_plan_graph_replays(self.h))

    def graph_failures(self):
        return int(self.lib.drvae_plan_graph_failures(self.h))

    def set_step_kernel(self, enable):
        """Persistent step kernel on / off (default: one launch per GEMM and row operation)."""
        _lib.check(self.lib.drvae_set_step_kernel(self.h, 1 if enable else 0))

    def step_kernel_launches(self):
        return int(self.lib.drvae_plan_step_kernel_launches(self.h))

    def set_gemm_impl(self, impl):
        _lib.check(self.lib.drvae_set_gemm_impl(self.h, {"tc": 0, "simt": 1}[impl]))

    def debug_side_delay(self, cycles):
        _lib.check(self.lib.drvae_debug_side_delay(self.h, int(cycles)), "debug_side_delay")

    def launch_count(self):
        return int(self.lib.drvae_plan_launch_count(self.h))

    def profile_begin(self):
        _lib.check(self.lib.drvae_profile_begin(self.h), "profile_begin")

    def profile_end(self):
        """-> {tag: (launches, total_ms)} for everything launched since profile_begin()."""
        buf = ctypes.create_string_buffer(1 << 16)
        _lib.check(self.lib.drvae_profile_end(self.h, buf, len(buf)), "profile_end")
        out = {}
        for line in buf.value.decode().splitlines():
            tag, n, ms = line.rsplit(" ", 2)
            out[tag] = (int(n), float(ms))
        return out

    def dwa_stats(self, enable):
        """enable=True: start counting; False: -> dict of the grouped dW+Adam kernel's role wait cycles."""
        out = (ctypes.c_ulonglong * 8)()
        _lib.check(self.lib.drvae_debug_dwa_stats(self.h, int(bool(enable)), out), "dwa_stats")
        names = ("epi_wait_acc", "epi_wait_state", "loader_wait_empty", "storer_wait_done", "storer_wait_read",
                 "producer_wait_empty", "mma_wait_full", "cta_total")
        return None if enable else dict(zip(names, [int(x) for x in out]))

    def trace_begin(self, max_launches=4096):
        _lib.check(self.lib.drvae_trace_begin(self.h, int(max_launches)), "trace_begin")

    def trace_end(self):
        """-> [(index, tag, start_ns, end_ns)] for every kernel launched since trace_begin()."""
        buf = ctypes.create_string_buffer(1 << 20)
        _lib.check(self.lib.drvae_trace_end(self.h, buf, len(buf)), "trace_end")
        out = []
        for line in buf.value.decode().splitlines():
            i, tag, a, b = line.rsplit(" ", 3)
            out.append((int(i), tag, int(a), int(b)))
        return out

    def workspace_bytes(self):
        return int(self.lib.drvae_plan_workspace_bytes(self.h))

    def debug_buffer(self, name, dtype=torch.float32):
        """Zero-copy [n_models, elems_per_model] view of a workspace buffer (tests only)."""
        ptr, ms, nb = ctypes.c_void_p(), ctypes.c_longlong(), ctypes.c_longlong()
        rcap, fcap = ctypes.c_int(), ctypes.c_int()
        _lib.check(self.lib.drvae_debug_buffer(self.h, name.encode(), ctypes.byref(ptr), ctypes.byref(ms), ctypes.byref(nb),
                                               ctypes.byref(rcap), ctypes.byref(fcap)), "debug_buffer")
        item = {torch.float32: (4, "<f4"), torch.int32: (4, "<i4"), torch.bfloat16: (2, "<i2")}[dtype]
        per = ms.value // item[0]
        t = torch.as_tensor(_CudaView(ptr.value, (self.E, per), item[1]), device=self.device)
        if dtype == torch.bfloat16:
            t = t.view(torch.bfloat16)
        return t[:, :nb.value // item[0]], rcap.value, fcap.value

    def debug_c8(self, name, rows, feats, model=0):
        from .layout import unpack_c8
        t, rcap, fcap = self.debug_buffer(name, torch.bfloat16)
        return unpack_c8(t[model].view(fcap // 8, rcap, 8), rows, feats)


def losses_to_dict(kind, row):
    """One row of the [n_models, 8] loss tensor -> the reference's OrderedDict of 0-dim tensors
    (DrVAE.py:611-626; PVAE has no YL, VFAE has no PERT)."""
    out = OrderedDict()
    for i, k in enumerate(LOSS_KEYS):
        if (kind == "pvae" and k == "YL") or (kind == "vfae" and k == "PERT"):
            continue
        out[k] = row[i]
    return out
