"""Training-loop surface of the reference around the accelerated step: dataset wrappers, evaluation
metrics and `fit()` with the reference's early-stopping rule.

Reference (paths relative to /root/reference/src): `DrVAEDataset` / `wrap_in_DrVAEDataset`
DrVAE.py:880-963, `VFAEDataset` / `wrap_in_VFAEDataset` VFAE.py:658-721, `eval_x_reconstruction` /
`eval_y_prediction` DGMMixin.py:128-190, `evaluate_performance[_on_dataset]` DrVAE.py:628-741,
`fit` DrVAE.py:743-877 (PVAE.py:554-671, VFAE.py:523-655).  SURVEY.md §8(f) ranks these as the
components next to the hot path: they stay host-side Python, but everything per-sample runs on
the GPU — the forward pass through `drvae_infer`, and the reconstruction metrics (RMSE, variance-
weighted R², the per-row Pearson correlation the reference computes in a Python loop over
scipy.stats.pearsonr, Gaussian log-likelihood) as batched device reductions, and accuracy, AUROC and
AUPR from exact rank counts (drvae_eval_members, one call for every member of an ensemble).  The
sklearn form of the y metrics stays as the host path for CPU tensors and as the tests' reference.
"""
import math
import time
from collections import OrderedDict

import numpy as np
import torch


# ------------------------------------------------------------------------------------------------
# datasets (boundary format of the step: DrVAE.py:956-961)
# ------------------------------------------------------------------------------------------------
class DrVAEDataset(torch.utils.data.Dataset):
    """(x1, x2, s, y, has_x2, has_y) rows; singletons carry an all-zero x2 and has_x2 = 0."""
    fields = ("x1", "x2", "s", "y", "has_x2", "has_y")

    def __init__(self, x1, x2, s, y, has_x2, has_y):
        n = x1.size(0)
        for name, t in (("x2", x2), ("s", s), ("y", y), ("has_x2", has_x2), ("has_y", has_y)):
            if t.size(0) != n:
                raise ValueError("DrVAEDataset: %s has %d rows, x1 has %d" % (name, t.size(0), n))
        if x1.shape != x2.shape:
            raise ValueError("DrVAEDataset: x1 and x2 must have the same shape")
        self.x1, self.x2, self.s, self.y, self.has_x2, self.has_y = x1, x2, s, y, has_x2, has_y

    def __getitem__(self, i):
        return self.x1[i], self.x2[i], self.s[i], self.y[i], self.has_x2[i], self.has_y[i]

    def __len__(self):
        return self.x1.size(0)


class VFAEDataset(torch.utils.data.Dataset):
    """(x1, s, y, has_y) rows (VFAE.py:658-680)."""
    fields = ("x1", "s", "y", "has_y")

    def __init__(self, x1, s, y, has_y):
        n = x1.size(0)
        for name, t in (("s", s), ("y", y), ("has_y", has_y)):
            if t.size(0) != n:
                raise ValueError("VFAEDataset: %s has %d rows, x1 has %d" % (name, t.size(0), n))
        self.x1, self.s, self.y, self.has_y = x1, s, y, has_y

    def __getitem__(self, i):
        return self.x1[i], self.s[i], self.y[i], self.has_y[i]

    def __len__(self):
        return self.x1.size(0)


def _downlabel(d, keep_cids):
    """Keep labels only for `keep_cids` cell lines; others become unlabeled with y = -66 like the reference."""
    labeled = np.unique(d["cid"][d["has_y"].astype(bool)])
    np.random.shuffle(labeled)
    keep = set(labeled[:keep_cids].tolist())
    drop = np.array([c not in keep for c in d["cid"]])
    d["has_y"] = np.where(drop, 0, d["has_y"])
    for k in ("y", "ycont"):
        if k in d:
            d[k] = np.where(drop, -66, d[k])


def wrap_in_DrVAEDataset(sing, pair, y_key="y", concat="both", downlabel_to=None, remove_unlabeled=False):
    """dicts of numpy arrays (singletons, perturbation pairs) -> (DrVAEDataset, merged dict)."""
    if concat == "both":
        d = {k: np.concatenate((sing[k], pair[k])) for k in set(sing) & set(pair)}
        d["x2"] = np.concatenate((np.zeros_like(sing["x1"]), pair["x2"]))
        d["has_x2"] = np.concatenate((np.zeros(len(sing["x1"])), np.ones(len(pair["x2"]))))
    elif concat == "pair_only":
        d = dict(pair)
        d["has_x2"] = np.ones(len(pair["x2"]))
    elif concat == "sing_only":
        d = dict(sing)
        d["x2"] = np.zeros_like(sing["x1"])
        d["has_x2"] = np.zeros(len(sing["x1"]))
    else:
        raise ValueError("Invalid parameter for dataset concatenation type")
    if downlabel_to is not None:
        _downlabel(d, downlabel_to)
    if remove_unlabeled:
        keep = d["has_y"] != 0
        d = {k: v[keep] for k, v in d.items()}
    ds = DrVAEDataset(x1=torch.from_numpy(np.ascontiguousarray(d["x1"])).float(),
                      x2=torch.from_numpy(np.ascontiguousarray(d["x2"])).float(),
                      s=torch.from_numpy(d["s"].astype(np.int32)), y=torch.from_numpy(np.ascontiguousarray(d[y_key])),
                      has_x2=torch.from_numpy(d["has_x2"].astype(np.int32)),
                      has_y=torch.from_numpy(d["has_y"].astype(np.int32)))
    return ds, d


def wrap_in_VFAEDataset(sing, pair=None, y_key="y", concat="sing_only", downlabel_to=None, remove_unlabeled=False):
    """VFAE.py:683-721: singletons, optionally with the x1 side of the pairs appended."""
    if concat == "both" and pair is not None:
        d = {k: np.concatenate((sing[k], pair[k])) for k in set(sing) & set(pair)}
    elif concat in ("sing_only", "both"):
        d = dict(sing)
    elif concat == "pair_only":
        d = dict(pair)
    else:
        raise ValueError("Invalid parameter for dataset concatenation type")
    if downlabel_to is not None:
        _downlabel(d, downlabel_to)
    if remove_unlabeled:
        keep = d["has_y"] != 0
        d = {k: v[keep] for k, v in d.items()}
    ds = VFAEDataset(x1=torch.from_numpy(np.ascontiguousarray(d["x1"])).float(), s=torch.from_numpy(d["s"].astype(np.int32)),
                     y=torch.from_numpy(np.ascontiguousarray(d[y_key])), has_y=torch.from_numpy(d["has_y"].astype(np.int32)))
    return ds, d


# ------------------------------------------------------------------------------------------------
# metrics (DGMMixin.py:128-190), batched on the device
# ------------------------------------------------------------------------------------------------
def eval_x_reconstruction(x, x_rec, x_rec_sigma=None, mask=None):
    """rmse, variance-weighted r2, mean per-row Pearson r, mean per-row Gaussian log-likelihood over the rows with
    mask != 0 (DGMMixin.py:128-158).  CUDA tensors go through drvae_eval_x_reconstruction (fp64 device reductions, one
    4-double read back); CPU tensors (host-side tests) through the same formulas in torch."""
    if x.is_cuda:
        import ctypes
        from . import _lib
        lib = _lib.load()
        x = x.detach().float().contiguous()
        r = x_rec.detach().float().contiguous()
        sg = x_rec_sigma.detach().float().contiguous() if x_rec_sigma is not None else None
        mk = mask.detach().to(torch.int32).contiguous() if mask is not None else None
        N, X = x.shape
        ws = torch.empty(int(lib.drvae_eval_workspace_bytes(N, X)), dtype=torch.uint8, device=x.device)
        out = torch.empty(4, dtype=torch.float64, device=x.device)
        ptr = lambda t: ctypes.c_void_p(t.data_ptr()) if t is not None else None
        _lib.check(lib.drvae_eval_x_reconstruction(ptr(x), ptr(r), ptr(sg), ptr(mk), N, X, ptr(out), ptr(ws),
                                                   ctypes.c_void_p(torch.cuda.current_stream(x.device).cuda_stream)), "eval_x_reconstruction")
        v = out.cpu().tolist()
        return {"rmse": v[0], "r2": v[1], "pearr": v[2], "ll": v[3]}
    if mask is not None:
        idx = torch.nonzero(mask).view(-1)
        x, x_rec = x[idx], x_rec[idx]
        x_rec_sigma = x_rec_sigma[idx] if x_rec_sigma is not None else None
    x = x.double()
    r = x_rec.double()
    out = {}
    out["rmse"] = float(((x - r) ** 2).mean().sqrt())
    # sklearn.metrics.r2_score(multioutput='variance_weighted') = 1 - sum_f SSres_f / sum_f SStot_f
    ss_res = ((x - r) ** 2).sum()
    ss_tot = ((x - x.mean(0, keepdim=True)) ** 2).sum()
    out["r2"] = float(1.0 - ss_res / ss_tot) if float(ss_tot) > 0 else float("nan")
    xc = x - x.mean(1, keepdim=True)
    rc = r - r.mean(1, keepdim=True)
    den = xc.norm(dim=1) * rc.norm(dim=1)
    out["pearr"] = float(((xc * rc).sum(1) / den).mean())  # rows with zero variance give nan, like scipy
    if x_rec_sigma is not None:
        sg = x_rec_sigma.double()
        ll = -0.5 * (math.log(2 * math.pi) + (sg * sg).log() + (x - r) ** 2 / (sg * sg))
        out["ll"] = float(ll.sum(1).mean())
    else:
        out["ll"] = float("nan")
    return out


def eval_members(valid, x1=None, px1_mu=None, px1_sg=None, x2=None, px2_mu=None, px2_sg=None, has_x2=None, proba=None,
                 pred=None, y=None, has_y=None):
    """drvae_eval_members: the metrics of E models on padded device data in one call, no host synchronisation.

    valid: int [E, D], the rows of each member; x1 / px1_mu / px1_sg, x2 / px2_mu / px2_sg: float [E, D, X]; has_x2,
    pred, y, has_y: int [E, D]; proba: float [E, D, dim_y].  x2 metrics use the rows with valid and has_x2, y metrics
    those with valid and has_y.  A group left out (x1, x2 or y) gives nan.  -> float64 [E, 11] device tensor, columns
    _lib.EVAL_MEMBER_COLUMNS."""
    import ctypes
    from . import _lib
    lib = _lib.load()
    if not valid.is_cuda or valid.dim() != 2:
        raise ValueError("eval_members: valid must be a CUDA tensor [E, D]")
    dev = valid.device
    E, D = valid.shape
    X = x1.shape[2] if x1 is not None else (x2.shape[2] if x2 is not None else 1)
    Y = proba.shape[2] if proba is not None else 0
    keep = []

    def ptr(t, dtype, width=None):
        if t is None:
            return None
        if tuple(t.shape) != ((E, D) if width is None else (E, D, width)):
            raise ValueError("eval_members: a tensor of shape %s, expected [%d, %d%s]" % (
                tuple(t.shape), E, D, "" if width is None else ", %d" % width))
        t = t.detach().to(dev, dtype).contiguous()
        keep.append(t)
        return t.data_ptr()

    f, i = torch.float32, torch.int32
    args = _lib.EvalMembersIn(valid=ptr(valid, i), x1=ptr(x1, f, X), px1_mu=ptr(px1_mu, f, X), px1_sg=ptr(px1_sg, f, X),
                              x2=ptr(x2, f, X), px2_mu=ptr(px2_mu, f, X), px2_sg=ptr(px2_sg, f, X), has_x2=ptr(has_x2, i),
                              proba=ptr(proba, f, Y), pred=ptr(pred, i), y=ptr(y, i), has_y=ptr(has_y, i))
    ws = torch.empty(int(lib.drvae_eval_members_workspace_bytes(E, D, X, Y)), dtype=torch.uint8, device=dev)
    out = torch.empty(E, len(_lib.EVAL_MEMBER_COLUMNS), dtype=torch.float64, device=dev)
    _lib.check(lib.drvae_eval_members(ctypes.byref(args), E, D, X, Y, ctypes.c_void_p(out.data_ptr()),
                                      ctypes.c_void_p(ws.data_ptr()), ctypes.c_void_p(torch.cuda.current_stream(dev).cuda_stream)),
               "eval_members")
    return out


def eval_y_prediction(pred, proba, ylab, dim_y=2):
    """acc, auroc, aupr (DGMMixin.py:160-190) over all given rows.  CUDA tensors go through drvae_eval_members (one
    3-double read back); CPU tensors through sklearn, as the reference does."""
    if proba.is_cuda:
        n = int(ylab.shape[0])
        if n == 0:
            return {"acc": float("nan"), "auroc": float("nan"), "aupr": float("nan")}
        if proba.dim() != 2 or proba.shape[1] != dim_y:
            raise ValueError("eval_y_prediction: proba must be [N, dim_y]")
        ones = torch.ones(1, n, dtype=torch.int32, device=proba.device)
        v = eval_members(ones, proba=proba.unsqueeze(0), pred=pred.reshape(1, n), y=ylab.long().reshape(1, n),
                         has_y=ones)[0, :3].cpu().tolist()
        return {"acc": v[0], "auroc": v[1], "aupr": v[2]}
    import sklearn.metrics
    out = {}
    y = ylab.long().cpu().numpy()
    out["acc"] = float((pred.long().cpu().numpy() == y).mean()) if len(y) else float("nan")
    p = proba.float().cpu().numpy()
    try:
        if dim_y == 2:
            out["auroc"] = float(sklearn.metrics.roc_auc_score(y, p[:, 1]))
            out["aupr"] = float(sklearn.metrics.average_precision_score(y, p[:, 1]))
        else:
            hot = np.eye(dim_y)[y]
            out["auroc"] = float(sklearn.metrics.roc_auc_score(hot, p, average="macro"))
            out["aupr"] = float(sklearn.metrics.average_precision_score(hot, p, average="macro"))
    except ValueError:  # a single class present
        out.setdefault("auroc", float("nan"))
        out.setdefault("aupr", float("nan"))
    return out


def evaluate_performance(model, return_full_data=False, **batch):
    """evaluate_performance (DrVAE.py:640-741, PVAE/VFAE analogues): eval-mode losses, inference, y metrics on the
    labeled rows, x1 reconstruction on all rows, x2 perturbation prediction on the paired rows."""
    perf = OrderedDict()
    try:
        perf["losses"] = model.run_on_batch(train_mode=False, **batch)
    except Exception as e:  # the reference swallows loss failures in evaluation (DrVAE.py:647-653)
        print("Warning, computation of losses failed in evaluation!")
        print(e)
        perf["losses"] = None
    dev = model.plan.device
    x1 = batch["x1"].to(dev)
    res = model.forward(x1)
    parts = []
    if model.kind != "pvae":
        idx = torch.nonzero(batch["has_y"].to(dev)).view(-1)
        m = eval_y_prediction(res["pred"][idx], res["proba"][idx], batch["y"].to(dev)[idx], model.dim_y)
        perf.update(("y_" + k, v) for k, v in m.items())
        parts.append("Y: Accuracy: {:.3f}% AUROC: {:.3f} AUPR: {:.3f}".format(perf["y_acc"] * 100., perf["y_auroc"], perf["y_aupr"]))
    m = eval_x_reconstruction(x1, *res["px1"])
    perf.update(("x1_" + k, v) for k, v in m.items())
    parts.append("X1: RMSE: {:.3f} R2: {:.3f} Pearson: {:.3f}".format(perf["x1_rmse"], perf["x1_r2"], perf["x1_pearr"]))
    if model.kind != "vfae":
        hx2 = batch["has_x2"].to(dev)
        if bool(hx2.ne(0).any()):
            m = eval_x_reconstruction(batch["x2"].to(dev), res["px2"][0], res["px2"][1], mask=hx2)
            perf.update(("x2_" + k, v) for k, v in m.items())
            parts.append("X2: RMSE: {:.3f} R2: {:.3f} Pearson: {:.3f}".format(perf["x2_rmse"], perf["x2_r2"], perf["x2_pearr"]))
        else:
            perf.update(("x2_" + k, float("nan")) for k in ("rmse", "r2", "pearr", "ll"))
            parts.append("X2: no x2 data")
    if return_full_data:
        for k in ("z1", "z2", "x2_pert", "pred", "proba"):
            if k in res:
                perf[k] = res[k].cpu().numpy()
    perf["model_class"] = type(model).__name__
    return perf, "\t ".join(parts)


def _dataset_batch(model, ds):
    b = {k: getattr(ds, k) for k in ds.fields}
    return b


def evaluate_performance_on_dataset(model, ds, return_full_data=False):
    return evaluate_performance(model, return_full_data=return_full_data, **_dataset_batch(model, ds))


def validation_objective(model, perf):
    """The quantity early stopping maximises (DrVAE.py:822-826, PVAE.py:620, VFAE.py:590)."""
    if model.kind == "drvae":
        return perf["y_auroc"] + perf["y_aupr"] + perf["x1_pearr"] + perf["x2_pearr"]
    if model.kind == "pvae":
        return perf["x1_pearr"] + perf["x2_pearr"]
    return perf["y_auroc"] + perf["y_aupr"] + perf["x1_pearr"]


class SnapshotRule:
    """The early-stopping rule of the reference's fit (DrVAE.py:822-860): the rolling mean over 3 epochs of the
    validation objective, patience >= 50 epochs (40 for VFAE) extended to epoch + 15 at every 0.1 % improvement, a
    snapshot at every improvement (early_stop) or once when patience runs out, and, without early_stop, training that
    continues after patience with the patience pushed past the epoch cap.  Shared by fit() and sweep.fit_sweep()."""
    patience_increase, improvement_threshold, memory_length = 15, 0.999, 3

    def __init__(self, kind, epochs, early_stop=False, min_patience=None):
        self.patience = min_patience if min_patience is not None else (40 if kind == "vfae" else 50)
        self.epochs, self.early_stop = int(epochs), bool(early_stop)
        self.best, self.rolling, self.mean = -np.inf, [], float("nan")
        self.since_improvement, self.snapshotted = 0, False

    def update(self, epoch, vobj):
        """Record epoch `epoch`'s validation objective.  -> (snapshot, patience_reached, stop): take a snapshot now;
        patience ran out this epoch; training stops (early_stop only)."""
        self.since_improvement += 1
        self.rolling = (self.rolling + [vobj])[-self.memory_length:]
        self.mean = float(np.mean(self.rolling))
        self.best_before = self.best
        if self.mean * self.improvement_threshold > self.best:
            self.patience = max(self.patience, epoch + self.patience_increase)
            self.best, self.since_improvement = self.mean, 0
        snapshot = (self.early_stop and self.since_improvement == 0) or (self.patience <= epoch and not self.snapshotted)
        if snapshot:
            self.snapshotted = True
        reached = self.patience <= epoch
        if reached and not self.early_stop:
            self.patience, self.snapshotted = self.epochs + 1, False
        return snapshot, reached, reached and self.early_stop


def fit(model, train_loader, valid_loader, add_noise=False, verbose=False, early_stop=False, model_filename="best_model.pth",
        min_patience=None):
    """Train `model` (reference `fit`): epochs of run_on_batch(train_mode=True) over train_loader, evaluation of
    the full train / validation sets every epoch, early stopping on the rolling mean (3 rounds) of the validation
    objective with patience >= 50 epochs (40 for VFAE), extended by 15 epochs at every 0.1 % improvement, and a
    state_dict snapshot at the best epoch (SnapshotRule)."""
    rule = SnapshotRule(model.kind, model.epochs, early_stop, min_patience)
    fields = train_loader.dataset.fields
    model.w2log("Starting training at: {}".format(time.strftime("%c")))
    epoch = 0
    try:
        model.add_noise = add_noise
        for epoch in range(1, model.epochs + 1):
            t0 = time.time()
            train_loss, nb = 0.0, 0
            for bi, tensors in enumerate(train_loader):
                batch = dict(zip(fields, tensors))
                loss = model.run_on_batch(train_mode=True, **batch)
                train_loss += float(getattr(model, "yloss_rate", 0.) * loss.get("YL", 0.) + loss["RECL"])
                nb += 1
                if verbose and bi % max(10, len(train_loader) // 10) == 0:
                    model.w2log("training epoch: {} [{}/{}]\t{}".format(
                        epoch, bi * len(tensors[0]), len(train_loader.dataset),
                        "\t".join("{}: {:.3f}".format(k, float(loss[k])) for k in ("CMPL", "ELBO", "RECL", "PERT", "YL") if k in loss)))
            train_loss /= max(1, nb)
            _, train_str = evaluate_performance_on_dataset(model, train_loader.dataset)
            model.w2log("====> Epoch: {}\tIter: {}".format(epoch, model.finished_training_iters))
            model.w2log("Train: sec/epoch: {:.2f}\tAvg train loss: {:9.4f}\t{}".format(time.time() - t0, train_loss, train_str))
            t0 = time.time()
            vperf, vstr = evaluate_performance_on_dataset(model, valid_loader.dataset)
            vobj = validation_objective(model, vperf)
            model.w2log("Valid: sec/epoch: {:.2f}\tValid set loss: {:9.4f}\t{}".format(time.time() - t0, vobj, vstr))
            snapshot, reached, stop = rule.update(epoch, vobj)
            model.w2log("Valid rolling mem: {}\tmean: {:.4f}\tbest: {:.4f}".format(np.array(rule.rolling), rule.mean, rule.best_before))
            if snapshot:
                model.save_to_file(model_filename)
                model.w2log("* Snapshotting at epoch {}".format(epoch))
            if reached:
                model.w2log("Early stopping at: {} with train: {:.4f} valid: {:.4f} best_valid_obj: {:.4f}".format(
                    epoch, train_loss, vobj, rule.best))
                if stop:
                    break
                model.w2log("Continuing")
    except KeyboardInterrupt:
        model.w2log("KeyboardInterrupt")
        if not rule.snapshotted:
            model.save_to_file(model_filename)
            model.w2log("* Snapshotting at epoch {}".format(epoch))
    model.w2log("Finished training at: {}".format(time.strftime("%c")))


# ------------------------------------------------------------------------------------------------
# device-resident training loop (SURVEY.md 8(f) rank 2: run_drvae.py:148-166 WeightedRandomSampler + DataLoader,
# utils.py:292-327 compute_balanced_weights, DrVAE.py:766-786 the minibatch loop of fit())
# ------------------------------------------------------------------------------------------------
def compute_balanced_weights(labels):
    """utils.compute_balanced_weights(labels, unlabeled_data_ratio=None): every class (cell line id) weighs 1 / its
    size, so minibatches are expected to hold the same number of samples of each class.  -> float64 tensor."""
    labels = np.asarray(labels)
    classes, inverse, counts = np.unique(labels, return_inverse=True, return_counts=True)
    return torch.from_numpy((1.0 / counts)[inverse]).double()


def device_epoch_indices(weights_dev, batch_size, generator=None):
    """The row indices of ONE epoch, drawn on the device: WeightedRandomSampler(weights, len(weights)) (multinomial with
    replacement) cut into DataLoader minibatches (drop_last when the dataset holds at least one full batch).
    -> int32 [n_batches, batch_size] (the last batch is dropped / the single short batch kept, like the reference)."""
    n = int(weights_dev.numel())
    idx = torch.multinomial(weights_dev.float(), n, replacement=True, generator=generator).to(torch.int32)
    if n >= batch_size:
        nb = n // batch_size
        return idx[:nb * batch_size].view(nb, batch_size).contiguous()
    return idx.view(1, n).contiguous()


def fit_resident(model, dataset, batch_size, epochs=1, weights=None, add_noise=False, seed=0):
    """The minibatch loop of fit() with the whole training set resident on the GPU.

    `dataset` is a DrVAEDataset / VFAEDataset (a few thousand x 978 floats).  Its fields are copied to the device once;
    per epoch ONE device multinomial draw gives every minibatch's row indices, and each step reads the dataset through
    its indices (drvae_batch_t.row_index): no gather kernel, no per-step host->device traffic, no host synchronisation
    inside an epoch — the loss terms of all steps stay in a device buffer and are read once at the end of the epoch.
    From the third step on every step of an epoch is one CUDA-graph replay (same buffers, same shapes).
    Returns [per-epoch OrderedDict of mean loss terms].  Early stopping / evaluation stay in fit()."""
    from .plan import LOSS_KEYS
    dev = model.plan.device
    fields = {k: getattr(dataset, k) for k in dataset.fields}
    fields.pop("s", None)
    batch_all = model._batch_kwargs(**{k: v for k, v in fields.items()})
    n = int(batch_all["x1"].shape[0])
    bs = min(int(batch_size), n)
    model._ensure_capacity(bs)
    plan = model.plan
    data = {k: (v.to(dev).float().contiguous() if v.is_floating_point() else v.to(dev).to(torch.int32).contiguous())
            for k, v in batch_all.items() if v is not None}
    w = (weights if weights is not None else torch.ones(n, dtype=torch.float64)).to(dev)
    gen = torch.Generator(device=dev).manual_seed(int(seed))
    model.add_noise = add_noise
    model.train()
    history = []
    cur = None
    noise_seed = (int(model.random_seed) << 20) ^ 0x5DEECE66D
    for _ in range(int(epochs)):
        idx = device_epoch_indices(w, bs, gen)
        ring = torch.zeros(idx.shape[0], 8, device=dev)
        if cur is None or cur.numel() != idx.shape[1]:
            cur = torch.empty(idx.shape[1], dtype=torch.int32, device=dev)  # fixed address: every step replays one graph
        for b in range(idx.shape[0]):
            cur.copy_(idx[b])
            out = plan.train_step(dict(data, row_index=cur), model._hparams(True), seed=noise_seed)
            ring[b].copy_(out[0], non_blocking=True)
            model.finished_training_iters += 1
        mean = ring.mean(0).cpu()
        history.append(OrderedDict((k, float(mean[i])) for i, k in enumerate(LOSS_KEYS) if k != "MMD"))
    return history
