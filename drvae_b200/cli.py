"""Command-line drivers with the reference's flags (run_drvae.py:245-297, run_pvae.py:235-281,
run_vfae.py:240-292; SURVEY.md Appendix E): `python -m drvae_b200.cli drvae --modelid auto --datafile ...`.

The reference drivers load `CTRPv2+L1000_FDAdrugs6h_v2.1.h5` (absent from the reference checkout), split it per
drug, train with `fit`, reload the best snapshot and write result JSONs.  Here the flags, their defaults, the
hard-coded constructor arguments (run_drvae.py:173-185) and the train -> snapshot -> reload -> evaluate -> JSON
flow are kept; the data source is either a `.npz` with the arrays of `wrap_in_DrVAEDataset` (keys sing_x1,
sing_y, sing_has_y, pair_x1, pair_x2, pair_y, pair_has_y) or `--datafile synthetic[:N]`, an L1000-shaped
synthetic set (978 genes).  The CV splitting / sklearn baselines of utils.py are out of scope (SURVEY.md §2)."""
import argparse
import json
import os
import sys

import numpy as np
import torch

from . import DrVAE, PVAE, VFAE
from .training import wrap_in_DrVAEDataset, wrap_in_VFAEDataset


def build_parser(kind):
    names = dict(drvae="Drug response VAE (DrVAE)", pvae="Perturbation VAE (PertVAE)", vfae="Variational Fair Autoencoder (VFAE / SSVAE)")
    p = argparse.ArgumentParser(prog="drvae_b200.cli " + kind, description=names[kind])
    a = p.add_argument
    a('--cuda', action='store_true', default=False, help='accepted for compatibility: this build is CUDA-only')
    a('--modelid', type=str, required=True, help='model ID')
    a('--datafile', type=str, required=True, help='input data file (.npz) or synthetic[:N]')
    a('--outdir', type=str, default=None, help='output directory')
    a('--fold', type=int, default=1, help='which data fold to run (1 to 5)')
    a('--test-only', action='store_true', default=False, help='load saved parameters and run tests')
    a('--batch-size', type=int, default=200, help='minibatch size')
    a('--L', type=int, default=1, help='number of samples from Q (default 1)')
    a('--stopearly', action='store_true', dest='stopearly', default=False, help='train with early stopping')
    a('--rseed', type=int, default=12345, help='random seed')
    a('--use-s', action='store_true', dest='useS', default=False, help='use model with nuisance variable S')
    a('--use-mmd', action='store_true', dest='useMMD', default=False, help='include MMD loss')
    a('--no-mf', action='store_true', dest='useMF', default=False, help='use molecular features of drugs')
    a('--mmd-rate', type=float, default=1., help='weight of MMD loss')
    a('--data-mode', type=str, default='strictC2C', help='which data to use for training and testing')
    a('--drug', type=str, default='26', help='select one drug to run or set of "26" or "all"')
    a('--train-w-noise', action='store_true', default=False, help='add Gaussian noise to the gene expression during training')
    a('--noise-var', type=float, default=0.01, help='scale of the Gaussian input noise')
    a('--x-dropout', type=float, default=0., help='input dropout rate')
    a('--downlabel-to', type=int, default=None, help='reduce the number of labeled training cell lines')
    a('--dim-z1', type=int, default=50, help='size of z1 & z2')
    a('--enc-z1', type=int, nargs='+', default=[200, 200], help='NN size of encoder q(z_k|x_k)')
    a('--dec-x', type=int, nargs='+', default=[200, 200], help='NN size of decoder p(x_k|z_k)')
    a('--type-y', type=str, default='discrete', help='("discrete" or "cont")')
    a('--epochs', type=int, default=None, help='override the hard-coded epoch cap (300 DrVAE, 1000 PVAE / VFAE)')
    if kind in ('drvae', 'vfae'):
        a('--yloss-rate', type=float, default=50., help='weight of prediction loss on variable Y')
        a('--fully-supervised', action='store_false', dest='semi_supervised', default=True, help='use only labeled data')
        a('--anneal-yloss-offset', type=int, default=1, help='offset for annealing "Y" loss')
        a('--dec-z1', type=int, nargs='+', default=[200], help='NN size of decoder p(z1|z3,y)')
        a('--class-y', type=int, nargs='+', default=[], help='NN size of classifier')
        a('--clf-1sig', action='store_true', default=False, help='1 sigmoid unit instead of softmax over 2 units')
        a('--clf-dataprior', action='store_true', default=False, help='use training data distribution prior')
    if kind == 'drvae':
        a('--pair-data-only', action='store_true', default=False, help='use only perturbation pair data')
        a('--dim-z3', type=int, default=50, help='size of z3')
        a('--enc-z2Fz1', type=int, nargs='+', default=[], help='NN size of encoder p(z2|z1) (ignored, as in the reference)')
        a('--enc-z3', type=int, nargs='+', default=[200], help='NN size of encoder q(z3|z1,y)')
    if kind == 'pvae':
        a('--kl-z2-rate', type=float, default=1., help='weight of KL(q(z2|x2) || p(z2|z1))')
        a('--pair-data-only', action='store_true', default=False, help='use only perturbation pair data')
        a('--with-pairdata-test', action='store_true', default=False, help='test on pair data')
        a('--enc-z2Fz1', type=int, nargs='+', default=[], help='NN size of encoder p(z2|z1)')
    if kind == 'vfae':
        a('--alldata', action='store_true', default=False, help='also use the x1 side of perturbation pairs')
        a('--dim-z2', type=int, default=50, help='size of z2')
        a('--enc-z2', type=int, nargs='+', default=[200], help='NN size of encoder q(z2|z1,y)')
    return p


def synthetic_data(n, dim_x=978, seed=0):
    """L1000-shaped synthetic singletons + pairs (SURVEY.md §8(d) recipe, split half / half)."""
    g = np.random.RandomState(seed)
    x1 = g.randn(n, dim_x).astype(np.float32)
    y = (x1[:, :8].sum(1) + 0.5 * g.randn(n) > 0).astype(np.int64)
    has_y = (np.arange(n) % 3 != 0).astype(np.int32)
    half = n // 2
    sing = dict(x1=x1[:half], y=y[:half], has_y=has_y[:half], s=np.zeros(half, np.int32), cid=np.arange(half))
    pair = dict(x1=x1[half:], x2=(x1[half:] + 0.3 * g.randn(n - half, dim_x)).astype(np.float32), y=y[half:],
                has_y=has_y[half:], s=np.zeros(n - half, np.int32), cid=np.arange(half, n))
    return sing, pair


def load_data(spec, seed):
    if spec.startswith("synthetic"):
        n = int(spec.split(":")[1]) if ":" in spec else 1200
        return synthetic_data(n, seed=seed)
    if spec.endswith(".npz"):
        z = np.load(spec)
        sing = {k[5:]: z[k] for k in z.files if k.startswith("sing_")}
        pair = {k[5:]: z[k] for k in z.files if k.startswith("pair_")}
        for d in (sing, pair):
            d.setdefault("s", np.zeros(len(d["x1"]), np.int32))
            d.setdefault("cid", np.arange(len(d["x1"])))
        return sing, pair
    raise SystemExit("--datafile: only .npz files and 'synthetic[:N]' are supported (the reference's HDF5 loader, "
                     "src/utils.py:506-555, is outside the hot path; SURVEY.md §2)")


def split(d, fold, n_folds=5):
    idx = np.arange(len(d["x1"]))
    test = idx % n_folds == (fold - 1) % n_folds
    valid = idx % n_folds == fold % n_folds
    train = ~(test | valid)
    return [{k: v[m] for k, v in d.items()} for m in (train, valid, test)]


def main(argv=None):
    argv = list(sys.argv[1:] if argv is None else argv)
    if argv and argv[0] == "sweep":
        return sweep_main(argv[1:])
    if not argv or argv[0] not in ("drvae", "pvae", "vfae"):
        raise SystemExit("usage: python -m drvae_b200.cli {drvae|pvae|vfae} --modelid ID --datafile FILE [flags]")
    kind = argv.pop(0)
    args = build_parser(kind).parse_args(argv)
    print(args)
    assert args.data_mode in ['strictC2C'], 'Unsupported data mode'
    assert args.type_y in ['discrete', 'cont'], 'Invalid type-y'
    assert args.useMF is False, 'use of mol.features not supported'
    torch.manual_seed(args.rseed)
    np.random.seed(args.rseed)
    sing, pair = load_data(args.datafile, args.rseed)
    train_ds, valid_ds, test_ds = fold_datasets(kind, args, sing, pair, args.fold)
    dim_x = train_ds.x1.shape[1]
    modelid = args.modelid
    if modelid == 'auto':
        modelid = 'RS{}_L{}_YR{}_FOLD{}'.format(args.rseed, args.L, getattr(args, 'yloss_rate', 0), args.fold)
    outdir = args.outdir or '.'
    os.makedirs(os.path.join(outdir, 'models'), exist_ok=True)
    os.makedirs(os.path.join(outdir, 'results'), exist_ok=True)
    # the reference's fixed constructor choices (run_drvae.py:173-185, run_pvae.py:169-179, run_vfae.py:169-180)
    common = dict(type_rec='diag_gaussian', batch_size=args.batch_size, nonlinearity='elu', learning_rate=0.0005, optim_alg='adam',
                  L=args.L, weight_decay=0.05, dropout_rate=0., input_x_dropout=args.x_dropout, add_noise_var=args.noise_var,
                  use_MMD=args.useMMD, kernel_MMD='rbf_fourier', mmd_rate=args.mmd_rate, use_s=args.useS, random_seed=args.rseed,
                  log_txt=None)
    prior = 'uniform'
    if kind != 'pvae' and args.clf_dataprior:
        lab = train_ds.y[train_ds.has_y != 0].long()
        prior = np.bincount(lab.numpy(), minlength=2).astype(float)
        prior = prior / prior.sum()
    if kind == 'drvae':
        model = DrVAE(dim_x=dim_x, dim_s=1, dim_y=2, dim_h_en_z1=args.enc_z1, dim_h_de_z1=args.dec_z1, dim_h_en_z2Fz1=args.enc_z2Fz1,
                      dim_h_en_z3=args.enc_z3, dim_h_de_x=args.dec_x, dim_h_clf=args.class_y, dim_z1=args.dim_z1, dim_z3=args.dim_z3,
                      clf_z1z2=True, type_y=args.type_y, prior_y=prior, clf_1sig=args.clf_1sig, epochs=args.epochs or 300,
                      yloss_rate=args.yloss_rate, anneal_yloss_offset=args.anneal_yloss_offset, kl_qz2pz2_rate=1., pertloss_rate=0.05,
                      anneal_perturb_rate_itermax=1, anneal_perturb_rate_offset=0, **common)
    elif kind == 'pvae':
        model = PVAE(dim_x=dim_x, dim_s=1, dim_y=2, dim_h_en_z1=args.enc_z1, dim_h_en_z2Fz1=args.enc_z2Fz1, dim_h_de_x=args.dec_x,
                     dim_z1=args.dim_z1, epochs=args.epochs or 1000, kl_qz2pz2_rate=args.kl_z2_rate, pertloss_rate=0.05,
                     anneal_perturb_rate_itermax=1, anneal_perturb_rate_offset=0, **common)
    else:
        model = VFAE(dim_x=dim_x, dim_s=1, dim_y=2, dim_h_en_z1=args.enc_z1, dim_h_de_z1=args.dec_z1, dim_h_en_z2=args.enc_z2,
                     dim_h_de_x=args.dec_x, dim_h_clf=args.class_y, dim_z1=args.dim_z1, dim_z2=args.dim_z2, type_y=args.type_y,
                     prior_y=prior, semi_supervised=True, clf_1sig=args.clf_1sig, epochs=args.epochs or 1000,
                     yloss_rate=args.yloss_rate, anneal_yloss_offset=args.anneal_yloss_offset, **common)
    fname = os.path.join(outdir, 'models', '{}_SD_{}_{}.pth'.format(type(model).__name__, modelid, args.drug))
    if not args.test_only:
        train_loader = torch.utils.data.DataLoader(train_ds, batch_size=args.batch_size, shuffle=True, drop_last=True)
        valid_loader = torch.utils.data.DataLoader(valid_ds, batch_size=args.batch_size)
        try:
            model.fit(train_loader, valid_loader, add_noise=args.train_w_noise, verbose=False, early_stop=args.stopearly,
                      model_filename=fname)
        except Exception as e:  # run_drvae.py:190-195
            print('>>> TRAINING CRASHED <<<')
            print(e)
        if not os.path.exists(fname):
            model.save_to_file(fname)
    model.load_params_from_file(fname)
    results = {}
    for name, ds in (('train', train_ds), ('valid', valid_ds), ('test', test_ds)):
        perf, s = model.evaluate_performance_on_dataset(ds)
        print('{:5s} {}'.format(name, s))
        results[name] = {k: (None if v is None else {kk: float(vv) for kk, vv in v.items()}) if k == 'losses' else v
                         for k, v in perf.items() if not isinstance(v, np.ndarray)}
    out = os.path.join(outdir, 'results', '{}_SD_all_{}.json'.format(type(model).__name__, modelid))
    with open(out, 'w') as f:
        json.dump({args.drug: results}, f, indent=1)
    print('wrote', out)
    return results


# ------------------------------------------------------------------------------------------------
# sweep: the reference's job grid (src/scripts/submitVAE.sh) as one ensemble plan (drvae_b200/sweep.py)
# ------------------------------------------------------------------------------------------------
def build_sweep_parser(kind):
    """The flags of `kind`'s driver plus the grid axes.  --modelid, --rseed and --fold do not apply: members are named
    per grid point as the reference's driver names them with --modelid auto."""
    p = build_parser(kind)
    p.prog = "drvae_b200.cli sweep " + kind
    for act in p._actions:
        if act.dest == 'modelid':
            act.required, act.default = False, 'auto'
    a = p.add_argument
    a('--rseeds', type=int, nargs='+', required=True, help='random seeds of the grid')
    a('--folds', type=int, nargs='+', required=True, help='data folds of the grid (1 to 5)')
    if kind in ('drvae', 'vfae'):
        a('--yloss-rates', type=float, nargs='+', default=None, help='y-loss rates of the grid (default: --yloss-rate)')
    return p


def sweep_grid(kind, args):
    """-> [(seed, rate, fold, modelid)] in the order seeds x rates x folds; rate is 0 for PVAE (no y loss)."""
    rates = (args.yloss_rates or [args.yloss_rate]) if kind != 'pvae' else [0]
    return [(s, r, f, 'RS{}_L{}_YR{}_FOLD{}'.format(s, args.L, r, f)) for s in args.rseeds for r in rates for f in args.folds]


def fold_datasets(kind, args, sing, pair, fold):
    """(train, valid, test) datasets of one fold, as the single-model driver builds them."""
    s_tr, s_va, s_te = split(sing, fold)
    p_tr, p_va, p_te = split(pair, fold)
    if kind == 'vfae':
        mode = 'both' if args.alldata else 'sing_only'
        wrap = lambda s_, p_, **kw: wrap_in_VFAEDataset(s_, p_, concat=mode, **kw)
    else:
        mode = 'pair_only' if args.pair_data_only else 'both'
        wrap = lambda s_, p_, **kw: wrap_in_DrVAEDataset(s_, p_, concat=mode, **kw)
    train_ds, _ = wrap(s_tr, p_tr, downlabel_to=args.downlabel_to,
                       remove_unlabeled=(kind != 'pvae' and not args.semi_supervised))
    return train_ds, wrap(s_va, p_va)[0], wrap(s_te, p_te)[0]


def class_prior(kind, args, train_ds, dim_y=2):
    """--clf-dataprior: class frequencies of the fold's labeled training rows; else uniform."""
    if kind == 'pvae' or not args.clf_dataprior:
        return [1.0 / dim_y] * dim_y
    lab = train_ds.y[train_ds.has_y != 0].long()
    prior = np.bincount(lab.numpy(), minlength=dim_y).astype(float)
    return list(prior / prior.sum())


def sweep_arch(kind, args, dim_x):
    """Plan's shape arguments of a sweep: the single-model driver's flags, --class-y included (DrVAE / VFAE)."""
    if kind == 'drvae':
        arch = dict(dim_z3=args.dim_z3, enc_z3=args.enc_z3, dec_z1=args.dec_z1)
    elif kind == 'vfae':
        arch = dict(dim_z3=args.dim_z2, enc_z3=args.enc_z2, dec_z1=args.dec_z1)
    else:
        arch = dict(dim_z3=0, enc_z3=[], dec_z1=[])
    arch.update(dim_x=dim_x, dim_y=2, dim_z1=args.dim_z1, enc_z1=args.enc_z1, dec_x=args.dec_x)
    if kind != 'pvae':
        arch.update(clf_hidden=list(args.class_y))
    return arch


def sweep_main(argv):
    from . import checkpoint
    from .sweep import evaluate_members, fit_sweep, pad_members
    if not argv or argv[0] not in ("drvae", "pvae", "vfae"):
        raise SystemExit("usage: python -m drvae_b200.cli sweep {drvae|pvae|vfae} --datafile FILE --rseeds S... --folds F... "
                         "[--yloss-rates R...] [flags]")
    kind = argv.pop(0)
    args = build_sweep_parser(kind).parse_args(argv)
    print(args)
    assert args.data_mode in ['strictC2C'], 'Unsupported data mode'
    assert args.type_y == 'discrete', 'sweep: only type-y discrete is supported'
    assert args.useMF is False, 'use of mol.features not supported'
    assert not (args.useS or args.useMMD), 'sweep: use-s and use-mmd are not supported'
    grid = sweep_grid(kind, args)
    data = {}  # the single-model driver loads the data with its --rseed
    for seed in args.rseeds:
        data[seed] = load_data(args.datafile, seed)
    folds = {(s, f): fold_datasets(kind, args, *data[s], f) for s in args.rseeds for f in args.folds}
    members, datasets = [], []
    for seed, rate, fold, _ in grid:
        train_ds, valid_ds, _ = folds[(seed, fold)]
        hp = dict(yloss_rate=rate, pertloss_rate=0.05 if kind != 'vfae' else 0.,
                  kl_qz2pz2_rate=args.kl_z2_rate if kind == 'pvae' else 1., noise_std=args.noise_var, lr=0.0005,
                  weight_decay=0.05, prior_y=class_prior(kind, args, train_ds))
        members.append(dict(seed=seed, hparams=hp))
        datasets.append((train_ds, valid_ds))
    arch = sweep_arch(kind, args, datasets[0][0].x1.shape[1])
    epochs = args.epochs or (300 if kind == 'drvae' else 1000)
    out = fit_sweep(kind, arch, members, datasets, batch_size=args.batch_size, L=args.L, epochs=epochs,
                    early_stop=args.stopearly, add_noise=args.train_w_noise,
                    anneal_perturb=(1, 0) if kind != 'vfae' else None, sample_seed=args.rseeds[0], log=print)
    plan = out['plan']
    outdir = args.outdir or '.'
    os.makedirs(os.path.join(outdir, 'models'), exist_ok=True)
    os.makedirs(os.path.join(outdir, 'results'), exist_ok=True)
    cls = {'drvae': 'DrVAE', 'pvae': 'PVAE', 'vfae': 'VFAE'}[kind]
    paths = [os.path.join(outdir, 'models', '{}_SD_{}_{}.pth'.format(cls, g[3], args.drug)) for g in grid]
    checkpoint.save_ensemble(plan, paths, out['best'])
    # eval-mode losses are not computed: loss_forward normalises by one N for all members, and padding rows would
    # enter the normalisers of every member with a smaller split
    perfs = {}
    for name, which in (('train', 0), ('valid', 1), ('test', 2)):
        fields, mask, _ = pad_members(kind, [folds[(g[0], g[2])][which] for g in grid])
        perfs[name] = evaluate_members(plan, kind, {k: v.to(plan.device) for k, v in fields.items()}, mask.to(plan.device))
    results = []
    for m, (seed, rate, fold, modelid) in enumerate(grid):
        res = {name: dict(perfs[name][m]) for name in perfs}
        path = os.path.join(outdir, 'results', '{}_SD_all_{}.json'.format(cls, modelid))
        with open(path, 'w') as f:
            json.dump({args.drug: res}, f, indent=1)
        print('wrote', path, '(snapshot at epoch {})'.format(out['snapshot_epoch'][m]))
        results.append(res)
    return results


if __name__ == '__main__':
    main()
