"""DrVAE / PVAE / VFAE: the reference's Python class surface over the B200 kernels.

Constructor signatures, attribute names, state_dict keys and the methods
    forward / predict / reconstruct / transform / loss_function / run_on_batch /
    save_to_file / load_params_from_file / _compute_anneal_coef
mirror the reference classes (src/DrVAE.py:26-331, src/PVAE.py:26-263, src/VFAE.py:26-232 and
the shared mixin src/DGMMixin.py).  The arithmetic of loss_function / run_on_batch / forward is
dispatched through the C ABI (include/drvae_b200.h) to hand-written sm_100a kernels: there is
no autograd graph, no torch.optim and no CPU fallback — `run_on_batch(train_mode=True)` is one
fused forward + ELBO + backward + Adam launch sequence.

Options the reference advertises but that are broken as shipped (SURVEY.md §0 fact 7) or outside
the hot path raise ValueError here instead of failing later: use_s=True, type_rec other than
'diag_gaussian', MMD with use_s, continuous y, clf_1sig, dropout, nonlinearities other than ELU and
softplus, Adamax.  `nonlinearity` is 'elu' (what the run_*.py drivers pass) or 'softplus' (the
constructors' default, nn.Softplus in the reference's table, src/blocks.py:21-24): it is the activation of
every hidden layer, the classifier's included.  The classifier's hidden layers (dim_h_clf, --class-y) are
supported: hidden layers in front of linear_p.
"""
import inspect
import warnings
from collections import OrderedDict

import numpy as np
import torch
import torch.nn as nn

from .init import init_state_dict
from .plan import Plan, anneal_coef, losses_to_dict


class _Node(nn.Module):
    """Anonymous container used to reproduce the reference's dotted parameter names."""


def _as_list(v):
    if v is None:
        return []
    if isinstance(v, (int, np.integer)):
        return [int(v)]
    return [int(x) for x in v]


class _B200Model(nn.Module):
    kind = None

    # ------------------------------------------------------------------------------------------
    def _setup(self, values, enc_top, dim_top):
        for arg, val in values.items():
            setattr(self, arg, val)
        # fixed internals of the reference constructors (DrVAE.py:79-97)
        # the reference hard-codes wn = False before _build_blocks (DrVAE.py:79); layers.WeightNormLinear is reachable
        # there only by editing that line.  Here: a class attribute, e.g. `class DrVAEwn(DrVAE): WN = True`
        self.wn = bool(getattr(type(self), 'WN', False))
        self.bn = False
        self.prior_mu = 0.
        self.prior_sg = 1.
        if self.weight_decay is None:
            self.weight_decay = 0.
        self.kl_min = 2.
        self.anneal_learning_rate = False
        self.anneal_kl = False
        self.anneal_kl_itermax = 100
        self.anneal_yloss = False
        self.anneal_yloss_itermax = 1
        self.finished_training_iters = 0
        self.add_noise = False
        self._eps_tape = None
        self._enc_top, self._dim_top = enc_top, dim_top
        self._check_supported()
        self.nprng = np.random.RandomState(self.random_seed)
        self._build_blocks()
        self._create_optimizer()

    def _check_supported(self):
        def bad(msg):
            raise ValueError("%s: %s is not supported by the B200 hot path (see DESIGN.md, out of scope)"
                             % (type(self).__name__, msg))
        if self.type_rec != 'diag_gaussian':
            bad("type_rec=%r (the reference only ships DiagGaussianSigmaModule)" % (self.type_rec,))
        if self.nonlinearity not in ('elu', 'softplus'):
            bad("nonlinearity=%r (only 'elu' and 'softplus')" % (self.nonlinearity,))
        if self.use_s:
            bad("use_s=True (crashes in the reference, SURVEY.md fact 7)")
        if self.dropout_rate or self.input_x_dropout:
            bad("dropout")
        if self.optim_alg != 'adam':
            bad("optim_alg=%r" % (self.optim_alg,))
        if getattr(self, 'use_c', False) or getattr(self, 'use_m', False):
            bad("use_c / use_m")
        if self.kind != 'pvae':
            if self.type_y != 'discrete':
                bad("type_y=%r" % (self.type_y,))
            if self.clf_1sig:
                bad("clf_1sig")
            if self.kind == 'drvae' and not self.clf_z1z2:
                bad("clf_z1z2=False")
            if self.kind == 'vfae' and not self.semi_supervised:
                bad("semi_supervised=False")
            if self.prior_y is not None and not isinstance(self.prior_y, str):
                assert isinstance(self.prior_y, np.ndarray) and len(self.prior_y) == self.dim_y

    def _build_blocks(self):
        """Allocate the flat parameter vector (reference state_dict layout), initialise it with the
        reference's RNG order and expose it as nn.Parameters that alias the kernel's memory."""
        arch = dict(dim_x=self.dim_x, dim_y=self.dim_y, dim_z1=self.dim_z1, dim_z3=self._dim_top,
                    enc_z1=_as_list(self.dim_h_en_z1), dec_x=_as_list(self.dim_h_de_x),
                    enc_z3=self._enc_top, dec_z1=_as_list(getattr(self, 'dim_h_de_z1', [])))
        if self.kind != 'pvae':
            arch['clf_hidden'] = _as_list(self.dim_h_clf)
        self._arch = arch
        self.plan = Plan(self.kind, L=self.L, max_batch=max(int(self.batch_size), 1), n_models=1,
                         weight_norm=self.wn, activation=self.nonlinearity, **arch)
        self._max_batch = self.plan.Ncap
        sd = init_state_dict(self.kind, seed=self.random_seed, weight_norm=self.wn, **arch)
        self.plan.load_state_dict(sd)
        for name, view in self.plan.tensor_views(self.plan.params, 0).items():
            parts = name.split('.')
            node = self
            for p in parts[:-1]:
                if not hasattr(node, p):
                    node.add_module(p, _Node())
                node = getattr(node, p)
            node.register_parameter(parts[-1], nn.Parameter(view, requires_grad=False))

    def _create_optimizer(self):
        """Adam is fused into the step (DGMMixin._create_optimizer creates torch.optim.Adam with the
        same lr / weight_decay, src/DGMMixin.py:31-40); moments live in plan.adam_m / plan.adam_v."""
        if self.optim_alg != 'adam':
            raise ValueError('Selected unknown optimizer: ' + self.optim_alg)
        self.optimizer = None

    def _ensure_capacity(self, n):
        if n > self._max_batch:
            # re-plan with a larger row capacity, keeping parameters and optimizer state
            old = self.plan
            self.plan = Plan(self.kind, L=self.L, max_batch=int(n), n_models=1, weight_norm=self.wn,
                             activation=old.activation, **self._arch)
            self.plan.params.copy_(old.params)
            self.plan.adam_m.copy_(old.adam_m)
            self.plan.adam_v.copy_(old.adam_v)
            self._max_batch = self.plan.Ncap
            for name, view in self.plan.tensor_views(self.plan.params, 0).items():
                node = self
                parts = name.split('.')
                for p in parts[:-1]:
                    node = getattr(node, p)
                getattr(node, parts[-1]).data = view
            self.plan.sync_shadows()

    # ------------------------------------------------------------------------------------------
    def w2log(self, *args):
        print(*args)
        if self.log_txt is not None:
            import os
            os.makedirs('logs', exist_ok=True)
            with open('logs/' + self.log_txt, 'a') as f:
                f.write(' '.join(str(e) for e in args) + '\n')

    def _compute_anneal_coef(self, iter_num, iter_max=1000, iter_offset=0, func_type='linear'):
        if func_type != 'linear':
            raise ValueError("Unknown annealing function: " + func_type)
        return anneal_coef(iter_num, iter_max, iter_offset)

    def set_eps_tape(self, draws):
        """Parity hook: the next loss / step consumes these normals (reference draw order, SURVEY.md
        Appendix B) instead of Philox noise."""
        self._eps_tape = list(draws) if draws is not None else None

    def load_state_dict(self, state_dict, strict=True):
        res = super().load_state_dict(state_dict, strict=strict)
        self.plan.sync_shadows()
        return res

    def sync(self):
        """Call after writing to parameters directly: refreshes the kernels' bf16 weight copies."""
        self.plan.sync_shadows()

    def save_to_file(self, filename):
        # parameters alias the kernels' flat vector (16-byte aligned rows): save compact copies, reference shapes
        torch.save(OrderedDict((k, v.detach().contiguous().cpu()) for k, v in self.state_dict().items()), filename)

    def load_params_from_file(self, filename):
        self.load_state_dict(torch.load(filename))

    # ------------------------------------------------------------------------------------------
    def _beta_pert(self):
        if getattr(self, 'anneal_perturb_rate_itermax', 0) > 0:
            return self._compute_anneal_coef(self.finished_training_iters, iter_max=self.anneal_perturb_rate_itermax,
                                             iter_offset=self.anneal_perturb_rate_offset)
        return 1.

    def _hparams(self, training):
        # the reference honours these attributes inside run_on_batch / loss_function (DGMMixin.py:100-104,
        # DrVAE.py:549-557); no shipped driver sets them and the kernels do not implement them: refuse rather than
        # train differently in silence
        for flag in ('anneal_learning_rate', 'anneal_kl', 'anneal_yloss'):
            if getattr(self, flag, False):
                raise ValueError("%s: %s=True is not supported by the B200 hot path" % (type(self).__name__, flag))
        prior = None
        if self.kind != 'pvae' and not isinstance(self.prior_y, str) and self.prior_y is not None:
            prior = [float(p) for p in self.prior_y]
        return self.plan.hparams(
            step=self.finished_training_iters, training=training, add_noise=bool(self.add_noise),
            noise_std=float(self.add_noise_var), beta_pert=self._beta_pert(),
            pertloss_rate=float(getattr(self, 'pertloss_rate', 0.)),
            kl_qz2pz2_rate=float(getattr(self, 'kl_qz2pz2_rate', 1.)),
            yloss_rate=float(getattr(self, 'yloss_rate', 0.)), kl_min=self.kl_min, lr=float(self.learning_rate),
            weight_decay=float(self.weight_decay), prior_y=prior)

    def _batch_kwargs(self, x1, x2=None, y=None, has_x2=None, has_y=None):
        b = dict(x1=x1)
        if self.kind in ('drvae', 'pvae'):
            b.update(x2=x2, has_x2=has_x2)
        if self.kind in ('drvae', 'vfae'):
            b.update(y=y, has_y=has_y)
        return b

    def _group_warnings(self, has_x2, has_y):
        """The reference warns about empty row groups (DrVAE.py:588-607); kept for callers that rely on it."""
        if self.kind == 'drvae':
            hx, hy = has_x2.bool().cpu(), has_y.bool().cpu()
            for mask, name in (((hy & ~hx), "Labeled Singleton"), ((~hy & ~hx), "Unlabeled Singleton"),
                               ((hy & hx), "Labeled Paired perturbation"), ((~hy & hx), "Unlabeled Paired perturbation")):
                if int(mask.sum()) == 0:
                    warnings.warn("No %s data in the minibatch" % name)

    def _eps_for(self, batch, training):
        if self._eps_tape is None:
            return None
        from .noise import eps_block_from_tape
        hx = batch.get('has_x2')
        hy = batch.get('has_y')
        eps = eps_block_from_tape(self.plan, self._eps_tape, hx.cpu() if hx is not None else None,
                                  hy.cpu() if hy is not None else None, noisy=bool(training and self.add_noise))
        self._eps_tape = None
        return eps

    def _losses(self, fn_name, batch, training):
        n = batch['x1'].shape[0]
        self._ensure_capacity(n)  # may replace self.plan: resolve the entry point afterwards
        fn = getattr(self.plan, fn_name)
        eps = self._eps_for(batch, training)
        seed = (int(self.random_seed) << 20) ^ 0x5DEECE66D
        out = fn(batch, self._hparams(training), eps=eps, seed=seed)
        return losses_to_dict(self.kind, out[0].clone())

    def run_on_batch(self, train_mode=False, **kwargs):
        """DGMMixin.run_on_batch (src/DGMMixin.py:91-126): one optimisation step (train_mode) or an
        eval-mode loss evaluation.  Returns the reference's OrderedDict of 0-dim tensors."""
        kwargs.pop('s', None)
        batch = self._batch_kwargs(**kwargs)
        if train_mode:
            self.train()
            losses = self._losses('train_step', batch, True)
            self.finished_training_iters += 1
        else:
            self.eval()
            losses = self._losses('loss_forward', batch, False)
        return losses

    def _loss_function(self, **kwargs):
        kwargs.pop('s', None)
        return self._losses('loss_forward', self._batch_kwargs(**kwargs), bool(self.training))

    # ------------------------------------------------------------------------------------------
    # training-loop surface (reference fit / evaluate_performance*; see drvae_b200/training.py)
    def fit(self, train_loader, valid_loader, add_noise=False, verbose=False, early_stop=False,
            model_filename='best_model.pth'):
        from . import training
        return training.fit(self, train_loader, valid_loader, add_noise=add_noise, verbose=verbose,
                            early_stop=early_stop, model_filename=model_filename)

    def evaluate_performance(self, return_full_data=False, **batch):
        from . import training
        return training.evaluate_performance(self, return_full_data=return_full_data, **batch)

    def evaluate_performance_on_dataset(self, ds, return_full_data=False):
        from . import training
        return training.evaluate_performance_on_dataset(self, ds, return_full_data=return_full_data)

    def eval_x_reconstruction(self, x, x_rec, x_rec_sigma=None):
        from . import training
        return training.eval_x_reconstruction(x, x_rec, x_rec_sigma)

    def eval_y_prediction(self, pred, proba, ylab):
        from . import training
        return training.eval_y_prediction(pred, proba, ylab, self.dim_y)

    # ------------------------------------------------------------------------------------------
    def _infer(self, x1):
        self.eval()  # as the reference's forward() does (DrVAE.py:262, PVAE.py:214, VFAE.py:186)
        self._ensure_capacity(x1.shape[0])
        r = self.plan.infer(x1)
        return {k: v[0] for k, v in r.items()}


class DrVAE(_B200Model):
    """Drug Response Variational Autoencoder (reference src/DrVAE.py:26-877)."""
    kind = 'drvae'

    def __init__(self, dim_x, dim_s, dim_y, dim_c=1, dim_m=1,
                 dim_h_en_z1=(50, 50), dim_h_de_z1=(50, 50), dim_h_en_z2Fz1=(50), dim_h_en_z3=(50, 50),
                 dim_h_de_x=(50, 50), dim_h_clf=(50, 50), dim_z1=50, dim_z3=50, type_rec='binary',
                 clf_z1z2=True, type_y='discrete', prior_y='uniform', clf_1sig=False,
                 epochs=500, batch_size=100, nonlinearity='softplus',
                 learning_rate=0.001, optim_alg='adam', L=1, weight_decay=None,
                 dropout_rate=0., input_x_dropout=0., add_noise_var=0.,
                 yloss_rate=1., anneal_yloss_offset=0,
                 use_MMD=True, kernel_MMD='rbf_fourier', mmd_rate=1.,
                 kl_qz2pz2_rate=1., pertloss_rate=0.1, anneal_perturb_rate_itermax=1, anneal_perturb_rate_offset=0,
                 use_s=False, use_c=False, use_m=False,
                 random_seed=12345, log_txt=None):
        super(DrVAE, self).__init__()
        _, _, _, values = inspect.getargvalues(inspect.currentframe())
        values.pop('self')
        values.pop('__class__', None)
        self.dim_z2 = dim_z1
        self._setup(values, _as_list(dim_h_en_z3), dim_z3)

    def loss_function(self, x1, x2, s, y, has_x2, has_y):
        self._group_warnings(has_x2, has_y)
        return self._loss_function(x1=x1, x2=x2, y=y, has_x2=has_x2, has_y=has_y)

    def forward(self, x1, s=[]):
        r = self._infer(x1)
        return {'pred': r['pred'].long(), 'proba': r['proba'], 'z1': r['z1_mu'], 'qz1': (r['z1_mu'], r['z1_lv']),
                'px1': (r['px1_mu'], r['px1_sg']), 'x1_rec': r['px1_mu'], 'z2': r['z2_mu'],
                'pz2': (r['z2_mu'], r['z2_lv']), 'px2': (r['px2_mu'], r['px2_sg']), 'x2_pert': r['px2_mu']}

    def predict(self, **kwargs):
        res = self.forward(**kwargs)
        return res['pred'].cpu().numpy().squeeze(), res['proba'].cpu().numpy()

    def reconstruct(self, **kwargs):
        res = self.forward(**kwargs)
        return (res['x1_rec'].cpu().numpy(), [t.cpu().numpy() for t in res['px1']],
                res['x2_pert'].cpu().numpy(), [t.cpu().numpy() for t in res['px2']])

    def transform(self, **kwargs):
        res = self.forward(**kwargs)
        return res['z1'].cpu().numpy(), res['z2'].cpu().numpy()


class PVAE(_B200Model):
    """Perturbation VAE (reference src/PVAE.py:26-671)."""
    kind = 'pvae'
    prior_y = None  # the reference constructor reads this attribute without ever setting it (PVAE.py:77)

    def __init__(self, dim_x, dim_s, dim_y, dim_c=1, dim_m=1,
                 dim_h_en_z1=(50, 50), dim_h_en_z2Fz1=(50), dim_h_de_x=(50, 50), dim_z1=50, type_rec='binary',
                 epochs=500, batch_size=100, nonlinearity='softplus',
                 learning_rate=0.001, optim_alg='adam', L=1, weight_decay=None,
                 dropout_rate=0., input_x_dropout=0., add_noise_var=0.,
                 use_MMD=True, kernel_MMD='rbf_fourier', mmd_rate=1.,
                 kl_qz2pz2_rate=1., pertloss_rate=0.1, anneal_perturb_rate_itermax=1, anneal_perturb_rate_offset=0,
                 use_s=False, use_c=False, use_m=False,
                 random_seed=12345, log_txt=None):
        super(PVAE, self).__init__()
        _, _, _, values = inspect.getargvalues(inspect.currentframe())
        values.pop('self')
        values.pop('__class__', None)
        self.dim_z2 = dim_z1
        self._setup(values, [], 1)

    def loss_function(self, x1, x2, s, has_x2):
        return self._loss_function(x1=x1, x2=x2, has_x2=has_x2)

    def forward(self, x1, s=[]):
        r = self._infer(x1)
        return {'z1': r['z1_mu'], 'qz1': (r['z1_mu'], r['z1_lv']), 'px1': (r['px1_mu'], r['px1_sg']),
                'x1_rec': r['px1_mu'], 'z2': r['z2_mu'], 'pz2': (r['z2_mu'], r['z2_lv']),
                'px2': (r['px2_mu'], r['px2_sg']), 'x2_pert': r['px2_mu']}

    def predict(self, **kwargs):
        raise NotImplementedError("This is not a classification model")

    def reconstruct(self, **kwargs):
        res = self.forward(**kwargs)
        return (res['x1_rec'].cpu().numpy(), [t.cpu().numpy() for t in res['px1']],
                res['x2_pert'].cpu().numpy(), [t.cpu().numpy() for t in res['px2']])

    def transform(self, **kwargs):
        res = self.forward(**kwargs)
        return res['z1'].cpu().numpy(), res['z2'].cpu().numpy()


class VFAE(_B200Model):
    """Variational Fair Autoencoder in SSVAE mode (reference src/VFAE.py:26-655)."""
    kind = 'vfae'

    def __init__(self, dim_x, dim_s, dim_y,
                 dim_h_en_z1=(50, 50), dim_h_de_z1=(50, 50), dim_h_en_z2=(50, 50), dim_h_de_x=(50, 50),
                 dim_h_clf=(50, 50), dim_z1=50, dim_z2=50, type_rec='binary',
                 type_y='discrete', prior_y='uniform', semi_supervised=False, clf_1sig=False,
                 epochs=500, batch_size=100, nonlinearity='softplus',
                 learning_rate=0.001, optim_alg='adam', L=1, weight_decay=None,
                 dropout_rate=0., input_x_dropout=0., add_noise_var=0.,
                 yloss_rate=1., anneal_yloss_offset=0,
                 use_MMD=True, kernel_MMD='rbf_fourier', mmd_rate=1., use_s=False,
                 random_seed=12345, log_txt=None):
        super(VFAE, self).__init__()
        _, _, _, values = inspect.getargvalues(inspect.currentframe())
        values.pop('self')
        values.pop('__class__', None)
        self._setup(values, _as_list(dim_h_en_z2), dim_z2)

    def loss_function(self, x1, s, y, has_y):
        return self._loss_function(x1=x1, y=y, has_y=has_y)

    def forward(self, x1, s=[]):
        r = self._infer(x1)
        return {'pred': r['pred'].long(), 'proba': r['proba'], 'z1': r['z1_mu'], 'qz1': (r['z1_mu'], r['z1_lv']),
                'px1': (r['px1_mu'], r['px1_sg']), 'x1_rec': r['px1_mu']}

    def predict(self, **kwargs):
        res = self.forward(**kwargs)
        return res['pred'].cpu().numpy().squeeze(), res['proba'].cpu().numpy()

    def reconstruct(self, **kwargs):
        res = self.forward(**kwargs)
        return res['x1_rec'].cpu().numpy(), [t.cpu().numpy() for t in res['px1']]

    def transform(self, **kwargs):
        res = self.forward(**kwargs)
        return res['z1'].cpu().numpy()
