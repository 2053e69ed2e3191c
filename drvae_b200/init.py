"""Parameter initialisation with the reference's RNG consumption order.

The reference seeds the global torch generator in the model constructor (src/DrVAE.py:103-106)
and then builds its blocks (src/DrVAE.py:112-183, src/PVAE.py:106-153, src/VFAE.py:103-165), each
nn.Linear drawing its default init and DiagGaussianModuleLinear drawing W_mu / bias_mu from
U(-1e-4, 1e-4) AFTER its linear_lv (src/blocks.py:332-340).  Creating the same torch modules in
the same order reproduces the reference's initial weights for a given seed and torch version.
"""
from collections import OrderedDict

import torch


def init_state_dict(kind, dim_x, dim_y, dim_z1, dim_z3, enc_z1, dec_x, enc_z3=(), dec_z1=(), seed=12345, weight_norm=False,
                    clf_hidden=(), activation=None):
    """weight_norm=True: every layer except decoder_z2Fz1 is a layers.WeightNormLinear, which adds a `.g`
    vector initialised to ones without consuming random numbers (reference layers.py:17-23).
    clf_hidden (dim_h_clf): the classifier's MLP layers encoder_y.nnet.model.linear{i}, created before its linear_p
    like every other block's MLP (CategoricalDecoder, blocks.py:456-463).
    activation: ignored (the initial weights do not depend on the nonlinearity); accepted so that a Plan's shape
    arguments, activation included, can be passed to both."""
    torch.manual_seed(seed)
    sd = OrderedDict()

    def lin(name, i, o, wn=None):
        m = torch.nn.Linear(i, o)
        sd[name + ".weight"] = m.weight.detach().clone()
        sd[name + ".bias"] = m.bias.detach().clone()
        if weight_norm if wn is None else wn:
            sd[name + ".g"] = torch.ones(o)

    def gauss(prefix, in_dim, hidden, out, second="lv"):
        prev = in_dim
        for i, h in enumerate(hidden):
            lin("%s.nnet.model.linear%d" % (prefix, i + 1), prev, h)
            prev = h
        lin("%s.encoder_mu.linear_mu" % prefix, prev, out)
        lin("%s.encoder_%s.linear_%s" % (prefix, second, second), prev, out)

    def categorical(prefix, in_dim, hidden, out):
        prev = in_dim
        for i, h in enumerate(hidden):
            lin("%s.nnet.model.linear%d" % (prefix, i + 1), prev, h)
            prev = h
        lin(prefix + ".decoder_p.linear_p", prev, out)

    def gauss_linear(prefix, z):
        lin(prefix + ".encoder_lv.linear_lv", z, z, wn=False)
        sd[prefix + ".W_mu"] = torch.Tensor(z, z).uniform_(-0.0001, 0.0001)
        sd[prefix + ".bias_mu"] = torch.Tensor(z).uniform_(-0.0001, 0.0001)

    gauss("encoder_z1", dim_x, enc_z1, dim_z1)
    if kind in ("drvae", "pvae"):
        gauss_linear("decoder_z2Fz1", dim_z1)
    if kind == "drvae":
        categorical("encoder_y", 2 * dim_z1, clf_hidden, dim_y)
        gauss("encoder_z3", dim_z1 + dim_y, enc_z3, dim_z3)
        gauss("decoder_z1", dim_z3 + dim_y, dec_z1, dim_z1)
    elif kind == "vfae":
        categorical("encoder_y", dim_z1, clf_hidden, dim_y)
        gauss("encoder_z2", dim_z1 + dim_y, enc_z3, dim_z3)
        gauss("decoder_z1", dim_z3 + dim_y, dec_z1, dim_z1)
    gauss("decoder_x", dim_z1, dec_x, dim_x, second="sg")
    return sd
