"""Generate tests/golden/*.npz from the REFERENCE ITSELF and pin the oracle against it.

Run in the build container only (needs /root/reference):  python -m oracle.make_golden
For each model family and two architectures (TINY, README) the unmodified reference classes are
constructed with random_seed=123, fed the synthetic batch of SURVEY.md §8(d) and an ε tape drawn
from torch.Generator().manual_seed(777 + step), and stepped twice with run_on_batch
(step 0: beta_pert = 0.01, step 1: beta_pert = 1).  Recorded per step: all loss terms, gradients
(full for TINY, norms + strided samples for README), and for the initial weights the inference
outputs of forward().  Before anything is written, oracle/drvae_oracle.py is run on the same
inputs and must agree with the reference to <= 1e-5 relative (losses) / 1e-4 (gradients).
"""
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle import drvae_oracle as orc  # noqa: E402
from oracle import ref_harness as rh  # noqa: E402

README = dict(dim_x=978, dim_y=2, dim_z1=100, dim_z3=100, dim_z2=100, enc_z1=[800], dec_x=[600], enc_z3=[200],
              enc_z2=[200], dec_z1=[200])
TINY = dict(dim_x=40, dim_y=2, dim_z1=12, dim_z3=10, dim_z2=10, enc_z1=[24], dec_x=[28], enc_z3=[20], enc_z2=[20],
            dec_z1=[18])
DEEP = dict(dim_x=40, dim_y=2, dim_z1=12, dim_z3=10, dim_z2=10, enc_z1=[24, 20], dec_x=[16, 28], enc_z3=[20, 12],
            enc_z2=[20, 12], dec_z1=[18, 14])
# (name, architecture, rows, weight_norm, model kinds)
ALL = ("drvae", "pvae", "vfae")
CASES = [("tiny", TINY, 24, False, ALL), ("deep", DEEP, 24, False, ALL), ("readme", README, 150, False, ALL),
         ("tiny_wn", TINY, 24, True, ALL),
         # the shapes bench.py times: README architecture with weight norm, and the 8192-row minibatch of BASELINE configs[3]
         ("readme_wn", README, 150, True, ALL), ("readme8192", README, 8192, False, ("drvae", "vfae"))]
SEED_MODEL, SEED_TAPE, L = 123, 777, 2
SAMPLE = 257


def rel(a, b):
    return abs(a - b) / (abs(a) + 1e-12)


def main():
    out_dir = os.path.join(ROOT, "tests", "golden")
    os.makedirs(out_dir, exist_ok=True)
    torch.set_num_threads(4)
    only = sys.argv[1:]
    for cname, arch, N, wn, kinds in CASES:
        if only and cname not in only:
            continue
        for kind in kinds:
            model = rh.build_reference_model(kind, arch, seed=SEED_MODEL, L=L, weight_norm=wn)
            if wn:
                # g is initialised to exactly 1 (layers.py:22): perturb it reproducibly so the g/||v|| scale and its
                # gradient are exercised away from the trivial point
                gg = torch.Generator().manual_seed(99)
                with torch.no_grad():
                    for k, prm in model.named_parameters():
                        if k.endswith(".g"):
                            prm.mul_(1.0 + 0.2 * torch.randn(prm.shape, generator=gg))
            sd0 = {k: v.detach().clone() for k, v in model.state_dict().items()}
            batch = orc.synthetic_batch(N, arch["dim_x"])
            cfg = orc.default_cfg(kind, L=L)
            om = orc.OracleModel(sd0, cfg)
            full = not cname.startswith("readme")
            rec = {}
            rec["meta/N"] = np.array(N)
            rec["meta/L"] = np.array(L)
            for k, v in sd0.items():
                a = v.numpy()
                rec["sdsum/" + k] = np.array([a.sum(dtype=np.float64), np.abs(a).sum(dtype=np.float64)])
                if full or k.endswith(".g"):  # (the perturbed g vectors are small: kept so that tests can rebuild the weights)
                    rec["sd/" + k] = a
            # inference on the initial weights
            fw = rh.reference_forward(model, batch["x1"])
            fo = om.forward(batch["x1"])
            for key in ("pred", "proba", "z1", "z2", "x1_rec", "x2_pert"):
                if key in fw:
                    r = fw[key].detach().numpy()
                    o = fo[key].numpy()
                    assert np.allclose(r, o, rtol=1e-4, atol=1e-5), (cname, kind, key)
                    # README shapes: the first 1024 rows x 8 columns (keeps the 8192-row fixture under 1 MB)
                    rec["fwd/" + key] = r if (full or key in ("pred", "proba")) else r[:1024, :8]
            # eval-mode loss (no noise draws, no update)
            le, draws_e = rh.reference_step(model, kind, batch, SEED_TAPE + 100, train=False)
            lo = om.loss(batch, orc.Tape(recorded=draws_e), train=False)
            for k in le:
                assert rel(le[k], float(lo[k])) < 1e-5, (cname, kind, "eval", k, le[k], float(lo[k]))
                rec["loss_eval/" + k] = np.array(le[k])
            rec["meta/eval_draws"] = np.array(len(draws_e))
            # two training steps
            for it in range(2):
                lr_, draws = rh.reference_step(model, kind, batch, SEED_TAPE + it, train=True)
                gr = rh.reference_grads(model)
                lo = om.step(batch, orc.Tape(seed=SEED_TAPE + it))  # the oracle draws its own tape: order is pinned
                for k in lr_:
                    assert rel(lr_[k], float(lo[k])) < 1e-5, (cname, kind, it, k, lr_[k], float(lo[k]))
                    rec["loss_train%d/%s" % (it, k)] = np.array(lr_[k])
                rec["meta/draws%d" % it] = np.array([len(draws), sum(d.numel() for d in draws)])
                if it == 0:
                    for k, g in gr.items():
                        go = om.sd[k].grad
                        e = ((g - go).abs().max() / (g.abs().max() + 1e-12)).item()
                        assert e < 1e-4, (cname, kind, "grad", k, e)
                        a = g.numpy()
                        rec["gradnorm0/" + k] = np.array(np.sqrt((a.astype(np.float64) ** 2).sum()))
                        if full:
                            rec["grad0/" + k] = a
                        else:
                            flat = a.reshape(-1)
                            stride = max(1, flat.size // SAMPLE)
                            rec["gradsample0/" + k] = flat[::stride][:SAMPLE].copy()
                            rec["gradstride0/" + k] = np.array(stride)
                    if full:
                        for i, d in enumerate(draws):
                            rec["tape0/%03d" % i] = d.numpy()
                        for k, v in model.state_dict().items():
                            rec["sd_after1/" + k] = v.detach().numpy().copy()
            if full:
                for k, v in batch.items():
                    rec["batch/" + k] = v.numpy()
            path = os.path.join(out_dir, "%s_%s.npz" % (kind, cname))
            np.savez_compressed(path, **rec)
            print("wrote", path, os.path.getsize(path) // 1024, "KiB", {k: round(float(v), 4) for k, v in lr_.items()})


if __name__ == "__main__":
    main()
