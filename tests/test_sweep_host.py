"""Host-side checks of the member-hyperparameter table and the sweep driver: struct layout, the `cli sweep` grid,
padding of per-member splits, and the early-stopping rule shared by training.fit and sweep.fit_sweep."""
import ctypes
import os
import re

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_member_hparams_struct_matches_header():
    from drvae_b200 import _lib
    hdr = open(os.path.join(ROOT, "include", "drvae_b200.h")).read()
    body = re.search(r"typedef struct \{([^}]*)\} drvae_member_hparams_t;", hdr).group(1)
    names = re.findall(r"(\w+)(?:\[\d+\])?\s*[,;]", body)
    assert [f[0] for f in _lib.MemberHParams._fields_] == names
    assert ctypes.sizeof(_lib.MemberHParams) == 4 * (6 + 8)
    assert "drvae_set_member_hparams" in _lib.EXPORTS


def _reference_rule(objectives, kind, epochs, early_stop, min_patience=None):
    """The rule as training.fit wrote it inline before it became training.SnapshotRule."""
    patience = min_patience if min_patience is not None else (40 if kind == "vfae" else 50)
    best, rolling, since, snapshotted = -np.inf, [], 0, False
    snaps, stops = [], []
    for epoch, vobj in enumerate(objectives, 1):
        since += 1
        rolling = (rolling + [vobj])[-3:]
        cur = float(np.mean(rolling))
        if cur * 0.999 > best:
            patience = max(patience, epoch + 15)
            best, since = cur, 0
        if (early_stop and since == 0) or (patience <= epoch and not snapshotted):
            snapshotted = True
            snaps.append(epoch)
        if patience <= epoch:
            stops.append(epoch)
            if early_stop:
                break
            patience, snapshotted = epochs + 1, False
    return snaps, stops


@pytest.mark.parametrize("early_stop", [False, True])
@pytest.mark.parametrize("kind,min_patience", [("drvae", None), ("vfae", None), ("pvae", 4)])
def test_snapshot_rule_matches_the_reference_rule(kind, min_patience, early_stop):
    from drvae_b200.training import SnapshotRule
    rng = np.random.RandomState(3)
    epochs = 120
    scripts = [
        np.linspace(0.5, 2.0, epochs),                                        # improves every epoch
        np.concatenate([np.linspace(0.5, 2.0, 20), np.full(epochs - 20, 1.0)]),  # peaks, then drops: patience runs out
        np.concatenate([np.linspace(0.5, 1.0, 10), np.full(60, 0.9), np.linspace(0.9, 3.0, epochs - 70)]),  # late recovery
        rng.rand(epochs),
    ]
    for objectives in scripts:
        want_snaps, want_stops = _reference_rule(list(objectives), kind, epochs, early_stop, min_patience)
        rule = SnapshotRule(kind, epochs, early_stop, min_patience)
        snaps, stops = [], []
        for epoch, v in enumerate(objectives, 1):
            snapshot, reached, stop = rule.update(epoch, float(v))
            if snapshot:
                snaps.append(epoch)
            if reached:
                stops.append(epoch)
            if stop:
                break
        assert (snaps, stops) == (want_snaps, want_stops)
    # the "continue after patience" branch is exercised: without early stopping the second script reaches patience,
    # snapshots once and trains on
    if not early_stop:
        snaps, stops = _reference_rule(list(scripts[1]), kind, epochs, False, min_patience)
        assert len(stops) == 1 and stops[0] < epochs and snaps == stops


def _ds(n, dim_x=6, seed=0):
    from drvae_b200.training import DrVAEDataset
    g = torch.Generator().manual_seed(seed)
    return DrVAEDataset(x1=torch.randn(n, dim_x, generator=g), x2=torch.randn(n, dim_x, generator=g),
                        s=torch.zeros(n, dtype=torch.int32), y=torch.arange(n) % 2,
                        has_x2=(torch.arange(n) % 2).to(torch.int32), has_y=torch.ones(n, dtype=torch.int32))


def test_pad_members_and_mask():
    from drvae_b200.sweep import pad_members, steps_per_epoch
    a, b = _ds(3, seed=1), _ds(5, seed=2)
    fields, mask, sizes = pad_members("drvae", [a, b])
    assert sizes == [3, 5]
    assert fields["x1"].shape == (2, 5, 6) and fields["x1"].dtype == torch.float32
    assert fields["y"].dtype == torch.int32 and fields["has_x2"].shape == (2, 5)
    assert torch.equal(mask, torch.tensor([[1, 1, 1, 0, 0], [1, 1, 1, 1, 1]], dtype=torch.int32))
    assert torch.equal(fields["x1"][0, :3], a.x1) and torch.equal(fields["x1"][1], b.x1)
    assert not fields["x1"][0, 3:].any() and not fields["has_y"][0, 3:].any()
    assert set(pad_members("vfae", [a, b])[0]) == {"x1", "y", "has_y"}
    assert set(pad_members("pvae", [a, b])[0]) == {"x1", "x2", "has_x2"}
    assert steps_per_epoch([3, 5], 2) == 2 and steps_per_epoch([3, 5], 8) == 1 and steps_per_epoch([450, 200], 200) == 2


def test_sweep_parser_grid_and_per_fold_prior():
    from drvae_b200 import cli
    args = cli.build_sweep_parser("drvae").parse_args(
        "--datafile synthetic:300 --rseeds 7 8 --folds 1 2 --yloss-rates 10 50 --clf-dataprior --L 2".split())
    assert args.modelid == "auto" and args.batch_size == 200 and args.yloss_rate == 50.
    grid = cli.sweep_grid("drvae", args)
    assert len(grid) == 8
    assert grid[0] == (7, 10., 1, "RS7_L2_YR10.0_FOLD1")
    assert [g[3] for g in grid][-1] == "RS8_L2_YR50.0_FOLD2"
    # default rate axis: the single --yloss-rate; PVAE has no rate axis
    a2 = cli.build_sweep_parser("vfae").parse_args("--datafile synthetic --rseeds 1 --folds 3".split())
    assert [g[3] for g in cli.sweep_grid("vfae", a2)] == ["RS1_L1_YR50.0_FOLD3"]
    a3 = cli.build_sweep_parser("pvae").parse_args("--datafile synthetic --rseeds 1 2 --folds 1".split())
    assert [g[3] for g in cli.sweep_grid("pvae", a3)] == ["RS1_L1_YR0_FOLD1", "RS2_L1_YR0_FOLD1"]
    with pytest.raises(SystemExit):
        cli.build_sweep_parser("drvae").parse_args("--datafile synthetic --folds 1".split())
    # --clf-dataprior: the class frequencies of each fold's labeled training rows, as the single-model driver computes
    sing, pair = cli.load_data("synthetic:300", 7)
    priors = []
    for fold in (1, 2):
        train_ds = cli.fold_datasets("drvae", args, sing, pair, fold)[0]
        lab = train_ds.y[train_ds.has_y != 0].long().numpy()
        want = np.bincount(lab, minlength=2) / len(lab)
        got = cli.class_prior("drvae", args, train_ds)
        assert np.allclose(got, want) and abs(sum(got) - 1) < 1e-12
        priors.append(got)
    assert priors[0] != priors[1]
    args.clf_dataprior = False
    assert cli.class_prior("drvae", args, train_ds) == [0.5, 0.5]


def test_single_model_parser_is_unchanged_by_the_sweep_parser():
    from drvae_b200 import cli
    cli.build_sweep_parser("drvae")
    with pytest.raises(SystemExit):  # --modelid stays required for the single-model driver
        cli.build_parser("drvae").parse_args(["--datafile", "x.npz"])
