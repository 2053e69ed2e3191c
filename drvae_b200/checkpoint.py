"""Checkpoint interchange for ensembles (SURVEY.md §8(f) rank 3; reference: DGMMixin.save_to_file /
load_params_from_file, src/DGMMixin.py:192-203 — `torch.save(self.state_dict())` per model).

An ensemble plan holds n_models parameter vectors in ONE device buffer.  Saving copies that buffer to the host once and
cuts it into per-member state_dicts with the reference's keys, order and shapes, so every member's file loads into the
reference's own classes (and back).  `save_resume` / `load_resume` add what the reference never persists — Adam moments
and the step counter — so that a run continues bit-exactly.
"""
import os
from collections import OrderedDict

import torch


def _host_views(plan, flat_cpu, model):
    out = OrderedDict()
    for (name, r, c, off), ld in zip(plan.tensors, plan.tensor_ld):
        if c > 0:
            out[name] = flat_cpu[model, off:off + r * ld].view(r, ld)[:, :c].clone(memory_format=torch.contiguous_format)
        else:
            out[name] = flat_cpu[model, off:off + r].clone()
    return out


def state_dicts(plan, params=None):
    """-> [state_dict of member 0, ..., n_models - 1] (CPU tensors, reference layout); one device->host copy.
    params: an [n_models, param_count] buffer in the plan's layout to read instead of plan.params (e.g. snapshots)."""
    flat = (plan.params if params is None else params).detach().cpu()
    return [_host_views(plan, flat, m) for m in range(plan.E)]


def save_ensemble(plan, pattern, params=None):
    """One reference-compatible .pth per member: pattern.format(i), e.g. 'models/drug{:03d}.pth', or the i-th entry of
    a list of paths.  params: as in state_dicts.  Returns the paths."""
    paths = []
    for m, sd in enumerate(state_dicts(plan, params)):
        path = pattern[m] if isinstance(pattern, (list, tuple)) else pattern.format(m)
        d = os.path.dirname(path)
        if d:
            os.makedirs(d, exist_ok=True)
        torch.save(sd, path)
        paths.append(path)
    return paths


def load_ensemble(plan, paths_or_dicts, strict=True):
    """Load one state_dict (path or mapping) per member; assembled on the host, ONE host->device copy, ONE shadow refresh."""
    if len(paths_or_dicts) != plan.E:
        raise ValueError("need %d state_dicts, got %d" % (plan.E, len(paths_or_dicts)))
    flat = plan.params.detach().cpu()
    for m, src in enumerate(paths_or_dicts):
        sd = torch.load(src, map_location="cpu") if isinstance(src, (str, os.PathLike)) else src
        names = [t[0] for t in plan.tensors]
        missing = [k for k in names if k not in sd]
        extra = [k for k in sd if k not in names]
        if strict and (missing or extra):
            raise KeyError("member %d: state_dict mismatch: missing %s unexpected %s" % (m, missing, extra))
        for (name, r, c, off), ld in zip(plan.tensors, plan.tensor_ld):
            if name not in sd:
                continue
            t = sd[name].detach().to(torch.float32).cpu()
            want = (r, c) if c > 0 else (r,)
            if tuple(t.shape) != want:
                raise ValueError("member %d: shape mismatch for %s: %s vs %s" % (m, name, tuple(t.shape), want))
            if c > 0:
                flat[m, off:off + r * ld].view(r, ld)[:, :c].copy_(t)
            else:
                flat[m, off:off + r].copy_(t)
    plan.params.copy_(flat)
    plan.sync_shadows()


def save_resume(plan, path, step):
    """Parameters + Adam moments + step of every member in one file (flat device layout; not a reference format)."""
    torch.save({"format": "drvae_b200.resume.v1", "kind": plan.kind, "n_models": plan.E, "param_count": plan.P, "step": int(step),
                "tensors": [(n, r, c, off, ld) for (n, r, c, off), ld in zip(plan.tensors, plan.tensor_ld)],
                "params": plan.params.detach().cpu(), "adam_m": plan.adam_m.detach().cpu(), "adam_v": plan.adam_v.detach().cpu()}, path)


def load_resume(plan, path):
    """-> step.  The plan must have the architecture the file was written from."""
    d = torch.load(path, map_location="cpu")
    if d.get("format") != "drvae_b200.resume.v1":
        raise ValueError("%s is not a drvae_b200 resume file" % path)
    if d["n_models"] != plan.E or d["param_count"] != plan.P or d["kind"] != plan.kind:
        raise ValueError("resume file does not match the plan (kind / n_models / parameter layout)")
    plan.params.copy_(d["params"])
    plan.adam_m.copy_(d["adam_m"])
    plan.adam_v.copy_(d["adam_v"])
    plan.sync_shadows()
    return int(d["step"])
