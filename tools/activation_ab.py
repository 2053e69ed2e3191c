"""A/B timing of the hidden-layer activation on the 32-member README DrVAE ensemble step (bench.py's default workload).

Variants, alternated within ONE GPU session, each in its own process, `--repeats` times:
  parent     the previous commit's package and library: its Python package (a copy of its drvae_b200/ directory)
             under --parent-tree, its library through DRVAE_B200_LIB (build it in a worktree of that commit with
             `python -m drvae_b200.build`; no GPU needed)
  elu        this build, the default activation (ELU)
  softplus   this build, Plan(activation="softplus")
Every variant runs the same seeded steps; each run prints a hash of its last step's [32, 8] losses and of the parameters,
and the summary says whether the ELU variant's equal the parent's bit for bit.  Prints the card name and power limit,
then one JSON line per run and a summary (median ms/step per variant).

  python tools/activation_ab.py --parent-lib drvae_b200/lib/libdrvae_b200_parent.so \\
      --parent-tree drvae_b200/lib/parent_tree --out profiles/activation_ab.txt
"""
import argparse
import functools
import hashlib
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
VARIANTS = {"parent": None, "elu": "elu", "softplus": "softplus"}


def child(variant, steps, warmup, tree):
    sys.path.insert(0, ROOT)
    import torch
    import bench  # puts ROOT on sys.path; the parent's package must come before it
    if tree:
        assert "drvae_b200" not in sys.modules
        sys.path.insert(0, os.path.abspath(tree))
    import drvae_b200
    assert os.path.dirname(os.path.dirname(os.path.abspath(drvae_b200.__file__))) == os.path.abspath(tree or ROOT)
    act = VARIANTS[variant]
    if act == "softplus":
        # bench.build_ensemble imports Plan from this module when called
        import drvae_b200.plan as plan_mod
        plan_mod.Plan = functools.partial(plan_mod.Plan, activation=act)
    plan, _, devb, _ = bench.build_ensemble("drvae", 32, 0, torch.device("cuda:0"))
    ms, launches, _ = bench.time_steps(plan, devb, steps, warmup, seed=1234)
    torch.cuda.synchronize()
    digest = lambda t: hashlib.sha256(t.detach().cpu().contiguous().numpy().tobytes()).hexdigest()[:16]
    print(json.dumps({"variant": variant, "ms_per_step": ms / steps, "launches_per_step": launches / steps,
                      "graph_replays": plan.graph_replays(), "graph_failures": plan.graph_failures(),
                      "losses_sha": digest(plan.losses), "params_sha": digest(plan.params),
                      "cmpl_member0": float(plan.losses[0, 6])}))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--variant", choices=list(VARIANTS))
    ap.add_argument("--tree", default=None, help=argparse.SUPPRESS)
    ap.add_argument("--parent-lib", default=os.path.join(ROOT, "drvae_b200", "lib", "libdrvae_b200_parent.so"))
    ap.add_argument("--parent-tree", default=os.path.join(ROOT, "drvae_b200", "lib", "parent_tree"))
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if a.variant:
        return child(a.variant, a.steps, a.warmup, a.tree)
    lines = [subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                            capture_output=True, text=True).stdout.strip()]
    print(lines[0])
    runs = {v: [] for v in VARIANTS}
    hashes = {v: set() for v in VARIANTS}
    for rep in range(a.repeats):
        for v in VARIANTS:
            env = dict(os.environ)
            cmd = [sys.executable, os.path.abspath(__file__), "--variant", v, "--steps", str(a.steps), "--warmup", str(a.warmup)]
            if v == "parent":
                env["DRVAE_B200_LIB"] = os.path.abspath(a.parent_lib)
                cmd += ["--tree", a.parent_tree]
            r = subprocess.run(cmd, capture_output=True, text=True, env=env, cwd=ROOT)
            if r.returncode != 0:
                raise SystemExit("variant %s failed:\n%s" % (v, r.stderr[-4000:]))
            line = [l for l in r.stdout.splitlines() if l.startswith("{")][-1]
            d = json.loads(line)
            d["repeat"] = rep
            runs[v].append(d["ms_per_step"])
            hashes[v].add((d["losses_sha"], d["params_sha"]))
            lines.append(json.dumps(d))
            print(lines[-1], flush=True)
    for v in VARIANTS:
        xs = sorted(runs[v])
        lines.append("%-9s median %.4f ms/step  (min %.4f, max %.4f, n=%d)" % (v, xs[len(xs) // 2], xs[0], xs[-1], len(xs)))
        print(lines[-1])
    lines.append("elu losses and parameters bit-identical to the parent's: %s" % (hashes["elu"] == hashes["parent"] and len(hashes["elu"]) == 1))
    print(lines[-1])
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
