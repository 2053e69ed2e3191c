#!/usr/bin/env python
"""bench.py — DrVAE training throughput (samples/s, forward + ELBO + backward + Adam) on B200.

Contract: `python bench.py --gpus N --steps K --warmup W` (under torchrun for N > 1) prints ONE
JSON line from rank 0.  Default workload (BASELINE.json configs[4], weak scaling): an ensemble of
independent DrVAE models in the README architecture (dim-z1 100, dim-z3 100, enc-z1 800,
dec-x 600, enc-z3 200, dec-z1 200, L=2, --train-w-noise, batch 150 each), `--models-per-gpu`
(32) models per GPU, i.e. the 256-model drug x fold ensemble at 8 GPUs; members are independent,
so ranks exchange nothing on the data path.  A "step" trains every member of the shard once.

The same line carries, as extra keys, the other BASELINE configurations: `other_workloads` (single
DrVAE / PVAE / VFAE models at batch 150 and PVAE / VFAE ensembles) and, when launched on more than
one rank, `dp8192` (configs[3]: one model, global batch 8192 row-sharded over the ranks).

`--impl reference` times the reference's CPU implementation of the same step on this box's host
cores the way the reference deploys it (src/scripts/submitVAE.sh:14, src/run_drvae.py:38-41):
cores/4 concurrent processes of 4 threads, one ensemble member each.  /root/reference is not
present on the GPU box, so that arm runs the oracle port (oracle/drvae_oracle.py: the same torch
CPU ops, autograd and torch.optim.Adam the reference calls; pinned to the reference in
oracle/make_golden.py).

`--dump-outputs DIR` writes what the last timed step computed (rank 0's models) as .npy files, so that two builds can
be compared output for output: every input is seeded, so the same arguments give the same inputs in every run.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

README = dict(dim_x=978, dim_y=2, dim_z1=100, dim_z3=100, enc_z1=[800], dec_x=[600], enc_z3=[200], dec_z1=[200])
L = 2
BATCH = 150
N_PARAMS = {"drvae": 2321758, "pvae": 2199756, "vfae": 2301358}  # SURVEY.md 8(d)
FLOP_PER_SAMPLE = {"drvae": 3.792e7, "pvae": 3.590e7, "vfae": 2.083e7}  # GEMM FLOPs, fwd + dX + dW (SURVEY.md 8(d))
FIELDS = {"drvae": ("x1", "x2", "y", "has_x2", "has_y"), "pvae": ("x1", "x2", "has_x2"), "vfae": ("x1", "y", "has_y")}
METRIC = "DrVAE train samples/sec (fwd+bwd+Adam)"
UNIT = "samples/s"
DATASET_ROWS = 600  # synthetic device-resident dataset per ensemble member (end-to-end loop)
DUMP_PARAMS = 1 << 22  # parameters written by --dump-outputs (16 MB of float32); a larger model is sampled


_STDOUT_FD = None


def quiet_stdout():
    """stdout carries exactly one JSON line: native libraries that print there (NCCL's version banner at communicator
    creation) are pointed at stderr for the duration of the run; emit() restores the real stdout for the result."""
    global _STDOUT_FD
    if _STDOUT_FD is None:
        sys.stdout.flush()
        _STDOUT_FD = os.dup(1)
        os.dup2(2, 1)


def emit(line):
    sys.stdout.flush()
    if _STDOUT_FD is not None:
        os.dup2(_STDOUT_FD, 1)
    print(json.dumps(line), flush=True)


def measured_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            p = json.load(f)
        return dict(hbm=p["hbm_gbs"], bf16=p["bf16_tflops"], bf16_sustained=p["bf16_tflops_sustained"], which="measured")
    except Exception:
        return dict(hbm=6650.0, bf16=1590.0, bf16_sustained=1400.0, which="fallback")


def dump_outputs(out_dir, losses, params):
    """losses.npy: the [models, 8] loss terms the step returned.  params.npy: the flat [models, parameters] buffer the
    step updated, or, when it holds more than DUMP_PARAMS values, those at DUMP_PARAMS indices drawn with seed 0 and
    sorted, the same for every run of the same workload.  Both float32."""
    import numpy as np
    import torch
    os.makedirs(out_dir, exist_ok=True)
    flat = params.reshape(-1)
    if flat.numel() > DUMP_PARAMS:
        idx = torch.randint(flat.numel(), (DUMP_PARAMS,), generator=torch.Generator().manual_seed(0)).sort().values
        flat = flat[idx.to(flat.device)]
    np.save(os.path.join(out_dir, "losses.npy"), losses.detach().float().cpu().numpy())
    np.save(os.path.join(out_dir, "params.npy"), flat.detach().float().cpu().numpy())


def ncu_traffic(kernel_tag):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of `kernel_tag`, from the committed
    `ncu --set full` capture of this workload (profiles/ncu_traffic.json names the source report)."""
    try:
        with open(os.path.join(ROOT, "profiles", "ncu_traffic.json")) as f:
            t = json.load(f)["kernels"].get(kernel_tag)
        return None if t is None else t["dram_read_bytes"] + t["dram_write_bytes"]
    except Exception:
        return None


# ------------------------------------------------------------------------------------------------
# clocks
# ------------------------------------------------------------------------------------------------
class ClockSampler(threading.Thread):
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        super().__init__(daemon=True)
        self.gpu = gpu_index
        self.rows = []
        self.stop_flag = False

    def run(self):
        while not self.stop_flag:
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.rows.append([c.strip() for c in out.split(",")])
            except Exception:
                pass
            time.sleep(0.1)

    def summary(self):
        sm = sorted(float(r[1]) for r in self.rows if len(r) > 2 and r[1].replace(".", "").isdigit())
        mx = [float(r[2]) for r in self.rows if len(r) > 2 and r[2].replace(".", "").isdigit()]
        reasons = set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            for i, n in enumerate(names):
                if len(r) > 5 + i and r[5 + i].lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(self.rows)}


# ------------------------------------------------------------------------------------------------
# reference arm / cpu baseline: the oracle port of the reference step on host cores, deployed as the reference
# deploys it — independent processes of 4 threads (src/run_drvae.py:38-41 sets 4 intra-op threads, the sweep script
# src/scripts/submitVAE.sh:14 asks for 4 cores per job), one ensemble member per process
# ------------------------------------------------------------------------------------------------
def _cpu_worker(idx, threads, steps, warmup, start_evt, ready_q, out_q):
    import torch
    from oracle import drvae_oracle as orc
    from drvae_b200.init import init_state_dict
    torch.set_num_threads(threads)
    sd = init_state_dict("drvae", seed=1000 + idx, **README)
    batch = orc.synthetic_batch(BATCH, README["dim_x"], seed=idx)
    om = orc.OracleModel(sd, orc.default_cfg("drvae", L=L))
    for i in range(warmup):
        om.step(batch, orc.Tape(seed=i))
    ready_q.put(idx)
    start_evt.wait()
    t0 = time.perf_counter()
    for i in range(steps):
        om.step(batch, orc.Tape(seed=100 + i))
    out_q.put((idx, time.perf_counter() - t0))


def cpu_throughput(steps, warmup, procs=None, threads=4):
    """-> dict(value samples/s aggregate, ms_per_step, procs, threads, cores).  One member per process, all processes
    stepping at the same time; the aggregate is members x batch x steps / slowest process's time."""
    import multiprocessing as mp
    cores = os.cpu_count() or 1
    if procs is None:
        procs = max(1, cores // threads)
    ctx = mp.get_context("spawn")
    start_evt, ready_q, out_q = ctx.Event(), ctx.Queue(), ctx.Queue()
    ws = [ctx.Process(target=_cpu_worker, args=(i, threads, steps, warmup, start_evt, ready_q, out_q)) for i in range(procs)]
    for w in ws:
        w.start()
    for _ in ws:
        ready_q.get(timeout=600)
    start_evt.set()
    times = [out_q.get(timeout=1200)[1] for _ in ws]
    for w in ws:
        w.join(timeout=60)
    dt = max(times)
    return dict(value=procs * BATCH * steps / dt, ms_per_step=dt / steps * 1e3, procs=procs, threads=threads, cores=cores,
                per_process_samples_per_s=BATCH * steps / (sum(times) / len(times)))


def cpu_model_name():
    try:
        with open("/proc/cpuinfo") as f:
            for line in f:
                if line.startswith("model name"):
                    return line.split(":", 1)[1].strip()
    except Exception:
        pass
    return "unknown"


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    r = cpu_throughput(max(1, args.steps), max(1, args.warmup))
    sample = ("%d concurrent processes x %d threads (the reference's deployment: src/scripts/submitVAE.sh:14, "
              "src/run_drvae.py:38-41), one DrVAE README-config ensemble member (batch 150) each, %d steps; host: %d "
              "logical cores, %s; /root/reference does not travel to the GPU box: oracle port of the step"
              % (r["procs"], r["threads"], args.steps, r["cores"], cpu_model_name()))
    line = {
        "impl": "reference", "metric": METRIC, "value": r["value"], "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": r["ms_per_step"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": workload_config(args),
        "cpu_baseline": {"value": r["value"], "unit": UNIT, "cores": r["procs"] * r["threads"], "kind": "port", "sample": sample,
                         "per_process_samples_per_s": r["per_process_samples_per_s"]},
        "e2e": {"value": r["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(line)


def workload_config(args):
    return {"workload": "DrVAE README-config ensemble (BASELINE configs[4] shard): %d independent models per GPU x batch %d, "
                        "L=2, train-w-noise, Philox noise drawn in-step" % (args.models_per_gpu, BATCH),
            "models_per_gpu": args.models_per_gpu, "batch_per_model": BATCH, "parallelism": "ensemble-shard x%d (no collective)" % args.gpus,
            "l2_policy": "working set per step (%.1f GB of parameters, Adam state and activations) exceeds the 126 MB L2"
                         % (args.models_per_gpu * N_PARAMS["drvae"] * 16 / 1e9)}


# ------------------------------------------------------------------------------------------------
# algorithmic work per launch class (SURVEY.md §8(d)): GEMM FLOPs from the valid dims
# ------------------------------------------------------------------------------------------------
def gemm_dims(N=BATCH):
    Np, Nlab = (N + 1) // 2, N - (N + 2) // 3
    R0, LN, Rd, F = N + Np, L * N, L * (N + 2 * Np), L * (Nlab + 2 * (N - Nlab))
    a = README
    d = {}

    def block(name, rows, kin, hidden, out2, first_dx):
        prev = kin
        for i, h in enumerate(hidden):
            d["%s.fwd:gemm_nt.h%d" % (name, i)] = (rows, h, prev)
            d["%s.bwd:gemm_dw.h%d" % (name, i)] = (h, prev, rows)
            if i > 0 or first_dx:
                d["%s.bwd:gemm_dx.h%d" % (name, i)] = (rows, prev, h)
            prev = h
        d["%s.fwd:gemm_nt.head" % name] = (rows, out2, prev)
        d["%s.bwd:gemm_dw.head" % name] = (out2, prev, rows)
        d["%s.bwd:gemm_dx.head" % name] = (rows, prev, out2)

    block("enc", R0, a["dim_x"], a["enc_z1"], 2 * a["dim_z1"], False)
    block("dec", Rd, a["dim_z1"], a["dec_x"], 2 * a["dim_x"], True)
    d["dec.fwd:gemm_nt_decloss.head"] = d.pop("dec.fwd:gemm_nt.head")
    block("z3", F, a["dim_z1"], a["enc_z3"], 2 * a["dim_z3"], True)
    block("dz1", F, a["dim_z3"], a["dec_z1"], 2 * a["dim_z1"], True)
    d["T.fwd:gemm_nt.head"] = (LN, 2 * a["dim_z1"], a["dim_z1"])
    d["T.bwd:gemm_dw.head"] = (2 * a["dim_z1"], a["dim_z1"], LN)
    d["T.bwd:gemm_dx.head"] = (LN, a["dim_z1"], 2 * a["dim_z1"])
    return d


def gemm_layer_params():
    """Parameters (weights + biases) of the layers the grouped dW+Adam launch updates: everything but the classifier."""
    a = README
    return N_PARAMS["drvae"] - (a["dim_y"] * 2 * a["dim_z1"] + a["dim_y"])


# ------------------------------------------------------------------------------------------------
# distributed helpers
# ------------------------------------------------------------------------------------------------
class Ranks:
    def __init__(self):
        import torch
        self.torch = torch
        self.rank = int(os.environ.get("RANK", "0"))
        self.local_rank = int(os.environ.get("LOCAL_RANK", "0"))
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        if not torch.cuda.is_available():
            raise RuntimeError("bench.py needs a GPU (there is no CPU fallback); use --impl reference for the CPU arm")
        torch.cuda.set_device(self.local_rank)
        self.dev = torch.device("cuda", self.local_rank)
        self.dist = None
        if self.world > 1:
            import torch.distributed as dist
            dist.init_process_group("nccl", device_id=self.dev)
            self.dist = dist

    def barrier(self):
        self.torch.cuda.synchronize()
        if self.dist is not None:
            self.dist.barrier()
            self.torch.cuda.synchronize()

    def max(self, x):
        if self.dist is None:
            return x
        t = self.torch.tensor([x], dtype=self.torch.float64, device=self.dev)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())

    def close(self):
        if self.dist is not None:
            self.dist.destroy_process_group()


def build_ensemble(kind, M, first_model, dev, dataset_rows=0):
    """Plan with M README-architecture models (seeds 1000 + global index) and their synthetic batches (pinned host +
    device).  dataset_rows > 0: additionally a device-resident synthetic dataset per member."""
    import torch
    from drvae_b200.init import init_state_dict
    from drvae_b200.plan import Plan
    from drvae_b200.synth import synthetic_batch
    plan = Plan(kind, L=L, max_batch=BATCH, n_models=M, **README)
    host = {k: [] for k in FIELDS[kind]}
    data = {k: [] for k in FIELDS[kind]}
    for m in range(M):
        gm = first_model + m
        plan.load_state_dict(init_state_dict(kind, seed=1000 + gm, **README), model=m)
        b = synthetic_batch(BATCH, README["dim_x"], seed=gm)
        for k in host:
            host[k].append(b[k])
        if dataset_rows:
            d = synthetic_batch(dataset_rows, README["dim_x"], seed=100000 + gm)
            for k in data:
                data[k].append(d[k])
    host = {k: torch.stack(v).contiguous().pin_memory() for k, v in host.items()}
    devb = {k: v.to(dev) for k, v in host.items()}
    dataset = {k: torch.stack(v).contiguous().to(dev) for k, v in data.items()} if dataset_rows else None
    return plan, host, devb, dataset


def time_steps(plan, devb, steps, warmup, seed, ranks=None, step0=0):
    """CUDA-event time of `steps` train steps on device-resident batches -> (ms total, launches)."""
    import torch
    from drvae_b200.plan import anneal_coef
    s = step0
    for _ in range(warmup):
        plan.train_step(devb, plan.hparams(step=s, beta_pert=anneal_coef(s, 1, 0)), seed=seed)
        s += 1
    if ranks is not None:
        ranks.barrier()
    else:
        torch.cuda.synchronize()
    l0 = plan.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        plan.train_step(devb, plan.hparams(step=s, beta_pert=anneal_coef(s, 1, 0)), seed=seed)
        s += 1
    e1.record()
    if ranks is not None:
        ranks.barrier()
    else:
        torch.cuda.synchronize()
    return e0.elapsed_time(e1), plan.launch_count() - l0, s


def parity_check():
    """Member-0 configuration (README DrVAE, seed 123, batch 0) through the C ABI with an injected eps tape vs the fp32
    oracle: every loss term within north_star's 1e-3.  (The timed steps draw Philox noise, which no CPU tape reproduces.)"""
    import torch
    from oracle import drvae_oracle as orc
    from drvae_b200.init import init_state_dict
    from drvae_b200.noise import eps_block_from_tape
    from drvae_b200.plan import LOSS_KEYS, Plan, anneal_coef
    sd = init_state_dict("drvae", seed=123, **README)
    batch = orc.synthetic_batch(BATCH, README["dim_x"])
    om = orc.OracleModel(sd, orc.default_cfg("drvae", L=L))
    tape = orc.Tape(seed=777)
    want = om.loss(batch, tape, train=True)
    plan = Plan("drvae", L=L, max_batch=BATCH, n_models=1, **README)
    plan.load_state_dict(sd)
    eps = eps_block_from_tape(plan, tape.log, batch["has_x2"], batch["has_y"], noisy=True)
    b = {k: batch[k] for k in FIELDS["drvae"]}
    got = plan.train_step(b, plan.hparams(step=0, beta_pert=anneal_coef(0, 1, 0)), eps=eps)[0].cpu()
    torch.cuda.synchronize()
    worst = 0.0
    for i, k in enumerate(LOSS_KEYS):
        if k in want and k != "MMD":
            ref = float(want[k])
            worst = max(worst, abs(float(got[i]) - ref) / (abs(ref) + 1e-12))
    if worst > 1e-3:
        raise RuntimeError("parity check failed before timing: worst relative loss error %.3e > 1e-3" % worst)
    return {"config": "README DrVAE, seed 123, batch 150, injected eps tape 777, step 0", "worst_rel_loss_err_vs_fp32_oracle": worst,
            "tolerance": 1e-3, "ELBO": float(got[5]), "ELBO_oracle": float(want["ELBO"])}


def dp8192_result(ranks, steps, warmup, dump_dir=None):
    """BASELINE configs[3]: DrVAE README architecture, ONE model, global minibatch 8192, rows sharded over the ranks
    (drvae_b200.dp).  Strong scaling: the global batch is fixed."""
    import torch
    from drvae_b200 import dp as dpm
    from drvae_b200.init import init_state_dict
    from drvae_b200.plan import Plan
    from drvae_b200.synth import synthetic_batch
    GLOBAL_N = 8192
    dev, world, rank = ranks.dev, ranks.world, ranks.rank
    lo, hi = dpm.shard_rows(GLOBAL_N, world, rank)
    plan = Plan("drvae", L=L, max_batch=hi - lo, n_models=1, **README)
    plan.load_state_dict(init_state_dict("drvae", seed=123, **README))
    full = synthetic_batch(GLOBAL_N, README["dim_x"], seed=0)
    host = {k: full[k][lo:hi].contiguous().pin_memory() for k in FIELDS["drvae"]}
    devb = {k: v.to(dev) for k, v in host.items()}
    backend = None
    if world > 1 and os.environ.get("DRVAE_B200_DP_BACKEND", "peer") == "peer":
        try:
            backend = dpm.PeerBackend(plan)  # gradients summed over NVLink peer memory inside the optimizer kernel
        except Exception as e:  # symmetric memory unavailable: NCCL all-reduce per bucket
            print("PeerBackend unavailable (%s): falling back to NCCL" % e, file=sys.stderr)
    if backend is None:
        backend = dpm.PlanBackend(plan)
    runner = dpm.DataParallel(backend)
    for _ in range(max(warmup, 4)):
        runner.step(devb, seed=1, row_offset=lo, host_flags=host)
    ranks.barrier()
    l0 = plan.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        losses = runner.step(devb, seed=1, row_offset=lo, host_flags=host)
    e1.record()
    ranks.barrier()
    if dump_dir and rank == 0:
        dump_outputs(dump_dir, losses, plan.params)
    ms = ranks.max(e0.elapsed_time(e1))
    launches = plan.launch_count() - l0
    peaks = measured_peaks()
    flops = FLOP_PER_SAMPLE["drvae"] * GLOBAL_N
    tf = flops / (ms / steps * 1e-3) / 1e12
    out = losses.detach().cpu()
    return {"workload": "DrVAE README config, single model, global batch 8192 (BASELINE configs[3]), rows sharded over %d rank(s); "
                        "gradients summed over NVLink; Philox noise keyed by global row" % world,
            "value": GLOBAL_N * steps / (ms / 1e3), "unit": UNIT, "ms_per_step": ms / steps, "scaling": "strong", "n_gpus": world,
            "rows_per_rank": hi - lo, "gpu_launches": launches, "graph": bool(getattr(runner.backend, "graphs", None)),
            "exchange": ("NVLink peer memory, all-reduce fused into the Adam kernel" + (" (NVLS multicast)" if getattr(backend, "multicast", False) else ""))
                        if getattr(backend, "peer", False) else ("NCCL all-reduce per bucket" if world > 1 else "none (1 rank)"),
            "gemm_tflops_per_gpu": tf / world, "frac_of_bf16_sustained_per_gpu": tf / world / peaks["bf16_sustained"],
            "losses": {k: float(out[i]) for i, k in enumerate(("RECL", "KLD", "PERT", "YL", "MMD", "ELBO", "CMPL"))}}


def other_workloads(ranks, steps):
    """BASELINE configs[0..2] (single DrVAE / PVAE / VFAE model, batch 150) and PVAE / VFAE ensembles, device-timed."""
    peaks = measured_peaks()
    out = {}
    for kind in ("drvae", "pvae", "vfae"):
        plan, host, devb, _ = build_ensemble(kind, 1, 0, ranks.dev)
        ms, launches, _ = time_steps(plan, devb, steps, 5, seed=1)
        per = ms / steps
        floor_us = max(24.0 * N_PARAMS[kind] / (peaks["hbm"] * 1e9), FLOP_PER_SAMPLE[kind] * BATCH / (peaks["bf16_sustained"] * 1e12)) * 1e6
        out["%s150" % kind] = {"workload": "%s README config, ONE model, batch 150 (BASELINE configs[%d])" % (kind, ("drvae", "pvae", "vfae").index(kind)),
                               "ms_per_step": per, "value": BATCH / (per * 1e-3), "unit": UNIT, "launches_per_step": launches / steps,
                               "floor_us": floor_us, "frac_of_floor": floor_us / (per * 1e3),
                               "floor": "max(24 B x parameters / measured HBM GB/s, GEMM FLOPs / sustained bf16): launch/latency-bound (SURVEY 8(d))"}
        # the same step through the persistent step kernel (one cooperative launch for the whole forward + dX chain,
        # grid barriers between dependent stages): measured next to the default graph of launches, not the default
        plan.set_step_kernel(True)
        ms2, launches2, _ = time_steps(plan, devb, steps, 5, seed=1)
        out["%s150" % kind]["persistent_step_kernel"] = {"ms_per_step": ms2 / steps, "launches_per_step": launches2 / steps}
        del plan
    M = 32
    for kind in ("pvae", "vfae"):
        plan, host, devb, _ = build_ensemble(kind, M, 0, ranks.dev)
        ms, launches, _ = time_steps(plan, devb, steps, 5, seed=1)
        per = ms / steps
        out["%s_ensemble%d" % (kind, M)] = {"workload": "%s README config, %d independent models x batch 150" % (kind, M), "ms_per_step": per,
                                            "value": M * BATCH / (per * 1e-3), "unit": UNIT, "launches_per_step": launches / steps,
                                            "adam_state_frac_of_hbm": 24.0 * N_PARAMS[kind] * M / (per * 1e-3) / 1e9 / peaks["hbm"],
                                            "gemm_frac_of_bf16_sustained": FLOP_PER_SAMPLE[kind] * BATCH * M / (per * 1e-3) / 1e12 / peaks["bf16_sustained"]}
        del plan
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--models-per-gpu", type=int, default=32)
    ap.add_argument("--workload", default="ensemble", choices=["ensemble", "dp8192"],
                    help="ensemble: BASELINE configs[4] shard (default, weak scaling); dp8192: only configs[3] (one model, "
                         "global batch 8192 row-sharded over the ranks with an NCCL gradient all-reduce, strong scaling)")
    ap.add_argument("--cpu-baseline-steps", type=int, default=12)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip other_workloads / dp8192 / parity (profiling runs)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write the last step's loss terms and "
                                                          "updated parameters (a seeded sample of them) to DIR/*.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of the GPU step (--impl b200)")
    if args.warmup < 3:
        args.warmup = 3
    quiet_stdout()
    if args.impl == "reference":
        return run_reference(args)

    import torch
    from drvae_b200.plan import anneal_coef
    ranks = Ranks()
    rank, world, dev = ranks.rank, ranks.world, ranks.dev
    if args.workload == "dp8192":
        r = dp8192_result(ranks, args.steps, args.warmup, dump_dir=args.dump_outputs)
        line = {"metric": METRIC, "value": r["value"], "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": r["ms_per_step"], "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "bf16",
                "data": "synthetic", "config": {"workload": r["workload"], "global_batch": 8192, "parallelism": "dp%d" % world},
                "gpu_launches": r["gpu_launches"], "dp8192": r}
        if rank == 0:
            emit(line)
        return ranks.close()

    parity = None
    if rank == 0 and not args.no_extras:
        parity = parity_check()  # raises when the step does not match the oracle: no number without parity
    M = args.models_per_gpu
    plan, host, devb, dataset = build_ensemble("drvae", M, rank * M, dev, dataset_rows=DATASET_ROWS)
    comp = torch.cuda.Stream(device=dev)
    torch.cuda.set_stream(comp)
    step_no = 0
    # ---- device-resident timed region ----
    _, _, step_no = time_steps(plan, devb, 0, args.warmup, seed=rank, ranks=ranks)
    sampler = ClockSampler(ranks.local_rank)
    sampler.start()
    time.sleep(0.25)
    ms, launches, step_no = time_steps(plan, devb, args.steps, 0, seed=rank, ranks=ranks, step0=step_no)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, plan.losses, plan.params)  # train_step's result buffer still holds the last step
    ms = ranks.max(ms)
    samples = world * M * BATCH * args.steps
    value = samples / (ms / 1e3)

    # ---- end to end through the public API ----
    # What a training loop over a device-resident dataset does every step (the reference's fit() draws minibatches from
    # an in-memory dataset through a sampler, src/DrVAE.py:743-781): the host draws the row indices of every member's
    # minibatch, copies them from pinned memory to the device (H2D), Plan.train_step reads the dataset through them
    # (drvae_batch_t.row_index), and the step's loss terms are copied back to pinned memory (D2H).  The host reads
    # step i's losses after it has enqueued step i+1, so the device never waits for it.
    SLOTS = 4
    idx_pin = [torch.zeros(M, BATCH, dtype=torch.int32).pin_memory() for _ in range(SLOTS)]
    idx_dev = torch.zeros(M, BATCH, dtype=torch.int32, device=dev)
    loss_pin = [torch.empty(M, 8).pin_memory() for _ in range(SLOTS)]
    loss_ready = [torch.cuda.Event() for _ in range(SLOTS)]
    gen = torch.Generator().manual_seed(1234 + rank)
    e2e_batch = dict(dataset, row_index=idx_dev)

    def e2e_loop(n, s0):
        for i in range(n):
            slot = i % SLOTS
            if i >= SLOTS:
                loss_ready[slot].synchronize()  # the slot's previous copies are done: host buffers may be reused
            torch.randint(0, DATASET_ROWS, (M, BATCH), generator=gen, dtype=torch.int32, out=idx_pin[slot])
            idx_dev.copy_(idx_pin[slot], non_blocking=True)
            res = plan.train_step(e2e_batch, plan.hparams(step=s0 + i, beta_pert=anneal_coef(s0 + i, 1, 0)), seed=rank)
            loss_pin[slot].copy_(res, non_blocking=True)
            loss_ready[slot].record()
        for slot in range(min(n, SLOTS)):
            loss_ready[slot].synchronize()
        return loss_pin[(n - 1) % SLOTS].clone()

    e2e_loop(4, step_no)
    step_no += 4
    windows = []
    for _ in range(5):
        ranks.barrier()
        t0 = time.perf_counter()
        losses = e2e_loop(args.steps, step_no)
        torch.cuda.synchronize()
        windows.append(ranks.max(time.perf_counter() - t0))
        step_no += args.steps
    sampler.stop_flag = True
    sampler.join(timeout=2)
    e2e_s = sorted(windows)[len(windows) // 2]
    e2e_value = samples / e2e_s
    h2d = idx_dev.numel() * idx_dev.element_size()
    d2h = losses.numel() * losses.element_size()
    finite = bool(torch.isfinite(losses).all())

    # ---- dominant kernel: live CUDA-event time over a few extra steps (events on the launching stream) ----
    plan.profile_begin()
    PSTEPS = 3
    for _ in range(PSTEPS):
        plan.train_step(devb, plan.hparams(step=step_no, beta_pert=1.0), seed=rank)
        step_no += 1
    prof = plan.profile_end()
    total_prof = sum(v[1] for v in prof.values())
    peaks = measured_peaks()
    dims = gemm_dims()
    rows = []
    for tag, (n, tms) in prof.items():
        per = tms / n  # ms per launch
        r = {"kernel": tag, "ms_per_launch": per, "share": tms / total_prof}
        base = tag.replace("gemm_dw_adam", "gemm_dw")
        if tag == "bwd:dw_adam_all":
            # grouped weight gradients + Adam of every layer: streams the optimizer state once (read p, m, v; write p, m,
            # v: 24 B/param, SURVEY.md 8(d)) -> HBM-bound
            by = 24.0 * gemm_layer_params() * M
            fl = sum(2.0 * a * b * c for k, (a, b, c) in dims.items() if ":gemm_dw." in k) * M
            r.update(bound="hbm", achieved=by / (per * 1e-3) / 1e9, peak=peaks["hbm"], unit="GB/s", algorithmic_bytes=by,
                     gemm_tflops=fl / (per * 1e-3) / 1e12)
        elif base != tag and base in dims:
            mm, nn, kk = dims[base]
            by = 24.0 * (mm * nn + mm) * M
            r.update(bound="hbm", achieved=by / (per * 1e-3) / 1e9, peak=peaks["hbm"], unit="GB/s", algorithmic_bytes=by,
                     gemm_tflops=2.0 * mm * nn * kk * M / (per * 1e-3) / 1e12)
        elif tag in dims:
            mm, nn, kk = dims[tag]
            fl = 2.0 * mm * nn * kk * M
            r.update(bound="tensor", achieved=fl / (per * 1e-3) / 1e12, peak=peaks["bf16_sustained"], unit="TFLOP/s")
        elif tag == "opt:adam":
            by = 24.0 * N_PARAMS["drvae"] * M
            r.update(bound="hbm", achieved=by / (per * 1e-3) / 1e9, peak=peaks["hbm"], unit="GB/s")
        if "achieved" in r:
            r["frac"] = r["achieved"] / r["peak"]
        rows.append(r)
    rows.sort(key=lambda r: -r["share"])
    top = next((r for r in rows if "achieved" in r), None)
    roofline = None
    if top is not None:
        roofline = {"kernel": top["kernel"], "bound": top["bound"], "achieved": top["achieved"], "peak": top["peak"],
                    "unit": top["unit"], "frac": top["frac"], "traffic": ncu_traffic(top["kernel"]),
                    "traffic_note": "dram__bytes_read.sum + dram__bytes_write.sum per launch, ncu --set full (profiles/ncu_traffic.json); "
                                    "algorithmic bytes per launch = 24 B x parameters of the updated layers x models",
                    "algorithmic_bytes": top.get("algorithmic_bytes"), "share_of_step": top["ms_per_launch"] / (ms / args.steps),
                    "timing": "CUDA events around the launch on its own stream, %d steps after the timed region" % PSTEPS,
                    "note": "timed as ONE launch over all layers (per-launch timing serialises the step); inside the timed step the same "
                            "tiles are issued in two parts: the decoder heads on 92 SMs next to the tail of the backward chain, the "
                            "rest on all SMs (profiles/r02_experiments.md 2b)" if top["kernel"] == "bwd:dw_adam_all" else None,
                    "peak_source": "%s (MEASURED_PEAKS.json %s)" % (peaks["which"], "hbm_gbs" if top["bound"] == "hbm" else "bf16_tflops_sustained")}
    step_flops = sum(2.0 * a * b * c for a, b, c in dims.values())
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "bf16", "data": "synthetic", "config": workload_config(args),
        "clocks": sampler.summary(),
        "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                "how": "median of 5 windows of %d steps; every step: minibatch row indices H2D from pinned memory -> "
                       "Plan.train_step on the device-resident dataset (%d rows per member) -> loss terms D2H to pinned memory"
                       % (args.steps, DATASET_ROWS),
                "windows_ms_per_step": [w / args.steps * 1e3 for w in windows]},
        "gpu_launches": launches,
        "roofline": roofline,
        "step_roofline": {"gemm_tflops": step_flops * M / (ms / args.steps * 1e-3) / 1e12,
                          "gemm_frac_of_bf16_sustained": step_flops * M / (ms / args.steps * 1e-3) / 1e12 / peaks["bf16_sustained"],
                          "adam_state_gbs": 24.0 * N_PARAMS["drvae"] * M / (ms / args.steps * 1e-3) / 1e9,
                          "adam_state_frac_of_hbm": 24.0 * N_PARAMS["drvae"] * M / (ms / args.steps * 1e-3) / 1e9 / peaks["hbm"]},
        "breakdown": [{k: (round(v, 6) if isinstance(v, float) else v) for k, v in r.items()} for r in rows[:12]],
        "losses_finite": finite,
        "parity": parity,
    }
    del plan
    if not args.no_extras:
        if world == 1:
            line["other_workloads"] = other_workloads(ranks, args.steps)
        else:
            line["dp8192"] = dp8192_result(ranks, args.steps, args.warmup)  # collective: every rank takes part
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        r = cpu_throughput(args.cpu_baseline_steps, 2)
        line["cpu_baseline"] = {"value": r["value"], "unit": UNIT, "cores": r["procs"] * r["threads"], "kind": "port",
                                "sample": "%d concurrent processes x %d threads (the reference's deployment), one ensemble member "
                                          "(batch 150) each, %d steps per process, oracle port of the step; host: %d logical cores, %s"
                                          % (r["procs"], r["threads"], args.cpu_baseline_steps, r["cores"], cpu_model_name()),
                                "per_process_samples_per_s": r["per_process_samples_per_s"]}
    if rank == 0:
        dump = os.environ.get("BENCH_BREAKDOWN")
        if dump:
            with open(dump, "w") as f:
                json.dump({"ms_per_step": ms / args.steps, "profiled_ms_per_step": total_prof / PSTEPS, "kernels": rows}, f, indent=1)
        emit(line)
    ranks.close()


if __name__ == "__main__":
    main()
