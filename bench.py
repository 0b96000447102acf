#!/usr/bin/env python
"""bench.py -- meshes/sec of CAPE's graph-conv hot path on B200.

    python bench.py --gpus N --steps K --warmup W [--config c3|c2|c5]     (N > 1: under torch.distributed.run)
    python bench.py --impl reference --gpus N --steps K --warmup W        (CPU arm: the oracle port, host threads)

Workloads (BASELINE.json `configs`; SURVEY.md section 8 IDs):
  c3 (default; the config the metric is quoted on; = configs[3] when launched on 8 GPUs): full CAPE-affineconv nz64
     VAE+GAN train step = condition nets + encoder + decoder + discriminator (real+fake) forward, all backward passes,
     losses, global-norm clip + momentum update of both players; 64 meshes per GPU per step (weak scaling).
  c2: CAPE-affineconv nz64 encoder+decoder FORWARD, 32 meshes per GPU per step (configs[1]).
  c5: CAPE nz18_pose24_clotype8 (GroupNorm decoder blocks, the plain chebyshev5 path) train step, 64 meshes per GPU
     (configs[4] = 4 GPUs x 64).
Synthetic [N,6890,3] offsets, random-init weights (the reference's initialisers), fp32 throughout.

One JSON line on stdout (rank 0).  `value`: device-resident inputs, CUDA-event timing of exactly K steps, max over
ranks.  `e2e`: the same step through the public API with pinned HOST inputs copied in and the result copied out every
step.  `roofline`: the dominant kernel family of one profiled eager step -- algorithmic bytes (SURVEY.md 8d) of its
launches / their CUDA-event time -- against the measured HBM peak.  `cpu_baseline`: the oracle (torch-CPU port of the
reference graph) on a bounded sample of the same step, plus the literal NumPy/SciPy transcription of one conv.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

# alg_mb: algorithmic bytes per mesh of the whole step (SURVEY.md 8d "logical tensors once")
CONFIGS = {
    "c3": dict(metric="meshes/sec fwd+bwd CAPE-affineconv nz64", params="NZ64_AFFINE", mode="train", batch=64,
               alg_mb=383.1, workload="CAPE-affineconv nz64_pose32_clotype32 full VAE+GAN train step "
                                      "(BASELINE configs[2]; configs[3] when n_gpus=8)"),
    "c2": dict(metric="meshes/sec fwd CAPE-affineconv nz64 (encoder+decoder)", params="NZ64_AFFINE", mode="fwd",
               batch=32, alg_mb=135.6, workload="CAPE-affineconv nz64_pose32_clotype32 encoder+decoder forward "
                                                "(BASELINE configs[1])"),
    "c5": dict(metric="meshes/sec fwd+bwd CAPE nz18 (GroupNorm decoder)", params="NZ18_PLAIN", mode="train", batch=64,
               alg_mb=712.2, workload="CAPE nz18_pose24_clotype8 (non-affine, GroupNorm residual decoder blocks) full "
                                      "VAE+GAN train step (BASELINE configs[4] when n_gpus=4)"),
}


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="cape_b200", choices=["cape_b200", "reference"])
    ap.add_argument("--config", default="c3", choices=sorted(CONFIGS))
    ap.add_argument("--batch", type=int, default=0, help="meshes per GPU per step (0 = the config's own)")
    ap.add_argument("--no-graph", action="store_true", help="launch kernels eagerly instead of replaying CUDA graphs")
    ap.add_argument("--cpu-sample", type=int, default=16, help="meshes per step of the in-line cpu_baseline leg")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-profile", action="store_true")
    ap.add_argument("--tune", default="", help="experiment knobs key=value,... passed to cape_set_tuning")
    ap.add_argument("--dump-outputs", metavar="DIR", default="",
                    help="write what the last timed step computed to DIR/<name>.npy (float32), for comparing builds")
    return ap.parse_args()


def config_and_hierarchy(name):
    from cape_b200 import params as P
    from cape_b200 import topology as T
    L, D, U, p, L_d, D_d, _ = T.load_graph_mtx(load_for_demo=True)
    cfg = dict(getattr(P, CONFIGS[name]["params"]), decay_steps=100)
    return cfg, dict(L=L, D=D, U=U, p=p, L_d=L_d, D_d=D_d)


def config_dict(name, batch, world):
    """The `config` object of the JSON line -- identical for the cape_b200 and the reference arm."""
    c = CONFIGS[name]
    return {"workload": c["workload"], "id": name, "meshes_per_gpu": batch, "global_batch": batch * world,
            "parallelism": "dp%d" % world,
            "l2": "no explicit flush between timed steps: one step streams %.1f GB of activations (>> 126 MB L2)"
                  % (c["alg_mb"] * 1e-3 * batch),
            "update_rule": "real discriminator gradients (ref_compat=False); the lib/models.py:466 quirk is available "
                           "as ref_compat=True" if c["mode"] == "train" else "n/a (forward only)"}


# ---------------------------------------------------------------------------------------------------
# CPU arm: the oracle port of the reference graph (the reference's TF-1.13 CPU path cannot run here)
# ---------------------------------------------------------------------------------------------------
def cpu_port_rate(name, n_sample, steps, warmup):
    """meshes/sec of the oracle on the config's step (same work as the GPU step) with the host threads."""
    import torch
    from oracle import cape_oracle as O
    from cape_b200 import topology as T
    from cape_b200.params import init_params, param_specs
    from cape_b200.synthetic import make_batch
    cfg, h = config_and_hierarchy(name)
    # all host cores up to 32: beyond that the oracle's small sparse/dense ops get SLOWER (measured on the GPU box:
    # 67 s/step for 4 meshes with one thread per core vs. ~0.6 s/step capped at 32), and the baseline should be the
    # CPU's best
    torch.set_num_threads(min(os.cpu_count() or 1, 32))
    specs = param_specs(cfg, [l.shape[0] for l in h["L"]], [l.shape[0] for l in h["L_d"]])
    params = init_params(specs, cfg["seed"])
    o = O.Oracle(h["L"], h["D"], h["U"], h["L_d"], h["D_d"], cfg)
    P = {k: torch.from_numpy(v) for k, v in params.items()}
    mom = {k: torch.zeros_like(v) for k, v in P.items()}
    b = {k: torch.from_numpy(v) for k, v in make_batch(n_sample, cfg["nz"], seed=cfg["seed"]).items()}
    edges = T.smpl_edges()

    def one(i):
        if CONFIGS[name]["mode"] == "train":
            O.train_update(o, P, mom, b, i, edges)
        else:
            with torch.no_grad():
                y, y2 = o.cond_embeddings(b["cond_g"], b["cond2_g"], P)
                o.generator(b["x_g"], y, y2, b["eps"], P)

    for i in range(warmup):
        one(1000 + i)
    t0 = time.perf_counter()
    for i in range(steps):
        one(2000 + i)
    dt = time.perf_counter() - t0
    return n_sample * steps / dt, dt / steps, torch.get_num_threads()


def numpy_literal_baseline():
    """The literal NumPy/SciPy transcription of chebyshev5 (oracle/np_ops.py: SciPy fp32 CSR SpMM, single-threaded, +
    BLAS sgemm) on one encoder-sized conv -- the closest thing to the reference's 'TF1 CPU path' per-op arithmetic."""
    import numpy as np
    from oracle import np_ops
    from cape_b200 import topology as T
    L = T.load_graph_mtx(load_for_demo=True)[0]
    rng = np.random.RandomState(0)
    N, M, Fin, Fout, K = 8, 6890, 64, 64, 2
    x = rng.normal(size=(N, M, Fin)).astype(np.float32)
    W = rng.normal(0, 0.1, size=(Fin * K, Fout)).astype(np.float32)
    np_ops.chebyshev5_np(x, L[1], W, K)
    t0 = time.perf_counter()
    reps = 3
    for _ in range(reps):
        np_ops.chebyshev5_np(x, L[1], W, K)
    dt = (time.perf_counter() - t0) / reps
    alg = 4 * N * M * (Fin + Fout) + 4 * Fin * K * Fout + 12 * 41328
    return {"op": "chebyshev5 K=2 64->64 on [8,6890,64] (enc conv2 shape), numpy/scipy literal transcription",
            "ms": dt * 1e3, "layer_meshes_per_s": N / dt, "alg_GBps": alg / dt / 1e9}


def dump_outputs(net, train, directory, per_param=65536):
    """What a caller of the timed step receives after it: the reconstruction, the posterior mean / log-variance and,
    for a train step, the loss terms and the updated parameters of both players.  The parameters (65 MB for nz64) are a
    fixed sample: up to `per_param` entries of each tensor, at indices drawn from a generator seeded by the tensor's
    name and size, concatenated in name order."""
    import zlib
    import numpy as np
    out = {"x_hat": net.x_hat, "z_mean": net.z_mean, "z_logvar": net.z_logvar}
    if train:
        out["losses"] = net.losses[:6]                     # recon, edge, kl, gan_g, gan_d_real, gan_d_fake
    out = {k: v.detach().float().cpu().numpy() for k, v in out.items()}
    if train:
        parts = []
        for name, v in sorted(net.get_params().items()):
            v = v.reshape(-1)
            if v.size > per_param:
                rng = np.random.RandomState(zlib.crc32(("%s:%d" % (name, v.size)).encode()))
                v = v[np.sort(rng.choice(v.size, per_param, replace=False))]
            parts.append(v)
        out["params_sample"] = np.concatenate(parts).astype(np.float32)
    os.makedirs(directory, exist_ok=True)
    for name, v in out.items():
        np.save(os.path.join(directory, name + ".npy"), v)


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    world = int(os.environ.get("WORLD_SIZE", str(args.gpus)))
    c = CONFIGS[args.config]
    batch = args.batch or c["batch"]
    rate, sps, threads = cpu_port_rate(args.config, batch, args.steps, args.warmup)
    sample = ("%d meshes per step = one GPU's share of the global batch (%s), torch-CPU oracle port of lib/models.py, "
              "%d threads" % (batch, "full update: enc+dec+2xdisc fwd/bwd+clip+momentum" if c["mode"] == "train"
                              else "encoder+decoder forward", threads))
    line = {"impl": "reference", "metric": c["metric"], "value": rate, "unit": "meshes/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": sps * 1e3, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": config_dict(args.config, batch, world),
            "note": "the reference's TF-1.13 cannot be installed (no tensorflow wheel, py3.12): this is the oracle port "
                    "of lib/models.py on the host cores, %d meshes per step on rank 0 whatever n_gpus is" % batch,
            "cpu_baseline": {"value": rate, "unit": "meshes/s", "cores": threads, "kind": "port", "sample": sample},
            "e2e": {"value": rate, "unit": "meshes/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


# ---------------------------------------------------------------------------------------------------
# clocks sampler (B200_PROFILING.md recipe)
# ---------------------------------------------------------------------------------------------------
class Clocks:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.proc = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(gpu_index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.proc = None

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            out = self.proc.communicate(timeout=5)[0]
        except Exception:
            self.proc.kill()
            out = ""
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in out.strip().splitlines():
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                mx.append(float(f[2]))
            except ValueError:
                continue
            for nm, v in zip(names, f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def main():
    args = parse()
    if args.impl == "reference":
        return run_reference(args)

    import torch
    import torch.distributed as dist
    from cape_b200 import _lib
    from cape_b200 import distributed as DP
    from cape_b200 import engine as E
    from cape_b200.network import CapeNetwork
    from cape_b200.synthetic import make_batch

    # stdout carries exactly one JSON line: keep NCCL's version banner (NCCL_DEBUG=VERSION in some images) off it
    if os.environ.get("NCCL_DEBUG", "").upper() in ("", "VERSION"):
        os.environ["NCCL_DEBUG"] = "WARN"
    assert torch.cuda.is_available(), "bench.py (impl cape_b200) needs a GPU; there is no CPU fallback"
    rank, world, local = DP.init("nccl")
    torch.cuda.set_device(local)
    lib = _lib.load()
    for kv in filter(None, args.tune.split(",")):
        k, v = kv.split("=")
        lib.cape_set_tuning(int(k), int(v))
    c = CONFIGS[args.config]
    train = c["mode"] == "train"
    cfg, h = config_and_hierarchy(args.config)
    N = args.batch or c["batch"]
    net = CapeNetwork(h["L"], h["D"], h["U"], h["L_d"], h["D_d"], cfg, N, device=local)
    DP.broadcast_params([net.PG.flat, net.PD.flat])          # replicas start from rank 0's weights
    net.prep_weights()
    hb = {k: torch.from_numpy(v).pin_memory()
          for k, v in make_batch(N, cfg["nz"], seed=DP.rank_seed(cfg["seed"], rank)).items()}
    order = ("x_g", "cond_g", "cond2_g", "eps", "x_d", "cond_d", "cond2_d") if train else ("x_g", "cond_g", "cond2_g", "eps")
    h2d_bytes = sum(hb[k].numel() * 4 for k in order)
    batch = [hb[k] for k in order]
    net.set_inputs(*batch)
    allreduce = DP.make_allreduce(world) if train else None   # forward-only replicas have nothing to exchange
    # opt-in (CAPE_DP_OVERLAP=1): the bucketed all-reduce inside the step graph; the default is one all-reduce of the two
    # flat gradient buffers between the graphs
    overlap = train and world > 1 and os.environ.get("CAPE_DP_OVERLAP", "0") == "1"
    if overlap:
        net.set_data_parallel(world)                          # bucketed all-reduce inside the step, behind the backward

    use_graph = not args.no_graph
    c0 = lib.cape_launch_count()
    if train:
        net.train_step(step=0, allreduce=allreduce)          # eager step: lazy inits + launch count of one step
    else:
        net.forward_generator()
    torch.cuda.synchronize()
    launches_per_step = lib.cape_launch_count() - c0
    graph_note = "eager"
    if use_graph:
        try:
            if train:
                net.capture_graphs()
                graph_note = "2 CUDA graphs/step (fwd+bwd, update)" + (
                    "" if world == 1 else ("; bucketed NCCL all-reduce captured inside the first, overlapping the backward"
                                           if overlap else "; NCCL all-reduce between them"))
            else:
                net.capture_forward_graph()
                graph_note = "1 CUDA graph/step (generator forward)"
        except Exception as e:                              # pragma: no cover
            use_graph = False
            graph_note = "eager (graph capture failed: %s)" % str(e)[:80]
            torch.cuda.synchronize()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def step(i):
        if train:
            net.train_step(step=i, allreduce=allreduce, use_graph=use_graph)
        elif use_graph:
            net.graph_fwd.replay()
        else:
            net.forward_generator()

    # ---- device-resident timing ----------------------------------------------------------------------------------
    for i in range(args.warmup):
        step(1 + i)
    barrier()
    clocks = Clocks(local) if rank == 0 else None
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    for i in range(args.steps):
        step(100 + i)
    ev1.record()
    barrier()
    ms = ev0.elapsed_time(ev1)
    t = torch.tensor([ms], device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t.item())

    # ---- end to end: pinned host inputs in, result out, every step --------------------------------------------------
    # Every step's batch crosses PCIe inside the timed region (prefetch_inputs: pinned host -> staging buffers on a
    # copy stream, overlapping the previous step; commit_inputs: staging -> the step's input buffers) and every step's
    # result (train: the loss terms; forward: the predicted meshes) is read back before the next step is enqueued.
    result = net.losses if train else net.x_hat
    d2h_bytes = result.numel() * 4
    host_out = torch.empty(result.shape, dtype=result.dtype).pin_memory()
    for i in range(2):
        net.prefetch_inputs(*batch); net.commit_inputs(); step(300 + i); host_out.copy_(result)
    barrier()
    t0 = time.perf_counter()
    net.prefetch_inputs(*batch)
    for i in range(args.steps):
        net.commit_inputs()
        if i + 1 < args.steps:
            net.prefetch_inputs(*batch)                   # next step's inputs: H2D while this step computes
        step(400 + i)
        host_out.copy_(result)                            # D2H of the step's result (synchronises)
    barrier()
    e2e_s = time.perf_counter() - t0
    clk = clocks.stop() if clocks else None        # sampled over both timed regions (device-resident and end-to-end)
    if args.dump_outputs and rank == 0:
        dump_outputs(net, train, args.dump_outputs)
    te = torch.tensor([e2e_s], device="cuda")
    if world > 1:
        dist.all_reduce(te, op=dist.ReduceOp.MAX)
    e2e_s = float(te.item())

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    total_meshes = N * world * args.steps
    conf = config_dict(args.config, N, world)
    line = {"metric": c["metric"], "value": total_meshes / (ms * 1e-3), "unit": "meshes/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": conf,
            "launch": graph_note,
            "l2": "no explicit flush: one step streams ~%.0f GB of activations, >> 126 MB L2" % (c["alg_mb"] * 1e-3 * N),
            "clocks": clk,
            "e2e": {"value": total_meshes / e2e_s, "unit": "meshes/s", "h2d_bytes_per_step": h2d_bytes,
                    "d2h_bytes_per_step": d2h_bytes},
            "gpu_launches": int(launches_per_step * args.steps)}
    if train:
        line["loss"] = {k: float(v) for k, v in zip(("recon", "edge", "kl", "gan_g", "gan_d_real", "gan_d_fake"),
                                                    host_out.tolist())}

    # ---- roofline of the dominant kernel family (one profiled eager step, CUDA events per launch) ---------------------
    if not args.no_profile:
        E.PROFILE = []
        net.set_inputs(*batch)
        if train:
            net.train_step(step=500, allreduce=None, update=False)
        else:
            net.forward_generator()
        torch.cuda.synchronize()
        fam = {}
        rows = []
        for family, tag, nbytes, e0, e1 in E.PROFILE:
            dt = e0.elapsed_time(e1) * 1e-3
            f = fam.setdefault(family, [0.0, 0.0, 0])
            f[0] += nbytes; f[1] += dt; f[2] += 1
            rows.append({"family": family, "launch": tag, "alg_bytes": nbytes, "us": dt * 1e6,
                         "GBps": nbytes / dt / 1e9 if dt > 0 else None})
        E.PROFILE = None
        peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
        if os.path.exists(peaks_path):
            peak, peak_src = float(json.load(open(peaks_path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        else:
            peak, peak_src = 6650.0, "fallback (B200_PROFILING.md)"
        dom = max(fam.items(), key=lambda kv: kv[1][1])
        nb, dt, cnt = dom[1]
        traffic, traffic_src = None, None
        tp = os.path.join(ROOT, "profiles", "roofline_traffic.json")
        if os.path.exists(tp):
            tj = json.load(open(tp))
            traffic = tj.get(dom[0])
            traffic_src = "static: %s" % tj.get("source", "profiles/roofline_traffic.json (ncu --set full capture)")
        tot_b = sum(f[0] for f in fam.values())
        tot_t = sum(f[1] for f in fam.values())
        line["roofline"] = {"bound": "hbm", "kernel": dom[0] + " (family of %d launches per step)" % cnt,
                            "achieved": nb / dt / 1e9, "peak": peak, "unit": "GB/s",
                            "frac": nb / dt / 1e9 / peak, "traffic": traffic, "traffic_source": traffic_src,
                            "peak_source": peak_src,
                            "launches_per_step": cnt, "alg_bytes_per_launch": nb / cnt, "us_per_launch": dt / cnt * 1e6,
                            "share_of_profiled_time": dt / tot_t,
                            "families": {k: {"alg_GB": v[0] / 1e9, "ms": v[1] * 1e3, "launches": v[2],
                                             "GBps": v[0] / v[1] / 1e9} for k, v in fam.items()},
                            "alg_mb_per_mesh_profiled": tot_b / N / 1e6,
                            "whole_step_frac_of_hbm_roofline": (c["alg_mb"] * 1e6 * N / (ms / args.steps * 1e-3)) / 1e9 / peak}
        # per-launch rows go to a temporary file: the tree the benchmark runs from may be read-only
        fd, line["roofline"]["launch_profile"] = tempfile.mkstemp(prefix="cape_b200_launch_profile_%s_" % args.config,
                                                                  suffix=".json")
        with os.fdopen(fd, "w") as f:
            json.dump(rows, f, indent=1)

    # ---- CPU baseline: the oracle port on a bounded sample (rank 0, N=1 only) ------------------------------------------
    if world == 1 and not args.no_cpu_baseline:
        rate, sps, threads = cpu_port_rate(args.config, args.cpu_sample, 2, 1)
        line["cpu_baseline"] = {"value": rate, "unit": "meshes/s", "cores": threads, "kind": "port",
                                "sample": "%d meshes x 2 steps after 1 warm-up, same step, torch-CPU oracle port "
                                          "(%.1f s/step)" % (args.cpu_sample, sps),
                                "numpy_literal": numpy_literal_baseline()}
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
