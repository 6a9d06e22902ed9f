#!/usr/bin/env python
"""bench.py -- env-steps/sec (agents x envs x steps / s) of the GCBF+ rollout hot path.

Contract: `python bench.py --gpus N --steps K --warmup W [--impl reference] [--config 3|4|5] [--dump-outputs DIR]`
(N > 1: launched by torch.distributed.run, one rank per GPU).  One JSON line on rank 0.

A "step" is one steady-state T = 256-step closed-loop rollout (SURVEY 8d) of E envs per GPU of a BASELINE.json
config -- default configs[2] `DoubleIntegrator n=512, 16 envs, obs 8, n-rays 32` (the config the metric is quoted
on); `--config 4` = DubinsCar n=256, obs 16, 32 envs over 8 GPUs (4 per GPU); `--config 5` = LinearDrone n=1024,
64 envs over 8 GPUs (8 per GPU; `--envs-per-gpu` runs the E in {64,128,256,512} sweep).  Per env-step: actor GNN
forward, a = 2 pi + u_ref, clip, Euler, reward / cost, LiDAR ray cast + top-k, radius neighbour lists, with the
reference's pretrained weights of that environment.
`value` : inputs resident in HBM (CUDA events around K replays of the rollout CUDA graph).
`e2e`   : through RolloutEngine with HOST (pinned) initial conditions, H2D + D2H inside.
`roofline`: the kernel with the largest measured share of the env-step (every kernel of the step is timed alone,
            back to back in a CUDA graph on the buffers a real step left behind), algorithmic FLOPs / its time.
`--impl reference`: the restated reference (dense padded N x N formulation of gcbfplus/utils/graph.py + nn/gnn.py,
torch-CPU fp32, host threads) -- JAX is not installable in this image (DESIGN.md 3; re-probed on every run and
recorded in the line), so the CPU oracle is the arm.  Each of its K steps is ONE env-step of ONE env of the workload.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

T_STEPS = 256
# BASELINE.json configs[2..4] (1-based 3..5).  area: density-preserving sqrt(2N) / N^(1/3) (BASELINE.md 3).
# F_edge / F_node: SURVEY 8d FLOP per real edge / per agent (actor net, unfolded reference formulation);
# F_edge_folded / F_node_folded: what the folded inference kernels execute; B_alg: algorithmic bytes per agent-env-step.
CONFIGS = {
    3: dict(env="DoubleIntegrator", N=512, envs_total=16, gpus=1, obs=8, rays=32, area=32.0, F_edge=267520,
            F_node=461312, B_alg=312, name="configs[2]"),
    4: dict(env="DubinsCar", N=256, envs_total=32, gpus=8, obs=16, rays=32, area=22.63, F_edge=267520, F_node=461312,
            B_alg=312, name="configs[3]"),
    5: dict(env="LinearDrone", N=1024, envs_total=64, gpus=8, obs=4, rays=32, area=10.08, F_edge=268544, F_node=461824,
            B_alg=276, name="configs[4]"),
}
STEP_KERNELS = ["edge message + chained gate GEMM (gemm_tc_prod_kernel<...,CHAIN>)", "segment softmax + aggregate",
                "update layer GEMM 128->256", "folded update/head GEMM 256->256 + output partial sums",
                "policy tail + LiDAR + neighbour lists (graph_build_kernel)"]


def metric_name(cfg) -> str:
    return f"env-steps/sec (agents x envs x steps/s) {cfg['env']} n={cfg['N']}"


def folded_flops(cfg):
    """FLOP per real edge / per agent of the FOLDED inference path (DESIGN 4.2): layer 1 (ed + bias table) x 256,
    W23 256x128, gate 128x128 + gate vector; per agent update 128x256, UH 256x256, output 256 x nu."""
    ed = {"SingleIntegrator": 2, "DoubleIntegrator": 4, "DubinsCar": 4, "LinearDrone": 6}[cfg["env"]]
    nu = 3 if cfg["env"] == "LinearDrone" else 2
    return 2 * ((ed + 1) * 256 + 256 * 128 + 128 * 128 + 128), 2 * (128 * 256 + 256 * 256 + 256 * nu)


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return d.get("hbm_gbs", 6650.0), d.get("bf16_tflops", 1590.0), d.get("bf16_tflops_sustained", 1400.0), "measured"
    return 6650.0, 1590.0, 1400.0, "fallback"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md)."""

    def __init__(self, index: int):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self) -> dict:
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0]))
                mx.append(float(f[1]))
            except ValueError:
                continue
            for nm, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


# ======================================================================================== ours
def run_ours(args):
    import torch
    import torch.distributed as dist
    from helpers import product_algo
    from gcbfplus_b200 import _lib
    from gcbfplus_b200.env import make_env
    from gcbfplus_b200.trainer.rollout import RolloutEngine

    cfg = CONFIGS[args.config]
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise RuntimeError("bench.py needs a CUDA device: the product path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    _lib.load(build_if_missing=False)

    env_id, N, T = cfg["env"], cfg["N"], args.T
    E = args.envs_per_gpu or max(cfg["envs_total"] // cfg["gpus"], 1)
    env = make_env(env_id, N, area_size=cfg["area"], num_obs=cfg["obs"], n_rays=cfg["rays"], device=dev)
    algo = product_algo(env, env_id)
    g0 = env.reset(1000 + rank, n_envs=E)
    eng = RolloutEngine(env, E, T=T, n_obs=cfg["obs"])
    eng.set_params(algo.actor_params)
    # host-side (pinned) copies for the e2e leg
    h_agent = g0.agent.cpu().pin_memory()
    h_goal = g0.goal.cpu().pin_memory()
    h_obs = g0.obstacle.packed.cpu().pin_memory()
    h_rew = torch.empty(T, E).pin_memory()
    h_cost = torch.empty(T, E).pin_memory()
    h_final = torch.empty(E, N, env.state_dim).pin_memory()
    eng.set_initial(g0.agent, g0.goal, g0.obstacle)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(ms: float) -> float:
        if world == 1:
            return ms
        t = torch.tensor([ms], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # ---- warm-up (first run captures the CUDA graph)
    for _ in range(max(args.warmup, 3)):
        eng.run(check=False)
    torch.cuda.synchronize()
    eng.check_overflow()
    n_edges = eng.counters[:, 0].float().mean().item()
    deg_real = n_edges / (E * N)

    if args.train_only:
        tr = train_step_bench(torch, dist if world > 1 else None, env, algo, eng, rank, world, cfg, max_over_ranks, barrier)
        if rank == 0:
            print(json.dumps({"train_step": tr}))
        if world > 1:
            import gc
            gc.collect()
            torch.cuda.synchronize()
            dist.destroy_process_group()
        return

    # ---- value: device-resident inputs
    sampler = ClockSampler(local_rank)
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    if rank == 0:
        sampler.start()
    ev0.record()
    for _ in range(args.steps):
        eng.run(check=False)
    ev1.record()
    barrier()
    ms_total = max_over_ranks(ev0.elapsed_time(ev1))
    clocks = sampler.stop() if rank == 0 else {}
    eng.check_overflow()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, eng.result())
    ms_per_step = ms_total / args.steps
    value = N * E * world * T / (ms_per_step * 1e-3)

    # ---- e2e: host buffers in, host results out, every step
    def e2e_step():
        eng.agent[0].copy_(h_agent, non_blocking=True)
        eng.goal.copy_(h_goal, non_blocking=True)
        eng.obstacles.copy_(h_obs, non_blocking=True)
        eng.run(check=False)
        h_rew.copy_(eng.rewards, non_blocking=True)
        h_cost.copy_(eng.costs, non_blocking=True)
        h_final.copy_(eng.agent[T], non_blocking=True)

    e2e_step()
    barrier()
    ev0.record()
    for _ in range(args.steps):
        e2e_step()
    ev1.record()
    barrier()
    ms_e2e = max_over_ranks(ev0.elapsed_time(ev1)) / args.steps
    e2e_value = N * E * world * T / (ms_e2e * 1e-3)
    h2d = (h_agent.numel() + h_goal.numel() + h_obs.numel()) * 4
    d2h = (h_rew.numel() + h_cost.numel() + h_final.numel()) * 4

    # ---- train step (update_inner, reported separately per SURVEY 8d): minibatch of 256 graphs of the
    # recorded rollout, sharded over ranks, incl. the packed-gradient all-reduce
    train = None if args.no_train else train_step_bench(torch, dist if world > 1 else None, env, algo, eng, rank, world,
                                                        cfg, max_over_ranks, barrier)

    # ---- every kernel of the env-step timed alone -> dominant kernel -> roofline
    roof = step_kernel_rooflines(torch, _lib, env, eng, cfg, n_edges, E * N, ms_per_step / T) if rank == 0 else None
    if rank == 0 and eng.persistent:
        roof = persistent_roofline(torch, env, algo, g0, cfg, E, n_edges, E * N, ms_per_step, T, roof)
    cpu = cpu_baseline(cfg, steps=1, warmup=1) if (rank == 0 and world == 1 and not args.no_cpu_baseline) else None

    if rank == 0:
        hbm, tf_burst, tf_sus, src = load_peaks()
        flop_step = (deg_real * cfg["F_edge"] + cfg["F_node"]) * N * E * world          # per env-step, whole job
        out = {
            "metric": metric_name(cfg), "value": value, "unit": "env-steps/s", "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": f"{env_id} n={N} envs/gpu={E} obs={cfg['obs']} n_rays={cfg['rays']} area={cfg['area']} "
                                   f"T={T} rollout ({cfg['name']})", "step": f"one {T}-step rollout of {E} envs per GPU",
                       "weights": f"reference pretrained {env_id} gcbf+ (tests/golden fixture)",
                       "l2": "no flush: each rollout streams its whole trajectory record (0.6 GB at configs[2], > 126 MB L2) "
                             "and every env-step rewrites the ~60 MB activation workspace",
                       "deg_real": deg_real, "edges_per_step": n_edges, "us_per_env_step": ms_per_step / T * 1e3},
            "e2e": {"value": e2e_value, "unit": "env-steps/s", "ms_per_step": ms_e2e, "h2d_bytes_per_step": h2d,
                    "d2h_bytes_per_step": d2h},
            "gpu_launches": eng.launches_per_run * args.steps,
            "clocks": clocks,
            "roofline": roof,
            "rollout_rooflines": {
                "hbm_frac_of_" + src: value * cfg["B_alg"] / (hbm * 1e9 * world),
                "algorithmic_tflops_per_gpu": value / (N * E * world) * flop_step / 1e12 / world,
                "note": f"whole rollout vs HBM ({cfg['B_alg']} B/agent-step) and achieved TFLOP/s per GPU counting the "
                        "reference's unfolded F_edge / F_node (SURVEY 8d); the path is latency-bound "
                        f"({eng.launches_per_run} launch(es) per {T}-step rollout; a dependent chain of phases per "
                        "env-step), not HBM-bound"},
            "train_step": train,
            "cpu_baseline": cpu,
        }
        print(json.dumps(out))
    if world > 1:
        import gc
        gc.collect()                      # captured graphs holding NCCL kernels must be freed before the communicator
        torch.cuda.synchronize()
        dist.destroy_process_group()


DUMP_LIMIT = 63_000_000      # array bytes: with the .npy headers the files stay under 64 MB


def dump_outputs(out_dir: str, res) -> None:
    """Writes the last timed rollout as its caller receives it (RolloutEngine.result(), [E, T or T + 1, ...] records) to
    out_dir/<name>.npy: float32, the per-step edge counts as float64.  Arrays are taken smallest first; each is written
    whole if it fits in an even share of what is left of DUMP_LIMIT, otherwise as that many of its rows (indices over
    all axes but the last, which is kept whole), drawn without replacement by one generator of fixed seed -- so the same
    arguments select the same rows on every run."""
    import numpy as np
    import torch
    outs = {"agent": res.agent, "actions": res.actions, "rewards": res.rewards, "costs": res.costs, "hits": res.hits,
            "n_edges": res.n_edges.double()}
    os.makedirs(out_dir, exist_ok=True)
    rng = np.random.default_rng(0)
    left = DUMP_LIMIT
    order = sorted(outs, key=lambda k: outs[k].numel() * outs[k].element_size())
    for i, name in enumerate(order):
        x = outs[name]
        share = left // (len(order) - i)
        if x.numel() * x.element_size() <= share:
            a = x.contiguous().cpu().numpy()
        else:
            rows = x.numel() // x.shape[-1]
            idx = np.sort(rng.choice(rows, share // (x.shape[-1] * x.element_size()), replace=False))
            sel = tuple(torch.from_numpy(j).to(x.device) for j in np.unravel_index(idx, x.shape[:-1]))
            a = x[sel].cpu().numpy()
        np.save(os.path.join(out_dir, f"{name}.npy"), a)
        left -= a.nbytes
        print(f"dump-outputs: {name}.npy {a.dtype} {list(a.shape)}"
              + ("" if a.shape == tuple(x.shape) else f" (seeded sample of the rows of {list(x.shape)})"), file=sys.stderr)


def train_step_bench(torch, dist, env, algo, eng, rank, world, cfg, max_over_ranks, barrier):
    """GCBF+ update_inner throughput: global minibatch of 256 graphs drawn from the recorded rollout, B/world graphs
    per rank, u_qp := u_ref + 0.1 (label values do not change the work), every optimizer step = ONE CUDA-graph
    replay (algo/train.py MinibatchRunner: gather -> neighbour lists -> train step -> all-reduce -> clip + AdamW)."""
    from gcbfplus_b200.algo import train as T
    B_glob = 256
    B = max(B_glob // world, 1)
    if os.environ.get("GCBF_BENCH_TRAIN_GRAPHS"):        # profiling aid: the per-rank share of an N-GPU run on one GPU
        B = int(os.environ["GCBF_BENCH_TRAIN_GRAPHS"])
    ro = eng.result()
    n_pool = 4 * B
    tsel = torch.arange(n_pool, device=env.device) % eng.T
    esel = (torch.arange(n_pool, device=env.device) // 7) % eng.E
    batch = {"agent": eng.agent[tsel, esel].contiguous(), "hits": eng.hits[tsel, esel].contiguous(),
             "goal": eng.goal[esel].contiguous()}
    g_all = env.get_graph(batch["agent"], batch["goal"], None, hits=batch["hits"])
    obs_rep = ro.obstacle.select(esel.cpu().numpy()) if hasattr(ro.obstacle, "select") else None
    unsafe = env.unsafe_mask(g_all._replace(obstacle=obs_rep))
    batch["unsafe"] = unsafe.to(torch.uint8).contiguous()
    batch["safe"] = (~unsafe).to(torch.uint8).contiguous()
    u_qp = env.u_ref(g_all) + 0.1
    per_graph = g_all.row_deg.reshape(n_pool, -1).sum(dim=1)
    cap = int(per_graph.max().item()) * B
    algo._trainer_state = None
    algo._trainer_state = T.TrainState(algo)
    runner = T.MinibatchRunner(algo, batch, B, cap, u_qp)
    sels = [torch.arange(i * B, (i + 1) * B, device=env.device) for i in range(4)]
    import numpy as np
    denoms = T._minibatch_counts(batch, torch.arange(n_pool, device=env.device), np.arange(0, n_pool + 1, B))
    if dist is not None:
        dist.all_reduce(denoms)
    for i in range(3):                      # eager warm-up, capture, first replay
        runner.run(sels[i % 4], denoms[i % 4])
    torch.cuda.synchronize()
    runner.graph.check_overflow()
    n_it = 8
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    ev0.record()
    for i in range(n_it):
        runner.run(sels[i % 4], denoms[i % 4])
    ev1.record()
    barrier()
    ms = max_over_ranks(ev0.elapsed_time(ev1)) / n_it
    # launch count of one step: one eager pass
    os.environ["GCBF_TRAIN_GRAPH"] = "0"
    n0 = env.lib.gcbf_launch_count()
    runner.run(sels[0], denoms[0])
    launches = env.lib.gcbf_launch_count() - n0
    os.environ["GCBF_TRAIN_GRAPH"] = "1"
    torch.cuda.synchronize()
    n_edges = float(per_graph[:B].sum().item())
    N = env.num_agents
    flops = 9.0 * (n_edges * cfg["F_edge"] + B * N * cfg["F_node"]) * world       # 3 passes x (fwd + ~2x bwd), SURVEY 8d
    return {"ms_per_minibatch": ms, "graphs_per_s": B * world / (ms * 1e-3),
            "agent_samples_per_s": B * world * N / (ms * 1e-3), "global_batch_graphs": B * world,
            "graphs_per_rank": B, "edges_per_rank": n_edges, "kernels_per_step": int(launches),
            "launch_mode": "one CUDA-graph replay per optimizer step (gather + graph build + folded train step + "
                           "all-reduce + clip/AdamW)",
            "approx_tflops_per_gpu": flops / world / (ms * 1e-3) / 1e12,
            "flops_basis": "the reference's layer-by-layer algorithmic FLOPs (SURVEY 8d: 3 passes x (fwd + 2x bwd)); the "
                           "folded step (DESIGN 4.3) executes ~2.6x fewer tensor-core FLOPs for the same gradient",
            "collectives_per_step": 1 if world > 1 else 0,
            "allreduce_bytes_per_step": 4 * algo._trainer_state.packed.numel() if world > 1 else 0}


def step_kernel_rooflines(torch, _lib, env, eng, cfg, n_edges: float, n_agents: int, step_ms: float):
    """Times every kernel of the env-step ALONE (gcbf_rollout_step_select: one launch per call, 40 calls captured in
    one CUDA graph, CUDA events around its replay, on the buffers the last full step left behind -- i.e. warm L2 and
    back-to-back launches, like inside the rollout graph), picks the one with the largest share and reports its
    algorithmic work / time against the measured peaks."""
    import ctypes as C
    hbm, tf_burst, tf_sus, src = load_peaks()
    lib = env.lib
    ch = eng.chains[0]
    d = ch.desc
    t = 1
    b = t % 2
    obs = eng.obstacles[ch.e0].data_ptr() if eng.O > 0 else None
    REP = 40

    def enqueue(select: int, stream: int):
        rc = lib.gcbf_rollout_step_select(
            C.byref(d), eng.params_buf.data_ptr(), eng.infer_blob.data_ptr(), 1,
            eng.agent[t, ch.e0].data_ptr(), eng.goal[ch.e0].data_ptr(), obs, env.ray_table.data_ptr(),
            eng.hits[t, ch.e0].data_ptr(), ch.row_start[b].data_ptr(), ch.row_deg[b].data_ptr(),
            ch.edge_recv[b].data_ptr(), ch.edge_src[b].data_ptr(), ch.counters[t].data_ptr(),
            eng.actions[t, ch.e0].data_ptr(), eng.agent[t + 1, ch.e0].data_ptr(), eng.hits[t + 1, ch.e0].data_ptr(),
            ch.row_start[1 - b].data_ptr(), ch.row_deg[1 - b].data_ptr(), ch.edge_recv[1 - b].data_ptr(),
            ch.edge_src[1 - b].data_ptr(), ch.counters[t + 1].data_ptr(), eng.rewards[t, ch.e0:].data_ptr(),
            eng.costs[t, ch.e0:].data_ptr(), ch.ws.data_ptr(), ch.ws.numel(), select, stream)
        _lib.check(rc, "gcbf_rollout_step_select")

    if not eng.use_tc:
        return None
    # bring the buffers of step t into the state a rollout leaves them in (edge lists of state t in half b)
    st = torch.cuda.current_stream(env.device).cuda_stream
    eng._build(ch, t, st)
    enqueue(31, st)
    torch.cuda.synchronize()
    us = []
    for k in range(5):
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            s = torch.cuda.current_stream(env.device).cuda_stream
            for _ in range(REP):
                enqueue(1 << k, s)
        g.replay()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(3):
            g.replay()
        e1.record()
        torch.cuda.synchronize()
        us.append(e0.elapsed_time(e1) * 1e3 / (3 * REP))
    total = sum(us)
    fe, fn = folded_flops(cfg)
    nu = 3 if cfg["env"] == "LinearDrone" else 2
    ed = {"SingleIntegrator": 2, "DoubleIntegrator": 4, "DubinsCar": 4, "LinearDrone": 6}[cfg["env"]]
    sd = {"SingleIntegrator": 2, "DoubleIntegrator": 4, "DubinsCar": 4, "LinearDrone": 6}[cfg["env"]]
    pd = 3 if cfg["env"] == "LinearDrone" else 2
    R = env.n_hits
    # algorithmic work per launch (flops, compulsory bytes): per edge / per agent figures x the units of one launch
    rays = env.n_rays_cast
    ray_flops = rays * max(cfg["obs"], 1) * (4 * 30 if pd == 2 else 40)        # SURVEY 8d: ~30 FLOP per ray-edge test
    work = [
        (n_edges * fe, n_edges * (2 * 4 + 4 * sd * 2 + 4 * 128 + 4)),                        # idx + states in, MSG + logit out
        (n_edges * (2 * 128 + 8), n_edges * (4 * 128 + 4) + n_agents * (8 + 4 * 128)),        # MSG + logit in, AG out
        (n_agents * 2 * 128 * 256, n_agents * 4 * (128 + 256)),
        (n_agents * 2 * (256 * 256 + 256 * nu), n_agents * 4 * (256 + 4)),
        (n_agents * (ray_flops + 8 * cfg["N"]), n_agents * (4 * sd * 3 + 4 * nu + 4 * pd * R + 8) + n_edges * 8),
    ]
    kernels = []
    for k in range(5):
        fl, by = work[k]
        kernels.append({"kernel": STEP_KERNELS[k], "us": us[k], "share": us[k] / total,
                        "algorithmic_gflop": fl / 1e9, "achieved_tflops": fl / (us[k] * 1e-6) / 1e12,
                        "algorithmic_mb": by / 1e6, "achieved_gbs": by / (us[k] * 1e-6) / 1e9})
    dom = max(range(5), key=lambda k: us[k])
    fl, by = work[dom]
    tensor = dom in (0, 2, 3)
    alu = dom == 4 and pd == 3          # 3-D ray cast (514 rays x O spheres per agent): fp32-ALU work, tiny bytes (SURVEY 8d)
    fp32_peak = 148 * 128 * 2 * 1.965e9 / 1e12      # SMs x lanes x FMA x max SM clock = 74.4 TFLOP/s
    achieved = fl / (us[dom] * 1e-6) / 1e12 if (tensor or alu) else by / (us[dom] * 1e-6) / 1e9
    peak = tf_burst if tensor else (fp32_peak if alu else hbm)
    traffic = load_traffic(dom)
    return {"kernel": STEP_KERNELS[dom], "bound": "tensor" if tensor else ("fp32-alu" if alu else "hbm"), "achieved": achieved,
            "peak": peak, "unit": "TFLOP/s" if (tensor or alu) else "GB/s", "frac": achieved / peak,
            "peak_source": src + (" bf16 cuBLAS burst (MEASURED_PEAKS.json; the kernel computes fp32-class results with "
                                  "3 tf32 MMAs per product, so its own ceiling is 1/6 of this)" if tensor else
                                  (" -- no measured fp32 figure: 148 SMs x 128 lanes x 2 x 1.965 GHz (stated fallback)" if alu
                                   else " HBM copy")),
            "us_per_launch": us[dom], "share_of_step": us[dom] / total,
            "algorithmic_flops": fl, "algorithmic_bytes": by, "traffic": traffic["bytes"] if traffic else None,
            "traffic_source": traffic["source"] if traffic else "no ncu capture of this build under profiles/ (null)",
            "step_kernels": kernels, "sum_of_isolated_us": total, "measured_step_us": step_ms * 1e3,
            "whole_step": {"algorithmic_gflop_folded": (n_edges * fe + n_agents * fn) / 1e9,
                           "achieved_tflops_folded": (n_edges * fe + n_agents * fn) / (step_ms * 1e-3) / 1e12,
                           "frac_of_bf16_peak": (n_edges * fe + n_agents * fn) / (step_ms * 1e-3) / 1e12 / tf_burst},
            "note": "each kernel timed alone: 40 back-to-back launches in a CUDA graph (warm L2, the buffers of a real "
                    "step), CUDA events; algorithmic FLOPs count the folded fp32-equivalent work (2 M K N per GEMM), "
                    "not the 3x tf32 MMAs the tensor pipe executes"}


PHASES = ["edge phase: features + message layer + chained gate GEMM -> logits", "segment softmax + aggregate",
          "update layer GEMM 128->256", "folded update/head GEMM 256->256 + output partial sums",
          "policy tail (tanh, 2 pi + u_ref, clip, Euler, record, reward / cost)", "LiDAR + top-k + neighbour bits",
          "cluster prefix + edge-list fill"]


def persistent_roofline(torch, env, algo, g0, cfg, E, n_edges, n_agents, ms_rollout, T, five_launch):
    """The timed graph of the persistent path is ONE kernel (rollout_persist_kernel: the whole T-step rollout): its
    roofline entry is the algorithmic (folded, fp32-equivalent) FLOPs of the rollout over its measured duration.  The
    phase breakdown comes from %globaltimer stamps the kernel writes (environment 0's first CTA, a separate 32-step run);
    the isolated timings of the 5-launch path's kernels are kept for comparison."""
    from gcbfplus_b200.trainer.rollout import RolloutEngine
    hbm, tf_burst, tf_sus, src = load_peaks()
    fe, fn = folded_flops(cfg)
    flops_rollout = (n_edges * fe + n_agents * fn) * T
    achieved = flops_rollout / (ms_rollout * 1e-3) / 1e12
    Tp = 32
    eng2 = RolloutEngine(env, E, T=Tp, n_obs=cfg["obs"], use_cuda_graph=False, persistent=True)
    eng2.phase_stamps = torch.zeros(Tp + 1, 8, dtype=torch.int64, device=env.device)
    eng2.set_params(algo.actor_params)
    eng2.set_initial(g0.agent, g0.goal, g0.obstacle)
    eng2.run()
    eng2.run()
    torch.cuda.synchronize()
    st = eng2.phase_stamps.cpu().numpy().astype("float64")[2:]          # skip the build row and the first step
    d = (st[:, 1:] - st[:, :-1]).mean(axis=0) / 1e3                      # us per phase
    step_us = float((st[-1, 7] - st[0, 0]) / 1e3 / (len(st) - 1 + 1e-9)) if len(st) > 1 else float(d.sum())
    traffic = load_traffic(5)
    return {"kernel": "rollout_persist_kernel (one launch = the whole T-step rollout; 8 CTAs per environment as hardware "
                      "clusters of 2 + one software barrier per step when 16 x 8-CTA clusters do not co-reside)",
            "bound": "tensor", "achieved": achieved, "peak": tf_burst, "unit": "TFLOP/s", "frac": achieved / tf_burst,
            "peak_source": src + " bf16 cuBLAS burst (MEASURED_PEAKS.json); fp32-class results cost 3 tf32 MMAs per "
                                 "product, so the kernel's own tensor ceiling is 1/6 of this",
            "us_per_launch": ms_rollout * 1e3, "algorithmic_flops": flops_rollout,
            "algorithmic_bytes": cfg["B_alg"] * n_agents * T,
            "traffic": traffic["bytes"] if traffic else None,
            "traffic_source": traffic["source"] if traffic else "no ncu capture of this build under profiles/ (null)",
            "hbm_frac": cfg["B_alg"] * n_agents * T / (ms_rollout * 1e-3) / 1e9 / hbm,
            "phases_us": {PHASES[i]: float(d[i]) for i in range(7)}, "phase_sum_us": float(d.sum()),
            "in_kernel_step_us": step_us,
            "five_launch_path": {"step_kernels": five_launch["step_kernels"] if five_launch else None,
                                 "sum_of_isolated_us": five_launch["sum_of_isolated_us"] if five_launch else None},
            "note": "achieved = folded fp32-equivalent FLOPs of the rollout (2 M K N per GEMM, not the 3x tf32 MMAs executed) "
                    "/ CUDA-event time of the launch; the step is a dependent chain of 5 phases per environment, bound by "
                    "per-CTA latency (MMA issue, operand production, TMEM read-out), not by HBM or tensor throughput"}


def load_traffic(kernel_index: int):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of step kernel `kernel_index`, from the ncu --set full
    capture of THIS build (profiles/r02_traffic.json, written by tools/ncu_traffic.py with the source digest of the
    build it profiled).  None when absent or stale -- never a hard-coded number."""
    p = os.path.join(ROOT, "profiles", "r02_traffic.json")
    if not os.path.exists(p):
        return None
    try:
        from gcbfplus_b200 import build as _b
        d = json.load(open(p))
        ent = d.get("kernels", {}).get(str(kernel_index))
        if ent is None:
            return None
        stale = d.get("source_digest") != _b._digest()
        return {"bytes": ent["dram_bytes_per_launch"],
                "source": f"profiles/r02_traffic.json ({ent['ncu_kernel']}, {ent['launches']} launches, ncu --set full"
                          + (", captured on an EARLIER build of the sources" if stale else ", this build") + ")"}
    except Exception:
        return None


# ======================================================================================== CPU arm
def cpu_baseline(cfg, steps: int = 1, warmup: int = 1, verbose: bool = False):
    """Restated reference (dense padded formulation), torch-CPU fp32, on a bounded sample: ONE env of the workload,
    `steps` timed env-steps after `warmup`.  The thread count is the fastest of a probe AT THE WORKLOAD'S SIZE
    (one dense policy forward per candidate)."""
    import numpy as np
    import torch
    from helpers import oracle_env, oracle_params
    from oracle.algo import act
    from oracle.geometry import Rectangle, Sphere
    ncpu = os.cpu_count() or 1
    rng = np.random.Generator(np.random.PCG64(0))
    env_id, N, area, n_obs = cfg["env"], cfg["N"], cfg["area"], cfg["obs"]
    ap, _ = oracle_params(env_id)
    oenv = oracle_env(env_id, N, area, n_obs, cfg["rays"])
    pd, sd = oenv.pos_dim, oenv.state_dim
    if pd == 2:
        obs = Rectangle.create(rng.uniform(0, area, (n_obs, 2)), rng.uniform(0.1, 0.5, n_obs),
                               rng.uniform(0.1, 0.5, n_obs), rng.uniform(0, 2 * np.pi, n_obs))
    else:
        obs = Sphere.create(rng.uniform(0, area, (n_obs, 3)), rng.uniform(0.075, 0.15, n_obs))
    agent = torch.zeros(N, sd)
    agent[:, :pd] = torch.from_numpy(rng.uniform(0, area, (N, pd)).astype(np.float32))
    goal = torch.zeros(N, sd)
    goal[:, :pd] = torch.from_numpy(rng.uniform(0, area, (N, pd)).astype(np.float32))
    cands = sorted({c for c in (ncpu, ncpu // 2, 64, 32, 16, 8) if 1 <= c <= ncpu}, reverse=True)
    timings = {}
    with torch.no_grad():
        g = oenv.get_graph(agent, goal, obs)
        for c in cands:                               # probe at the workload's own size
            torch.set_num_threads(c)
            act(oenv, ap, g)
            t0 = time.perf_counter()
            act(oenv, ap, g)
            timings[c] = time.perf_counter() - t0
        cores = min(timings, key=timings.get)
        torch.set_num_threads(cores)
        times = []
        for s in range(warmup + steps):
            t0 = time.perf_counter()
            a = act(oenv, ap, g)                     # dense: all padded edges, like the reference
            g, r, c = oenv.step(g, a)
            if s >= warmup:
                times.append(time.perf_counter() - t0)
        sec = sum(times) / max(len(times), 1)
        # same step with the masked edges dropped first (the CUDA path's formulation) -> separates the algorithmic
        # (dense -> sparse) factor from the hardware (CPU -> B200) one, BASELINE.md section 3
        sparse_times = []
        for s in range(2):
            t0 = time.perf_counter()
            gs = oenv.sparsify(g)
            a = act(oenv, ap, gs)
            g, r, c = oenv.step(gs, a)
            if s > 0:
                sparse_times.append(time.perf_counter() - t0)
    sec_sparse = sum(sparse_times) / max(len(sparse_times), 1)
    n_dense = g.edges.shape[0] if hasattr(g, "edges") else 0
    return {"value": N / sec, "unit": "env-steps/s", "cores": cores, "kind": "port", "sparse_value": N / sec_sparse,
            "sample": f"1 env x n={N} x {len(times)} timed env-step(s) after {warmup} warm-up step(s) of the restated "
                      f"reference (oracle/, dense padded formulation, torch-CPU fp32; NOT the JAX code); {sec:.2f} s per "
                      f"env-step; {cores} of {ncpu} host threads (fastest of {cands} on a dense forward at n={N}: "
                      + ", ".join(f"{c}: {timings[c]:.2f} s" for c in cands) + ")",
            "sec_per_env_step": sec, "steps_run": len(times)}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from helpers import probe_reference_stack
    cfg = CONFIGS[args.config]
    world = int(os.environ.get("WORLD_SIZE", "1"))
    t0 = time.perf_counter()
    # every "step" of this arm is ONE env-step of ONE env (bounded sample); W warm-up + exactly K timed steps are run
    cpu = cpu_baseline(cfg, steps=args.steps, warmup=args.warmup)
    value = cpu["value"]
    out = {"impl": "reference", "metric": metric_name(cfg), "value": value, "unit": "env-steps/s", "n_gpus": world,
           "steps": cpu["steps_run"], "warmup": args.warmup, "ms_per_step": cpu["sec_per_env_step"] * 1e3,
           "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
           "config": {"workload": f"{cfg['env']} n={cfg['N']} obs={cfg['obs']} n_rays={cfg['rays']} area={cfg['area']} "
                                  f"({cfg['name']}); bounded sample: per step ONE env-step of ONE env",
                      "arm": "restated reference (CPU oracle port, dense formulation) -- not the JAX code",
                      "reference_stack_probe": probe_reference_stack()},
           "cpu_baseline": {k: cpu[k] for k in ("value", "unit", "cores", "kind", "sample", "sparse_value")},
           "e2e": {"value": value, "unit": "env-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
           "gpu_launches": 0, "wall_s": time.perf_counter() - t0}
    print(json.dumps(out))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", type=str, default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", type=int, default=3, choices=sorted(CONFIGS))
    ap.add_argument("--envs-per-gpu", type=int, default=None,
                    help="default: the config's envs / its GPU count (16, 4, 8)")
    ap.add_argument("--T", type=int, default=T_STEPS)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-train", action="store_true")
    ap.add_argument("--train-only", action="store_true",
                    help="profiling aid: one short rollout, then the train-step measurement alone (prints its dict)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the last rollout's records (agent, actions, rewards, costs, hits, "
                         "n_edges) as DIR/<name>.npy, at most 64 MB in all (rank 0's environments)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "ours" or args.train_only):
        ap.error("--dump-outputs records the rollout of --impl ours and is not available with --train-only")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
