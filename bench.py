#!/usr/bin/env python
"""bench.py - headline benchmark: learner.update() env-steps/s, PPO-Clip 256 envs x 128 steps, Atari-shaped.

    python bench.py --gpus N --steps K --warmup W             (N > 1 is launched by torchrun, one rank per GPU)
    python bench.py --impl reference --gpus N --steps K --warmup W   (the reference's torch-CPU path, rank 0 only)

A "step" is one pass of the hot path over one resident synthetic rollout: ``train_epochs(n_epochs=4)`` =
4 x shuffle + 16 x (memory.sample(8192) + learner.update), exactly the loop of
xuance/torch/agents/core/on_policy.py:182-205.  env-steps/s = N*T*K / (device time of K steps, max over ranks).
Strong scaling: the 256 x 128 rollout and the 8192-row global minibatch are fixed, rank g owns 256/G envs and
contributes 8192/G rows to every update; one NCCL all-reduce of the 13.4 MB flat gradient bucket per update.

Prints ONE JSON line (see DESIGN.md "Measurement" for every field)."""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

N_ENVS, HORIZON, N_ACTIONS = 256, 128, 4
OBS_SHAPE = (84, 84, 4)
N_EPOCHS, N_MINIBATCH = 4, 4
METRIC = "learner.update() env-steps/s, PPO 256x128 Atari-shaped"
UNIT = "env-steps/s"
WORKLOAD = ("PPO-Clip train_epochs(4) = 16 x (sample 8192 + update) over a resident 256 envs x 128 steps rollout, "
            "84x84x4 uint8 obs, NatureCNN actor-critic 3.36M params (BASELINE.json configs[1])")


# ------------------------------------------------------------------------------------------------ helpers
def measured_peaks():
    """(HBM GB/s, sustained dense bf16 TFLOP/s, source)."""
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            d = json.load(open(p))
            return float(d["hbm_gbs"]), float(d.get("bf16_tflops_sustained", 1400.0)), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, 1400.0, "fallback (B200_PROFILING.md)"


def ncu_traffic(kernel_key):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch from the committed `ncu --set full` capture of that kernel at the
    bench shape (profiles/r02_traffic.json, written by tools/ncu_traffic.py from the .ncu-rep); None when not captured."""
    p = os.path.join(ROOT, "profiles", "r02_traffic.json")
    try:
        return json.load(open(p)).get(kernel_key, {}).get("dram_bytes_per_launch")
    except Exception:
        return None


class ClockSampler:
    """nvidia-smi clocks + throttle reasons sampled every 200 ms while the timed region runs."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index=0):
        self.gpu, self.proc, self.lines = gpu_index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._pump, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                mx.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def ppo_namespace(device, n_envs_local, distributed, compute):
    from argparse import Namespace
    return Namespace(agent="PPO", learner="PPO_Learner", representation="AC_CNN_Atari", env_name="Atari",
                     distributed_training=distributed, device=device, seed=1, parallels=N_ENVS,
                     running_steps=10_000_000, horizon_size=HORIZON, n_epochs=N_EPOCHS, n_minibatch=N_MINIBATCH,
                     learning_rate=2.5e-4, vf_coef=0.25, ent_coef=0.01, clip_range=0.2, gamma=0.99, use_gae=True,
                     gae_lambda=0.95, use_advnorm=True, use_grad_clip=True, grad_clip_norm=0.5,
                     use_obsnorm=False, use_rewnorm=False, obsnorm_range=5, rewnorm_range=5, activation="relu",
                     filters=[32, 64, 64], kernels=[8, 4, 3], strides=[4, 2, 1], fc_hidden_sizes=[512],
                     actor_hidden_size=[], critic_hidden_size=[], model_dir="models/ppo", log_dir="logs/ppo",
                     logger=None, compute=compute, use_linear_lr_decay=False, end_factor_lr_decay=1.0,
                     episode_length=None)


def synth_scalars(rng, T, N):
    acts = rng.integers(0, N_ACTIONS, size=(T, N)).astype(np.float32)
    rews = rng.choice(np.array([-1.0, 0.0, 1.0], np.float32), size=(T, N), p=[0.05, 0.9, 0.05])
    vals = rng.normal(size=(T, N)).astype(np.float32)
    terms = (rng.random((T, N)) < 0.01).astype(np.float32)
    logits = rng.normal(size=(T, N, N_ACTIONS)).astype(np.float32)
    logp = (np.take_along_axis(logits, acts.astype(np.int64)[..., None], -1)[..., 0]
            - np.log(np.exp(logits).sum(-1))).astype(np.float32)
    boot = rng.normal(size=N).astype(np.float32)
    return acts, rews, vals, terms, logp, boot


# ------------------------------------------------------------------------------------------------ reference arm
def cpu_reference_rate(rows_budget_s, steps, warmup, threads=None, verbose=False):
    """Times the reference's torch-CPU path (oracle port of DummyOnPolicyBuffer_Atari.sample + PPO_Learner.update on
    the NatureCNN actor-critic) on a bounded sample of the workload.  Returns (env_steps_per_s per step list, info)."""
    import torch
    from oracle.onpolicy import OnPolicyBufferOracle
    from oracle.nets import SharedActorCriticOracle
    from oracle.learners import PPOLearnerOracle
    # all the host cores: one intra-op thread per PHYSICAL core (torch's own default when OMP_NUM_THREADS is unset -
    # torchrun sets it to 1, so it is set explicitly here); SMT oversubscription (one thread per logical CPU) is slower
    if not threads:
        try:
            import psutil
            threads = psutil.cpu_count(logical=False) or os.cpu_count() or 1
        except Exception:
            threads = os.cpu_count() or 1
    torch.set_num_threads(int(threads))
    cores = torch.get_num_threads()
    torch.manual_seed(1)
    rng = np.random.default_rng(0)
    N, T = N_ENVS, HORIZON
    buf = OnPolicyBufferOracle(OBS_SHAPE, (), {"old_logp": ()}, N, T, obs_dtype=np.uint8)
    buf.observations = rng.integers(0, 256, size=(N, T) + OBS_SHAPE, dtype=np.uint8)
    acts, rews, vals, terms, logp, boot = synth_scalars(rng, T, N)
    buf.actions[...], buf.rewards[...], buf.values[...] = acts.T, rews.T, vals.T
    buf.terminals[...], buf.aux["old_logp"][...] = terms.T, logp.T
    buf.ptr, buf.size = 0, T
    t0 = time.perf_counter()
    for i in range(N):
        buf.finish_path(0.0 if terms[T - 1, i] else boot[i], i)
    t_gae = time.perf_counter() - t0
    model = SharedActorCriticOracle(N_ACTIONS)
    lrn = PPOLearnerOracle(model, total_iters=1000)
    np.random.seed(1)
    perm = np.arange(N * T)
    np.random.shuffle(perm)
    # calibrate: rows/s from the second of two 512-row sample+update calls (the first pays one-time oneDNN setup)
    lrn.update(**buf.sample(perm[:512]))
    t0 = time.perf_counter()
    lrn.update(**buf.sample(perm[:512]))
    per_row = (time.perf_counter() - t0) / 512
    rows = int(min(8192, max(256, rows_budget_s / max(per_row, 1e-9))))
    rates, pos = [], 512
    for it in range(warmup + steps):
        if pos + rows > perm.size:
            np.random.shuffle(perm)
            pos = 0
        t0 = time.perf_counter()
        lrn.update(**buf.sample(perm[pos:pos + rows]))
        dt = time.perf_counter() - t0
        pos += rows
        if it >= warmup:
            rates.append((rows / N_EPOCHS) / dt)   # one env-step is visited n_epochs times by train_epochs
    info = {"cores": cores, "logical_cpus": os.cpu_count(), "rows_per_step": rows, "finish_path_256_s": t_gae,
            "sample": "%d timed steps, each = sample(%d rows)+update of the 256x128 workload; env-steps = rows/%d"
                      % (steps, rows, N_EPOCHS)}
    return rates, info


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    budget = 150.0 / max(1, args.steps + args.warmup)
    rates, info = cpu_reference_rate(min(budget, 20.0), args.steps, args.warmup)
    value = float(np.mean(rates))
    rows = info["rows_per_step"]
    ms = 1000.0 * (rows / N_EPOCHS) / value
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": WORKLOAD, "arm": "reference torch-CPU path (oracle port: the reference is Python "
                       "and /root/reference does not travel to the GPU box)", "cpu_threads": info["cores"]},
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": info["cores"], "kind": "port",
                             "sample": info["sample"]},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------------ own arm
_T0 = time.time()


def parity_vs_single(agent, world):
    """Hardware evidence that G ranks compute the 1-GPU update: one global minibatch (every rank contributes batch_size of
    its own rollout rows) is applied (1) sharded - K4 scaled by 1/B_total, ONE sum all-reduce of gradient + statistics, K7 -
    and (2) by every rank alone on the all-gathered 8192 rows; the two parameter vectors are compared.  State is restored."""
    import torch
    import torch.distributed as dist
    lrn, mem = agent.learner, agent.memory
    snap, its, sched = lrn.optimizer.snapshot(), lrn.iterations, lrn.scheduler.state_dict()
    B = agent.batch_size
    idx = torch.arange(B, device=mem.device, dtype=torch.int64) * (agent.buffer_size // B)
    stats = mem.global_adv_stats(idx, 1)[0]
    s = mem.sample(idx, stats)
    local = [s["obs"], s["actions"].float().contiguous(), s["returns"].contiguous(), s["advantages"].contiguous(),
             s["aux_batch"]["old_logp"].contiguous()]
    lrn.optimizer.prepare()
    lrn._device_update(*local)
    torch.cuda.synchronize()
    p_dist = lrn.optimizer.bucket.flat.clone()
    lrn.optimizer.restore(snap)

    def gather(x):
        parts = [torch.empty_like(x) for _ in range(world)]
        dist.all_gather(parts, x.contiguous())
        return torch.cat(parts)
    full = [gather(x) for x in local]
    ws, lrn.world_size = lrn.world_size, 1
    lrn.optimizer.prepare()
    lrn._device_update(*full)
    lrn.world_size = ws
    torch.cuda.synchronize()
    p_single = lrn.optimizer.bucket.flat.clone()
    lrn.optimizer.restore(snap)
    lrn.iterations = its
    lrn.scheduler.load_state_dict(sched)
    d = torch.stack([(p_dist - p_single).abs().max(), (p_single - snap[0]).abs().max()]).double()
    dist.all_reduce(d, op=dist.ReduceOp.MAX)
    # time the one collective of an update in isolation (gradient bucket + statistics tail)
    buf = lrn.optimizer.bucket.grad_all
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for _ in range(3):
        dist.all_reduce(buf)
    torch.cuda.synchronize()
    a.record()
    for _ in range(10):
        dist.all_reduce(buf)
    b.record()
    torch.cuda.synchronize()
    lrn.optimizer.bucket.grad_all.zero_()
    return {"max_abs_param_diff": float(d[0]), "max_abs_param_step": float(d[1]), "global_rows": B * world,
            "what": "same global minibatch, sharded over %d ranks vs every rank alone on the gathered rows; one Adam step" % world,
            "allreduce_ms": a.elapsed_time(b) / 10.0, "allreduce_bytes": buf.numel() * 4}


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(out_dir, info, model):
    """What a caller of the timed path holds after its last step: the info dict train_epochs returned (float64 scalars,
    info.<key>.npy) and the parameters that step left in the model (float32, param.<name>.npy; 13.4 MB at this workload)."""
    arrays = {}
    for k, v in info.items():
        for kk, vv in (v.items() if isinstance(v, dict) else [("", v)]):
            arrays["info.%s%s" % (k, "." + kk if kk else "")] = np.asarray(float(vv), np.float64)
    for k, v in model.state_dict().items():
        arrays["param." + k] = v.detach().float().cpu().numpy()
    total = sum(a.nbytes for a in arrays.values())
    assert total <= DUMP_LIMIT_BYTES, "outputs to dump: %d bytes" % total
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)
    return total


def _log(msg):
    if os.environ.get("XB_BENCH_VERBOSE", "1") != "0":
        sys.stderr.write("[bench %6.1fs rank %s] %s\n" % (time.time() - _T0, os.environ.get("RANK", "0"), msg))
        sys.stderr.flush()


def run_own_arm(args):
    import torch
    import torch.distributed as dist
    from xuance_b200 import _lib
    from xuance_b200.common import Box, Discrete
    from xuance_b200.torch.agents import PPO_Agent
    from xuance_b200.torch.utils import init_distributed_mode

    _log("imports done")
    rank, world, local_rank = init_distributed_mode()
    _log("process group ready (world %d)" % world)
    if world > 1:
        assert world == args.gpus, "torchrun world size must equal --gpus"
    torch.cuda.set_device(local_rank)
    device = "cuda:%d" % local_rank
    torch.backends.cudnn.allow_tf32 = args.compute not in ("fp32", "fp32_cl", "tc")
    torch.backends.cuda.matmul.allow_tf32 = args.compute not in ("fp32", "fp32_cl", "tc")
    torch.backends.cudnn.benchmark = True
    assert N_ENVS % world == 0
    n_local = N_ENVS // world
    if args.shard_of > 1:      # diagnostic: ONE rank's share of a --shard-of G job run alone (no collective): its step time
        assert world == 1      # bounds the G-GPU scaling efficiency from the compute side; the line is marked, not a bench value
        n_local = N_ENVS // args.shard_of
    cfg = ppo_namespace(device, n_local, world > 1, args.compute)
    cfg.tc_planes = args.tc_planes
    if args.shard_of > 1:
        cfg.parallels = n_local
    cfg.use_cuda_graph = bool(args.graph) if args.graph >= 0 else True     # same execution mode at every N
    obs_space, act_space = Box(0, 255, OBS_SHAPE, np.uint8), Discrete(N_ACTIONS)
    agent = PPO_Agent(cfg, envs=None, observation_space=obs_space, action_space=act_space)  # buffer: n_local envs
    assert agent.n_envs == n_local
    torch.manual_seed(1)  # identical initial weights on every rank
    for p in agent.model.parameters():
        if world > 1:
            dist.broadcast(p.data, src=0)
    mem, T = agent.memory, HORIZON

    # ---- synthetic rollout: scalars from NumPy (global, sliced per rank), frames generated on the device
    rng = np.random.default_rng(0)
    acts, rews, vals, terms, logp, boot = synth_scalars(rng, T, N_ENVS)
    lo, hi = rank * n_local, (rank + 1) * n_local
    sl = lambda a: a[:, lo:hi]
    g = torch.Generator(device=device).manual_seed(100 + rank)
    host_obs = None
    if args.e2e_steps > 0:
        host_obs = torch.empty((T, n_local) + OBS_SHAPE, dtype=torch.uint8).pin_memory()
    for t in range(T):
        frame = torch.randint(0, 256, (n_local,) + OBS_SHAPE, dtype=torch.uint8, device=device, generator=g)
        if host_obs is not None:
            host_obs[t].copy_(frame)
        mem.store(frame, torch.from_numpy(sl(acts)[t]).to(device), torch.from_numpy(sl(rews)[t]).to(device),
                  torch.from_numpy(sl(vals)[t]).to(device), torch.from_numpy(sl(terms)[t]).to(device),
                  {"old_logp": torch.from_numpy(sl(logp)[t]).to(device)})
    for i in range(n_local):
        mem.finish_path(0.0 if terms[T - 1, lo + i] else boot[lo + i], i)
    np.random.seed(1)
    _log("synthetic rollout resident")

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def step():
        return agent.train_epochs(N_EPOCHS)

    for _ in range(args.warmup):
        step()
        _log("warm-up step done")
    barrier()
    sampler = ClockSampler(local_rank) if rank == 0 else None
    if sampler:
        sampler.start()
    launches0 = _lib.launch_count
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record()
    for _ in range(args.steps):
        info = step()
    e1.record()
    barrier()
    elapsed_ms = e0.elapsed_time(e1)
    _log("timed region done: %.1f ms/step" % (elapsed_ms / args.steps))
    if args.dump_outputs and rank == 0:      # before anything below (e2e steps) moves the weights on
        _log("dumped %d bytes of outputs to %s" % (dump_outputs(args.dump_outputs, info, agent.model), args.dump_outputs))
    launches = _lib.launch_count - launches0
    clocks = sampler.stop() if sampler else None
    t = torch.tensor([elapsed_ms], dtype=torch.float64, device=device)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    elapsed_ms = float(t.item())
    value = N_ENVS * T * args.steps / (elapsed_ms / 1000.0)
    if args.shard_of > 1:
        print(json.dumps({"diagnostic": "one rank's shard of a %d-GPU job, alone, no collective" % args.shard_of,
                          "rows_per_update": n_local * T // N_MINIBATCH, "ms_per_step": elapsed_ms / args.steps,
                          "ms_per_update": elapsed_ms / args.steps / (N_EPOCHS * N_MINIBATCH),
                          "implied_value_at_%d_gpus_without_collective" % args.shard_of: value}))
        return

    # ---- e2e: rollout in pinned HOST memory -> 128 x store (H2D) + finish_path + train_epochs + info D2H
    e2e = None
    if args.e2e_steps > 0:
        h_np = host_obs.numpy()
        scal = [np.ascontiguousarray(sl(a)) for a in (acts, rews, vals, terms, logp)]

        def e2e_step():
            mem.clear()
            mem.start_ids[:] = 0
            for tt in range(T):
                mem.store(h_np[tt], scal[0][tt], scal[1][tt], scal[2][tt], scal[3][tt], {"old_logp": scal[4][tt]})
            for i in range(n_local):
                mem.finish_path(0.0 if terms[T - 1, lo + i] else boot[lo + i], i)
            out = agent.train_epochs(N_EPOCHS)      # last update materialises the info dict (D2H of 8 floats)
            return out

        e2e_step()
        barrier()
        a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        w0 = time.perf_counter()
        a0.record()
        for _ in range(args.e2e_steps):
            e2e_step()
        a1.record()
        barrier()
        wall = time.perf_counter() - w0
        tt = torch.tensor([max(a0.elapsed_time(a1) / 1000.0, wall)], dtype=torch.float64, device=device)
        if world > 1:
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        per_step = float(tt.item()) / args.e2e_steps
        _log("e2e done: %.1f ms/step" % (per_step * 1000))
        h2d = n_local * T * (int(np.prod(OBS_SHAPE)) + 5 * 4) + N_EPOCHS * n_local * T * 8
        e2e = {"value": N_ENVS * T / per_step, "unit": UNIT, "h2d_bytes_per_step": int(h2d) * world,
               "d2h_bytes_per_step": 32 * world, "steps": args.e2e_steps,
               "what": "128 x memory.store(pinned host arrays) + finish_path + train_epochs(4) + info dict read"}

    parity = parity_vs_single(agent, world) if world > 1 else None
    if parity:
        _log("parity vs 1 GPU: max |dp| = %.3g (step %.3g), all-reduce %.3f ms" % (
            parity["max_abs_param_diff"], parity["max_abs_param_step"], parity["allreduce_ms"]))

    # ---- roofline of the dominant kernels: CUDA events around every launch of ONE epoch (n_minibatch updates) replayed
    # eagerly right after the timed region (graph replays hide per-kernel events); same buffers, same shapes, same stream
    hbm_peak, tc_peak, peak_src = measured_peaks()
    roofline, kernel_ms = None, {}
    names = ["xb_gemm_gather_tc", "xb_gemm_box_tc", "xb_gemm_halo_tc", "xb_wgrad_gather_tc", "xb_wgrad_box_tc", "xb_wgrad_reduce", "xb_split_bf16",
             "xb_pack_conv_weight", "xb_pack_weights", "xb_gather_obs_planes", "xb_gather_obs", "xb_ppo_loss_fwd_bwd",
             "xb_adam_step", "xb_grad_sumsq", "xb_gather_scalars", "nccl_all_reduce"]
    from xuance_b200.torch.utils import tc_conv
    saved_graph = agent.config.use_cuda_graph
    agent.config.use_cuda_graph = False
    snap = agent.learner.optimizer.snapshot()
    its, sched_state = agent.learner.iterations, agent.learner.scheduler.state_dict()
    agent.train_epochs(1)                                   # warm the eager path (cuDNN / cuBLAS handles, allocator)
    barrier()
    _lib.profile = {n: [] for n in names}
    tc_conv.flop_log = []
    p0, p1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    p0.record()
    agent.train_epochs(1)
    p1.record()
    torch.cuda.synchronize()
    prof, flog = _lib.profile, tc_conv.flop_log
    _lib.profile, tc_conv.flop_log = None, None
    agent.learner.optimizer.restore(snap)
    agent.learner.iterations = its
    agent.learner.scheduler.load_state_dict(sched_state)
    agent.config.use_cuda_graph = saved_graph
    eager_epoch_ms = p0.elapsed_time(p1)
    for n in names:
        if prof[n]:
            kernel_ms[n] = float(sum(a.elapsed_time(b) for a, b in prof[n]))
    if flog:
        # pair the FLOP log with the events in launch order (each ABI name keeps its own ordered list)
        it_f = {n: iter(prof[n]) for n in ("xb_gemm_gather_tc", "xb_gemm_box_tc", "xb_gemm_halo_tc", "xb_wgrad_gather_tc", "xb_wgrad_box_tc")}
        per_layer, tot_fl, tot_eq, tot_ms = {}, 0.0, 0.0, 0.0
        for nm, tag, fl, eq in flog:
            a, b = next(it_f[nm])
            ms = a.elapsed_time(b)
            d = per_layer.setdefault(nm.replace("xb_", "").replace("_tc", "") + " " + tag, [0.0, 0.0, 0.0, 0])
            d[0] += ms; d[1] += fl; d[2] += eq; d[3] += 1
            tot_fl += fl; tot_eq += eq; tot_ms += ms
        n_upd = max(1, N_MINIBATCH)
        top = max(per_layer.items(), key=lambda kv: kv[1][0])
        ach = tot_fl / (tot_ms * 1e-3) / 1e12
        roofline = {"kernel": "conv_tc_kernel (K12: tcgen05 gathered-operand GEMM; %d launches per update: forward, data and "
                              "weight gradients of conv1-3 + the 6400->512 layer)" % (len(flog) // n_upd),
                    "bound": "tensor", "achieved": ach, "peak": tc_peak, "unit": "TFLOP/s", "frac": ach / tc_peak,
                    "traffic": ncu_traffic("conv_tc_kernel:update_B%d_P%d" % (N_ENVS * T // N_MINIBATCH // world, args.tc_planes)),
                    "peak_source": peak_src + ", bf16_tflops_sustained",
                    "algorithmic_flops_per_update": tot_fl / n_upd,
                    "what": "algorithmic bf16 tensor FLOPs = 2 x real output sites x N x K (padding / halo / garbage sites of the padded "
                            "layouts NOT counted) x the plane products float32-grade arithmetic keeps (6 for 3x3 planes, 3 for "
                            "the raw-pixel first layer) / summed CUDA-event time of the K12 launches; traffic = DRAM bytes of "
                            "those launches per update (ncu --set full of one update at this shape, profiles/r02_traffic.json)",
                    "fp32_equivalent_tflops": tot_eq / (tot_ms * 1e-3) / 1e12,
                    "avg_update_ms": tot_ms / n_upd, "launches_timed": len(flog),
                    "timed": "CUDA events around every K12 launch of one eager epoch run right after the timed region",
                    "share_of_step": (tot_ms * N_EPOCHS) / (elapsed_ms / args.steps),
                    "slowest_layer": {"layer": top[0], "ms_per_update": top[1][0] / n_upd,
                                      "tflops_executed": top[1][1] / (top[1][0] * 1e-3) / 1e12},
                    "per_layer_ms_per_update": {k: round(v[0] / n_upd, 4) for k, v in sorted(per_layer.items(), key=lambda kv: -kv[1][0])}}
    elif kernel_ms.get("xb_gather_obs"):
        B_local = (N_ENVS * T // N_MINIBATCH) // world
        obs_bytes = int(np.prod(OBS_SHAPE))
        out_w = {"fp32": 4, "fp32_cl": 4, "tf32": 4, "bf16": 2}.get(args.compute, 4)
        alg_bytes = B_local * obs_bytes * (1 + out_w) + 8 * B_local
        k3_ms = kernel_ms["xb_gather_obs"] / len(prof["xb_gather_obs"])
        ach = alg_bytes / (k3_ms * 1e-3) / 1e9
        roofline = {"kernel": "gather_obs_kernel (K3: minibatch gather + u8->float)", "bound": "hbm",
                    "achieved": ach, "peak": hbm_peak, "unit": "GB/s", "frac": ach / hbm_peak,
                    "traffic": ncu_traffic("gather_obs_kernel:%s:%d" % (args.compute, B_local)),
                    "peak_source": peak_src, "algorithmic_bytes_per_launch": alg_bytes,
                    "avg_launch_ms": k3_ms, "launches_timed": len(prof["xb_gather_obs"]),
                    "timed": "CUDA events around every K3 launch of one eager epoch run right after the timed region",
                    "share_of_step": (k3_ms * N_EPOCHS * N_MINIBATCH) / (elapsed_ms / args.steps)}
    phases = {"eager_epoch_ms": eager_epoch_ms, "own_kernels_ms_per_epoch": {k: round(v, 3) for k, v in kernel_ms.items()}}

    if rank != 0:
        return
    cpu = None
    if world == 1 and not args.no_cpu_baseline:
        rates, cinfo = cpu_reference_rate(8.0, 2, 0)
        cpu = {"value": float(np.mean(rates)), "unit": UNIT, "cores": cinfo["cores"], "kind": "port",
               "sample": cinfo["sample"]}
    line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": elapsed_ms / args.steps, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "f32" if args.compute != "bf16" else "bf16",
            "data": "synthetic",
            "config": {"workload": WORKLOAD, "global_minibatch": N_ENVS * T // N_MINIBATCH,
                       "parallelism": ("dp%d (envs sharded; ONE all-reduce of the flat gradient bucket + statistics per update%s)"
                                       % (world, "; XB_EARLY_ALLREDUCE=1: Linear + head gradients reduced early, two pieces"
                                          if os.environ.get("XB_EARLY_ALLREDUCE", "0") == "1" else ""))
                                      if world > 1 else "dp1 (single GPU, no collective)",
                       "compute": {"fp32": "fp32, TF32 disabled (reference arithmetic)", "fp32_cl": "fp32, TF32 disabled, channels-last convolutions", "tf32": "fp32 storage, TF32 convs/matmuls",
                                   "bf16": "bf16 autocast convs, fp32 master weights",
                                   "tc": "tcgen05 layers (K12): every fp32 operand as %d bf16 planes (exact to 2^-%d), raw uint8 pixels as "
                                         "one exact plane, fp32 accumulation in TMEM per product order; heads / loss / Adam fp32"
                                         % (args.tc_planes, 8 * args.tc_planes)}[args.compute],
                       "l2": "inputs (925 MB uint8 rollout / G) exceed the 126 MB L2; no explicit flush",
                       "cuda_graph": bool(cfg.use_cuda_graph)},
            "clocks": clocks, "e2e": e2e, "gpu_launches": launches, "roofline": roofline, "cpu_baseline": cpu,
            "phases": phases, "parity_vs_1gpu": parity,
            "last_info": {k: (float(v) if not isinstance(v, dict) else v) for k, v in info.items()}}
    print(json.dumps(line))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--shard-of", type=int, default=1, help="diagnostic (1 GPU): time one rank's shard of a G-GPU job alone")
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="xuance_b200", choices=["xuance_b200", "reference"])
    ap.add_argument("--compute", default="tc", choices=["fp32", "fp32_cl", "tf32", "bf16", "tc"],
                    help="'tc' (default) = the K12 tcgen05 layers, float32-grade split-bf16 arithmetic; 'fp32' = cuDNN / cuBLAS "
                         "CUDA-core fp32 (round 1's headline); 'tf32' / 'bf16' = reduced-precision library paths, for context")
    ap.add_argument("--tc-planes", type=int, default=3, choices=[2, 3],
                    help="with --compute tc: bf16 planes per operand (3 = float32-grade, 2 = ~1e-5 forward error)")
    ap.add_argument("--e2e-steps", type=int, default=3)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--graph", type=int, default=-1, help="CUDA-graph the minibatch update: 1/0; default: on (every N)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the last step's info dict and model parameters to DIR/<name>.npy "
                         "(inputs are seeded: the same arguments give the same inputs, so two builds can be compared)")
    args = ap.parse_args()
    if args.warmup < 3 and args.impl != "reference":
        args.warmup = 3
    # exactly ONE line on stdout: libraries (NCCL prints its version banner on fd 1) are diverted to stderr, the JSON
    # line goes to the real stdout at the end
    real_stdout = os.fdopen(os.dup(1), "w")
    sys.stdout.flush()
    os.dup2(2, 1)
    import builtins
    _print = builtins.print

    def emit(*a, **k):
        k.setdefault("file", real_stdout)
        _print(*a, **k)
        real_stdout.flush()

    g = globals()
    g["print"] = emit
    if args.impl == "reference":
        run_reference_arm(args)
    else:
        run_own_arm(args)
    try:
        import torch.distributed as dist
        if dist.is_available() and dist.is_initialized():
            dist.destroy_process_group()
    except Exception:
        pass


if __name__ == "__main__":
    main()
