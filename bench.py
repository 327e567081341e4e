#!/usr/bin/env python
"""bench.py - DrQ critic grad-steps/sec on B200 (BASELINE.json metric), one JSON line on stdout.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--precision fp32|bf16] [--dump-outputs DIR]
  torchrun --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...        (N > 1)

Workload = the configuration BASELINE.json's metric is quoted on ("B=256, 2x128x128 obs" = configs[2]): `async_drq_sim` with
its stock dual 128x128x3 cameras, batch 256 drawn 50/50 (RLPD) from the online replay ring and a 20-trajectory demo ring,
replay 200k in HBM (`--cams 1 --no-rlpd --capacity 100000` gives configs[1], also reported under "single_camera").
A "step" = one critic gradient step (`update_critics` equivalent) INCLUDING replay sampling + DrQ shift
(SURVEY.md §8d unit of work).  N > 1: the global batch of 256 is split across ranks (strong scaling), each rank
owns a shard of the online ring (the small demo ring is replicated), ONE gradient all-reduce(mean) per step.

  value      steps/s with everything resident in HBM, CUDA-event timed, max over ranks.
  e2e        the same through the public API with host buffers: every step inserts one fresh transition from
             pinned host memory (H2D), draws the batch with the replay iterator, runs agent.update_critics and
             reads the loss back (D2H).
  roofline   frozen ResNet-10 trunk (the dominant kernels): algorithmic FLOPs / CUDA-event time of the trunk
             section inside the timed steps, vs MEASURED_PEAKS.json's sustained bf16 tensor peak; `sampler` gives
             the HBM roofline of the sampler/crop kernel.
  cpu_baseline / --impl reference   the CPU restatement of the reference step (oracle/, torch-CPU fp32, all host
             threads; jax is not installable in this image) on a bounded sample of the same workload.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

TRUNK_GFLOP_PER_IMAGE = 0.5804          # SURVEY.md §8d: 290,193,408 MAC
FRAME_BYTES = 128 * 128 * 3


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--precision", default=os.environ.get("SERL_PRECISION", "fp16"), choices=["fp32", "bf16", "fp16"],
                    help="trunk arithmetic: fp16 (default: tensor cores, fp32 accumulate, meets the 1e-2 bar), bf16, or fp32 (1e-5 parity build)")
    ap.add_argument("--batch", type=int, default=256)
    ap.add_argument("--cams", type=int, default=2)
    ap.add_argument("--capacity", type=int, default=None, help="online replay slots (default 200k dual-camera, 100k single)")
    ap.add_argument("--no-rlpd", dest="rlpd", action="store_false", help="draw the whole batch from the online ring (configs[1])")
    ap.add_argument("--ref-rows", type=int, default=64, help="rows of the batch the CPU reference processes per step")
    ap.add_argument("--sustain-s", type=float, default=1.0, help="length of the additional sustained run (seconds of timed steps)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the --steps timed steps, write what the last of them returned (loss / Q / lr infos, updated parameters and "
                         "target parameters, a fixed sample of the Adam moments) as DIR/<name>.npy; the inputs depend only on the arguments")
    a = ap.parse_args()
    if a.capacity is None:
        a.capacity = 200_000 if a.cams == 2 else 100_000
    return a


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm=d["hbm_gbs"], tensor=d.get("bf16_tflops_sustained", d["bf16_tflops"]), src="measured (MEASURED_PEAKS.json, sustained bf16)")
    return dict(hbm=6650.0, tensor=1400.0, src="fallback (B200_PROFILING.md)")


# ------------------------------------------------------------------------------------------------
# CPU reference arm: the oracle port of the reference step (sample on host + update_critics), bounded sample
# ------------------------------------------------------------------------------------------------
def cpu_reference_steps(args, steps, warmup, rows, budget_s=None, reference_structure=True):
    """reference_structure: the JAX reference evaluates the frozen encoder once per network call - policy(s'), target
    critic(s') and critic(s) in critic_loss_fn (sac.py:118-176): THREE trunk passes of `rows` images per camera - while
    the oracle (like the B200 path) shares one pass over obs and one over next_obs.  For a timing that has the reference's
    structure the third pass (target critic on next_obs) is executed as well and its result discarded."""
    import torch
    from helpers import random_transitions
    from oracle import drq as O
    from oracle.replay import OracleFrameRing, unpack
    from serl_b200.params import init_trainable, init_trunk, trainable_spec
    cores = min(os.cpu_count() or 1, 32)                  # beyond ~32 threads the small convs of a bounded sample only contend
    torch.set_num_threads(cores)
    cams = tuple(f"cam{i}" for i in range(args.cams))
    rng = np.random.default_rng(0)
    spec = trainable_spec(cams, 7, 4, 10, True)
    params = {k: torch.as_tensor(v) for k, v in init_trainable(rng, spec, 1e-2).items()}
    for cam in cams:
        for k, v in init_trunk(rng).items():
            params[f"modules_actor/encoder/encoder_{cam}/pretrained_encoder/{k}"] = torch.as_tensor(v)
    state = O.OracleState.create(params, np.array([0, 42], np.uint32), torch.float32)
    cfg = O.OracleConfig(cams=cams)
    ring = OracleFrameRing(1200, cams, (128, 128, 3), 1, 7, 4)
    for tr in random_transitions(rng, 1000, cams, mean_ep=100):
        ring.insert(tr)
    times, t_begin = [], time.perf_counter()
    for s in range(warmup + steps):
        t0 = time.perf_counter()
        _, packed = ring.sample(0, s, rows)
        batch = unpack(packed)
        O.update_critics(state, cfg, batch, dtype=torch.float32)
        if reference_structure:
            O._features(state, cfg, batch["next_observations"], torch.float32)
        dt = time.perf_counter() - t0
        if s >= warmup:
            times.append(dt)
        if budget_s is not None and times and time.perf_counter() - t_begin > budget_s:
            break                                          # bounded sample: stop once the time budget is spent
    t = sum(times) / len(times)
    # a full step processes `batch` rows; the sample processed `rows`: scale linearly (trunk-dominated, per-row cost)
    return (rows / args.batch) / t, t, cores, len(times)


def run_reference(args):
    rank = int(os.environ.get("RANK", 0))
    if rank != 0:
        return
    v, t, cores, done = cpu_reference_steps(args, args.steps, min(args.warmup, 1), args.ref_rows, budget_s=150.0)
    sample = (f"{done} timed steps (150 s budget) of {args.ref_rows} of {args.batch} rows per step: host numpy sampling + torch-CPU fp32 "
              f"restatement of update_critics with the reference's three frozen-encoder passes (policy(s'), target critic(s'), critic(s)); "
              f"steps/s EXTRAPOLATED x{args.batch / args.ref_rows:g} by rows/batch (per-row cost dominates); jax[cpu] is not installable here")
    line = {"metric": "drq_critic_grad_steps_per_sec", "value": v, "unit": "steps/s", "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1e3 / v, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic", "impl": "reference",
            "config": workload_config(args),
            "cpu_baseline": {"value": v, "unit": "steps/s", "cores": cores, "kind": "port", "sample": sample,
                             "extrapolated_x": args.batch / args.ref_rows},
            "e2e": {"value": v, "unit": "steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


TRUNK_KERNELS = {
    False: "frozen ResNet-10 trunk, fp32 build (conv_igemm_f32 + groupnorm_f32 + maxpool3x3s2_f32)",
    True: "frozen ResNet-10 trunk, tcgen05 build (stem_tc + conv3x3_tc + conv_tc kernels and their elementwise GroupNorm / pool / residual passes)",
}


def trunk_traffic(args):
    """DRAM bytes per step of the trunk kernels (dram__bytes_read.sum + dram__bytes_write.sum summed over the trunk's launches of
    one step) from the committed ncu capture of this same command, or None when no capture matches the configuration."""
    path = os.path.join(os.path.dirname(os.path.abspath(__file__)), "profiles", "trunk_traffic.json")
    try:
        with open(path) as f:
            t = json.load(f)
        key = f"{args.precision}_b{args.batch // max(int(os.environ.get('WORLD_SIZE', 1)), 1)}_c{args.cams}"
        return t.get(key, {}).get("dram_bytes_per_step")
    except (OSError, ValueError):
        return None


def workload_config(args):
    rl = (f" = {args.batch // 2} online + {args.batch - args.batch // 2} demo (50/50 RLPD, demo ring of 20 trajectories)" if args.rlpd else "")
    name = "BASELINE configs[2]" if (args.cams == 2 and args.rlpd) else ("BASELINE configs[1]" if args.cams == 1 and not args.rlpd else "custom")
    if args.cams == 2 and args.batch == 2048:
        name = "BASELINE configs[3] (dual camera, batch 2048, replay 200k sharded over the ranks)"
    return {"workload": f"{name}: async_drq_sim, {args.cams}x 128x128x3 camera(s), batch {args.batch} (global){rl}, replay {args.capacity} in HBM, "
                        "critic grad step incl. sampling + DrQ shift", "global_batch": args.batch, "cams": args.cams, "rlpd": bool(args.rlpd),
            "replay_capacity": args.capacity, "parallelism": f"dp{args.gpus}", "precision": args.precision,
            "step_pipeline": ("on: sampler + frozen trunk of step i+1 overlap heads / all-reduce / Adam of step i (agent.pipeline_critic_steps; "
                              "the next batch is drawn one call early, like the reference iterator's queue)" if os.environ.get("SERL_PIPELINE", "1") != "0" else "off"),
            "arithmetic": ("frozen ResNet-10 trunk: 16-bit operands on tcgen05 tensor cores with fp32 accumulation; trainable heads, losses, "
                           "Adam in fp32" if args.precision != "fp32" else "everything fp32 (CUDA cores): the 1e-5 parity build"),
            "l2": "inputs exceed L2: each step gathers fresh random frames from a multi-GB replay"}


# ------------------------------------------------------------------------------------------------
class ClockSampler:
    Q = "timestamp,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        self.p, self.index = None, index

    def start(self):
        try:
            self.p = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "50", "-i", str(self.index)],
                                      stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception:                       # noqa: BLE001
            self.p = None

    def stop(self, t_begin=None, t_end=None):
        import datetime
        if self.p is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.p.terminate()
        try:
            out, _ = self.p.communicate(timeout=5)
        except Exception:                       # noqa: BLE001
            self.p.kill()
            out = ""
        sm, mx, reasons = [], None, set()
        for ln in out.strip().splitlines():
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 8:
                continue
            try:
                ts = datetime.datetime.strptime(f[0], "%Y/%m/%d %H:%M:%S.%f").timestamp()
                if t_begin is not None and not (t_begin - 0.05 <= ts <= t_end + 0.05):
                    continue
                sm.append(float(f[1])); mx = float(f[2])
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons), "samples": len(sm)}


def fill_ring_synthetic(rb, seed):
    """SURVEY.md §8d synthetic replay: random frames, episodes of 100 (1 filler slot in 101), N(0,1) state, U(-1,1) actions."""
    import torch
    g = torch.Generator(device="cuda").manual_seed(seed)
    cap = rb._capacity
    for c in rb.cams:
        fr = rb.frames[c]
        chunk = 4096
        for lo in range(0, cap, chunk):
            hi = min(cap, lo + chunk)
            fr[lo:hi] = torch.randint(0, 256, (hi - lo, *fr.shape[1:]), dtype=torch.uint8, device="cuda", generator=g)
    slots = torch.arange(cap, device="cuda")
    valid = (slots % 101) != 0
    rb.valid.copy_(valid.to(torch.uint8))
    rb._valid_host[:] = valid.cpu().numpy()
    rb.state.copy_(torch.randn(rb.state.shape, device="cuda", generator=g))
    rb.next_state.copy_(torch.randn(rb.state.shape, device="cuda", generator=g))
    rb.actions.copy_(torch.rand(rb.actions.shape, device="cuda", generator=g) * 2 - 1)
    rb.rewards.copy_(torch.rand(cap, device="cuda", generator=g))
    ends = (slots % 101) == 100
    rb.masks.copy_((~ends).float())
    rb.dones.copy_(ends.to(torch.uint8))
    rb._size, rb._insert_index, rb._first = cap, 0, False
    rb.size_dev.fill_(cap)


class Workload:
    """Replay rings + agent + batch source of one configuration on the current device."""

    def __init__(self, args, cams_n, rlpd, capacity, batch, rank=0, world=1, seed_base=1000):
        import torch
        from helpers import fake_env, random_transitions
        from serl_b200.utils.launcher import make_drq_agent, make_replay_buffer
        from serl_b200.utils.train_utils import concat_batches
        self.torch = torch
        cams = tuple(f"cam{i}" for i in range(cams_n))
        env = fake_env(cams)
        self.cams, self.B, self.rlpd = cams, batch // world, rlpd
        self.rb = make_replay_buffer(env, capacity=capacity // world, type="memory_efficient_replay_buffer", image_keys=list(cams),
                                     seed=seed_base + rank)           # rank folded into the sampler stream
        fill_ring_synthetic(self.rb, seed=rank)
        rng = np.random.default_rng(0)
        self.transitions = random_transitions(rng, 8, cams, mean_ep=1000)
        self.agent = make_drq_agent(42, self.transitions[0]["observations"], self.transitions[0]["actions"], image_keys=cams,
                                    encoder_type="resnet-pretrained", precision=args.precision)
        self.agent.data_parallel = world > 1
        # cross-step pipeline (serl_b200/agents/continuous/drq.py): sampler + frozen trunk of step i+1 next to heads + Adam of step i
        self.agent.pipeline_critic_steps = os.environ.get("SERL_PIPELINE", "1") != "0"
        if rlpd:                                                       # async_drq_sim.py:275-277: batch_size // 2 from each buffer
            half = self.B // 2
            self.demo = make_replay_buffer(env, capacity=20 * 101, type="memory_efficient_replay_buffer", image_keys=list(cams),
                                           seed=seed_base + 500 + rank)
            fill_ring_synthetic(self.demo, seed=100 + rank)
            it = self.rb.get_iterator(sample_args={"batch_size": half, "pack_obs_and_next_obs": True})
            dit = self.demo.get_iterator(sample_args={"batch_size": self.B - half, "pack_obs_and_next_obs": True})
            self.next_batch = lambda: concat_batches(next(it), next(dit), axis=0)
        else:
            self.demo = None
            it = self.rb.get_iterator(sample_args={"batch_size": self.B, "pack_obs_and_next_obs": True})
            self.next_batch = lambda: next(it)

    def timed_steps(self, steps, barrier=None):
        """`steps` critic steps, CUDA-event timed on the launching stream, a synchronize (and barrier) on both sides."""
        torch = self.torch
        sync = barrier or torch.cuda.synchronize
        t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        sync()
        t0.record()
        for _ in range(steps):
            out = self.agent.update_critics(self.next_batch())
        t1.record()
        sync()
        self.last_info = out[1]
        return t0.elapsed_time(t1)

    def dump_outputs(self, path, moment_sample=1 << 20):
        """What the last timed step handed back: its info scalars and the updated agent state (trainable parameters and target
        parameters in full; the Adam moments as a fixed, seeded sample of `moment_sample` entries to stay well under 64 MB).
        Two runs with the same arguments draw the same batches and keys, but atomic accumulations (GroupNorm statistics, split-K
        reductions) round in a varying order, so their float outputs agree to a tolerance, not bit for bit."""
        torch = self.torch
        st = self.agent._store
        out = dict(self.last_info["critic"])                                     # critic_loss, predicted_qs, target_qs
        out.update({k: self.last_info[k] for k in ("critic_lr", "actor_lr", "temperature_lr")})
        out.update(params=st.params[:st.n_main], target_params=st.target[:st.n_main])
        idx = np.sort(np.random.default_rng(0).choice(st.n, min(moment_sample, st.n), replace=False))
        idx = torch.as_tensor(idx, device=st.m.device)
        out.update(adam_mu_sample=st.m[idx], adam_nu_sample=st.v[idx])
        os.makedirs(path, exist_ok=True)
        for name, v in out.items():
            np.save(os.path.join(path, f"{name}.npy"), v.detach().float().cpu().numpy())
        np.save(os.path.join(path, "rng.npy"), self.agent.state.rng.astype(np.float64))   # uint32 key: exact in float64

    def e2e_steps(self, steps, barrier=None):
        """The public-API loop with HOST buffers: every step inserts one fresh transition from host memory (pinned staging ->
        HBM), draws the batch through the replay iterators, runs agent.update_critics and reads the loss back."""
        torch = self.torch
        sync = barrier or torch.cuda.synchronize
        h0 = self.rb.h2d_bytes
        sync()
        e0 = time.perf_counter()
        for s in range(steps):
            self.rb.insert(self.transitions[s % len(self.transitions)])
            _, info = self.agent.update_critics(self.next_batch())
            loss = float(info["critic"]["critic_loss"])
        sync()
        dt = time.perf_counter() - e0
        assert np.isfinite(loss)
        return dt, (self.rb.h2d_bytes - h0) / steps, 4.0

    def close(self):
        self.agent._graphs.clear()
        self.torch.cuda.synchronize()


def measure_single_camera(args):
    """Supplementary measurement on BASELINE configs[1]: single camera, whole batch from one 100k ring."""
    steps = args.steps
    w = Workload(args, 1, False, 100_000, args.batch)
    for _ in range(11):
        w.agent.update_critics(w.next_batch())
    ms = w.timed_steps(steps) / steps
    dt, h2d, d2h = w.e2e_steps(steps)
    out = {"workload": f"BASELINE configs[1]: async_drq_sim, 1x 128x128x3 camera, batch {args.batch}, replay 100000 in HBM, critic grad step incl. sampling + DrQ shift",
           "value": 1e3 / ms, "unit": "steps/s", "ms_per_step": ms, "steps": steps,
           "e2e": {"value": steps / dt, "unit": "steps/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h}}
    w.close()
    del w
    return out


def run_b200(args):
    import torch
    import torch.distributed as dist
    rank, world, local = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1)), int(os.environ.get("LOCAL_RANK", 0))
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    assert args.batch % world == 0 and (not args.rlpd or (args.batch // world) % 2 == 0)
    w = Workload(args, args.cams, args.rlpd, args.capacity, args.batch, rank, world)
    agent, B = w.agent, w.B
    eng = agent._engine(B)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- device-resident throughput (whole step replayed as one CUDA graph): EXACTLY args.steps timed steps -------------
    ev = lambda: torch.cuda.Event(enable_timing=True)
    clocks = ClockSampler(local)
    clocks.start()
    # W warm-up steps; the step has up to four CUDA-graph variants (serial; pipeline start "W"; steady state "P" on either engine of the
    # ping-pong pair), each run eagerly once and captured on its second use: a few more untimed steps so that the timed region only replays
    settle = 6 if agent.pipeline_critic_steps else 0
    for _ in range(max(args.warmup, 3) + settle):
        agent.update_critics(w.next_batch())
    launches0 = agent.kernel_launches
    w0 = time.time()
    ms = w.timed_steps(args.steps, barrier)
    launches = agent.kernel_launches - launches0
    if args.dump_outputs and rank == 0:
        w.dump_outputs(args.dump_outputs)
    # ---- the same loop for >= sustain-s seconds: the sustained figure, and enough nvidia-smi samples under load -----------
    n_sus = max(args.steps, int(args.sustain_s * 1e3 / max(ms / args.steps, 1e-3)) + 1)
    if world > 1:
        t = torch.tensor([n_sus], device="cuda"); dist.all_reduce(t, op=dist.ReduceOp.MAX); n_sus = int(t.item())
    ms_sus = w.timed_steps(n_sus, barrier)
    clk = clocks.stop(w0, time.time())
    agent.check_status()

    # ---- per-section durations: the same steps launched EAGERLY with CUDA events around the sections (one rank's timeline;
    # eager launches add host gaps inside the short sections, so these are upper bounds of what the graph replay spends) ------
    orig_load = agent._load_batch
    agent.use_cuda_graphs = False
    agent.section_events = []
    n_eager = min(args.steps, 20)
    for _ in range(n_eager):
        agent.update_critics(w.next_batch())
    barrier()
    agent.use_cuda_graphs = True
    sec = {}
    for name, a_, b_ in agent.section_events:
        sec[name] = sec.get(name, 0.0) + a_.elapsed_time(b_) / n_eager
    agent.section_events = None
    trunk_ms = sec["trunk"]
    # the sampler kernel(s) of a step are ~10x shorter than a host launch: time them as 20 batch loads captured in one CUDA
    # graph, replayed back to back (each launch draws a fresh batch: the device step counter advances inside the graph)
    handle = w.next_batch()
    reps = 20
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        for _ in range(reps):
            orig_load(eng, handle, augment=True, keys=agent._keys, graph_mode=True)
    g.replay(); torch.cuda.synchronize()
    a, b = ev(), ev()
    a.record()
    for _ in range(5):
        g.replay()
    b.record(); torch.cuda.synchronize()
    samp_ms = a.elapsed_time(b) / (5 * reps)
    del g

    # ---- end to end through the public API with host buffers --------------------------------------------
    e2e_s, h2d, d2h = w.e2e_steps(args.steps, barrier)

    replicas_identical = None
    if world > 1:                                   # data-parallel replicas must stay bit-identical (same reduced gradient everywhere)
        mine = agent._store.params.clone()
        ref = mine.clone()
        dist.broadcast(ref, src=0)
        same = torch.tensor([int(torch.equal(mine, ref))], device="cuda")
        dist.all_reduce(same, op=dist.ReduceOp.MIN)
        replicas_identical = bool(same.item())
    names = sorted(sec)
    tmax = torch.tensor([ms, e2e_s * 1e3, ms_sus, trunk_ms, samp_ms] + [sec[k] for k in names], device="cuda", dtype=torch.float64)
    if world > 1:
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
    ms, e2e_ms, ms_sus, trunk_ms, samp_ms = tmax.tolist()[:5]
    sec = {k: v for k, v in zip(names, tmax.tolist()[5:])}

    def shutdown():
        # captured NCCL kernels inside live CUDA graphs can block process-group teardown: drop the graphs first, and never
        # let a teardown problem turn into a hung bench (os._exit after the line is out)
        agent._graphs.clear()
        torch.cuda.synchronize()
        sys.stdout.flush()
        if world > 1:
            os._exit(0)

    if rank != 0:
        shutdown()
        return
    pk = peaks()
    value = args.steps / (ms / 1e3)
    images = 2 * B * args.cams                                    # per rank per step (obs + next_obs, trunk shared)
    trunk_tflops = images * TRUNK_GFLOP_PER_IMAGE / 1e3 / (trunk_ms / 1e3)
    samp_bytes = 2 * B * args.cams * 2 * FRAME_BYTES              # read 2 frames + write 2 crops per sample per camera
    samp_gbs = samp_bytes / 1e9 / (samp_ms / 1e3)
    line = {"metric": "drq_critic_grad_steps_per_sec", "value": value, "unit": "steps/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": {"fp32": "f32", "bf16": "bf16", "fp16": "f16"}[args.precision], "data": "synthetic", "impl": "b200",
            "config": workload_config(args),
            "clocks": clk,
            "e2e": {"value": args.steps / (e2e_ms / 1e3), "unit": "steps/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h},
            "sustained": {"value": n_sus / (ms_sus / 1e3), "unit": "steps/s", "steps": n_sus, "seconds": ms_sus / 1e3,
                          "note": "same loop, run for >= --sustain-s seconds right after the K timed steps; the clock samples cover both"},
            "gpu_launches": launches, "cuda_graph": True, "replicas_identical": replicas_identical, "untimed_graph_settle_steps": settle,
            "sections_ms": {**{k: round(v, 4) for k, v in sec.items()},
                            "note": "eagerly launched steps, CUDA events per section, mean over steps, max over ranks; heads = encoder heads + critic / policy MLPs + losses + backward"},
            "roofline": {"kernel": TRUNK_KERNELS[args.precision != "fp32"], "bound": "tensor",
                         "achieved": trunk_tflops, "peak": pk["tensor"], "unit": "TFLOP/s", "frac": trunk_tflops / pk["tensor"],
                         "traffic": trunk_traffic(args), "traffic_source": "profiles/trunk_traffic.json, regenerated from the committed ncu launch list by scripts/trunk_traffic.py",
                         "peak_source": pk["src"], "ms_per_step": trunk_ms,
                         "timing": "CUDA events around the trunk section of eagerly launched steps (the headline loop replays a CUDA graph), max over ranks",
                         "algorithmic": f"{images} images x {TRUNK_GFLOP_PER_IMAGE} GFLOP per rank"},
            "sampler": {"kernel": "sample_frames_kernel", "timing": "20 batch loads captured in one CUDA graph, replayed 5x, CUDA events", "bound": "hbm", "achieved": samp_gbs, "peak": pk["hbm"], "unit": "GB/s",
                        "frac": samp_gbs / pk["hbm"], "ms_per_step": samp_ms, "algorithmic_bytes": samp_bytes, "launches_per_step": 2 if args.rlpd else 1}}
    w.close()
    if world == 1 and not os.environ.get("SERL_BENCH_SKIP_SINGLE") and (args.cams != 1 or args.rlpd):
        del w, eng
        try:
            line["single_camera"] = measure_single_camera(args)
        except Exception as e:                  # noqa: BLE001
            line["single_camera"] = {"value": None, "error": str(e)}
    try:
        if os.environ.get("SERL_BENCH_SKIP_CPU"):
            raise RuntimeError("skipped (SERL_BENCH_SKIP_CPU)")
        rows = 64
        v, t, cores, done = cpu_reference_steps(args, 2, 1, rows, budget_s=30.0)
        line["cpu_baseline"] = {"value": v, "unit": "steps/s", "cores": cores, "kind": "port", "extrapolated_x": args.batch / rows,
                                "sample": f"{done} timed step(s) of {rows}/{args.batch} rows, ~30 s budget: oracle torch-CPU fp32 restatement of sample + update_critics with the "
                                          f"reference's three frozen-encoder passes (jax not installable); steps/s EXTRAPOLATED x{args.batch / rows:g} by rows/batch"}
    except Exception as e:                      # noqa: BLE001
        line["cpu_baseline"] = {"value": None, "unit": "steps/s", "cores": os.cpu_count(), "kind": "port", "sample": f"failed: {e}"}
    print(json.dumps(line), flush=True)
    shutdown()


if __name__ == "__main__":
    a = parse()
    if a.impl == "reference":
        run_reference(a)
    else:
        run_b200(a)
