"""Reward-classifier benchmark (serl_b200/networks/reward_classifier.py): prints ONE JSON line.

    python scripts/bench_classifier.py [--steps 200] [--warmup 20] [--batch 256] [--capacity 10000]

  * training steps/s and ms/step at batch 256 (128 positive + 128 negative rows) from two 10 k-slot rings of synthetic
    transitions (the example's capacity=10000), for 1 and 2 cameras, fp16 and fp32: lazy batches, CUDA-graph replay;
  * kernel launches per step (the library's serl_launch_count over one eager step);
  * the frozen trunk's achieved FLOP/s: FLOPs from the layer shapes over CUDA-event time of the trunk alone (B images per camera);
  * median / p90 latency of one unbatched func(obs) call of load_classifier_func, host observation -> host logit;
  * the GPU name and power limit, read in the same process.
Every shape is warmed up before it is timed.  Writes nothing to the tree (checkpoints go to a temporary directory).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


class _Box:
    def __init__(self, shape, dtype=np.float32):
        self.shape, self.dtype = tuple(shape), np.dtype(dtype)


class _Dict:
    def __init__(self, spaces):
        self.spaces = dict(spaces)


def _env(cams, hw=128, S=7, A=4):
    """The observation / action spaces make_replay_buffer reads: one (1, hw, hw, 3) frame per camera, a (1, S) state, A actions."""
    obs = _Dict({**{c: _Box((1, hw, hw, 3), np.uint8) for c in cams}, "state": _Box((1, S))})
    return type("Env", (), {"observation_space": obs, "action_space": _Box((A,))})()


def trunk_flop_per_image(hw=128):
    """2 x multiply-adds of ResNet-10's convolutions (vision/resnet_v1.py:217-286) at an hw x hw input."""
    s = hw // 2
    mac = s * s * 64 * 7 * 7 * 3                                 # conv_init 7x7/2
    s //= 2                                                      # max-pool 3x3/2
    cin = 64
    for f, stride in ((64, 1), (128, 2), (256, 2), (512, 2)):
        so = s // stride
        mac += so * so * f * 9 * cin + so * so * f * 9 * f
        if stride != 1 or cin != f:
            mac += so * so * f * cin
        s, cin = so, f
    return 2.0 * mac


def gpu_info():
    import torch
    name = torch.cuda.get_device_name(0)
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader,nounits", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip().split(",")
        return {"name": name, "power_limit_w": float(out[0]), "sm_max_mhz": float(out[1])}
    except Exception as e:                                       # noqa: BLE001
        return {"name": name, "power_limit_w": None, "note": f"nvidia-smi unavailable: {e}"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--batch", type=int, default=256)
    ap.add_argument("--capacity", type=int, default=10000)
    ap.add_argument("--latency-calls", type=int, default=200)
    args = ap.parse_args()
    import torch
    from bench import fill_ring_synthetic
    from oracle import jax_prng as P
    from serl_b200 import _lib as L
    from serl_b200.networks.reward_classifier import create_classifier, load_classifier_func, sample_classifier_batch, train_step
    from serl_b200.utils.checkpoints import save_checkpoint
    from serl_b200.utils.launcher import make_replay_buffer
    assert torch.cuda.is_available(), "bench_classifier needs a GPU"
    torch.cuda.set_device(0)
    res = {"gpu": gpu_info(), "batch": args.batch, "capacity": args.capacity, "train": {}, "trunk": {}, "inference_latency_ms": {}}
    B = args.batch
    fpi = trunk_flop_per_image()
    for ncam in (1, 2):
        cams = tuple(f"cam{i}" for i in range(ncam))
        rings = []
        for k in range(2):
            rb = make_replay_buffer(_env(cams), capacity=args.capacity, type="memory_efficient_replay_buffer", image_keys=list(cams), seed=k)
            fill_ring_synthetic(rb, 100 + k)
            rings.append(rb)
        sample = {c: np.zeros((1, 1, 128, 128, 3), np.uint8) for c in cams}
        for precision in ("fp16", "fp32"):
            tag = f"{precision}_{ncam}cam"
            st = create_classifier(np.array([0, 1], np.uint32), sample, cams, pretrained_encoder_path=None, precision=precision)
            rng = P.prng_key(0)
            keys = []
            for _ in range(args.warmup + args.steps):
                rng, a = P.split(rng)
                rng, d = P.split(rng)
                keys.append((a, d))
            st.use_cuda_graphs = False                           # one eager step: the launches a step enqueues
            c0 = L.launch_count()
            train_step(st, sample_classifier_batch(rings[0], rings[1], B, keys[0][0]), keys[0][1])
            torch.cuda.synchronize()
            launches = L.launch_count() - c0
            st.use_cuda_graphs = True
            for a, d in keys[1:args.warmup]:
                train_step(st, sample_classifier_batch(rings[0], rings[1], B, a), d)
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for a, d in keys[args.warmup:]:
                st, loss, acc = train_step(st, sample_classifier_batch(rings[0], rings[1], B, a), d)
            e1.record()
            torch.cuda.synchronize()
            ms = e0.elapsed_time(e1) / args.steps
            st.check_status()
            res["train"][tag] = {"steps_per_s": round(1000.0 / ms, 1), "ms_per_step": round(ms, 4), "launches_per_step": launches,
                                 "loss_last": round(float(loss), 5), "accuracy_last": round(float(acc), 4)}
            # the trunk alone, B images per camera (what a step runs), eager launches timed by events
            b = st._bufs[B]
            for _ in range(3):
                st._trunk_forward(b)
            reps = 20
            e0.record()
            for _ in range(reps):
                st._trunk_forward(b)
            e1.record()
            torch.cuda.synchronize()
            tms = e0.elapsed_time(e1) / reps
            res["trunk"][tag] = {"images": B * ncam, "ms": round(tms, 4), "tflop_per_s": round(fpi * B * ncam / (tms * 1e-3) / 1e12, 1)}
            # unbatched inference: save, load, func(obs) host -> host
            with tempfile.TemporaryDirectory() as tmp:
                save_checkpoint(tmp, st, step=st.step)
                func = load_classifier_func(np.array([0, 1], np.uint32), sample, cams, tmp, precision=precision)
            gen = np.random.default_rng(0)
            obs = {**{c: gen.integers(0, 256, (1, 128, 128, 3), dtype=np.uint8) for c in cams}, "state": np.zeros((1, 7), np.float32)}
            for _ in range(20):
                func(obs)
            lat = []
            for _ in range(args.latency_calls):
                t0 = time.perf_counter()
                out = func(obs)
                lat.append((time.perf_counter() - t0) * 1e3)
            assert out.shape == (1,)
            res["inference_latency_ms"][tag] = {"median": round(float(np.median(lat)), 4), "p90": round(float(np.percentile(lat, 90)), 4)}
            del st, func
            torch.cuda.empty_cache()
        del rings
        torch.cuda.empty_cache()
    res["trunk_flop_per_image"] = fpi
    print(json.dumps(res))


if __name__ == "__main__":
    main()
