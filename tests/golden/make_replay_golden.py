"""Generate golden fixtures for the replay ring by running the REAL reference classes.

Needs a checkout of the reference repository (rail-berkeley/serl).  jax / flax / gym need not
be installed: the reference's replay code only *imports* them and uses
`gym.spaces.{Box,Dict}` as shape carriers, `gym.utils.seeding.np_random` for an RNG and
`flax.core.frozen_dict.freeze/unfreeze` as a dict wrapper - so minimal import stubs (below,
written for this script) are enough to execute the reference's own, unmodified
`MemoryEfficientReplayBuffer.insert` / `.sample` (data/memory_efficient_replay_buffer.py:53-164).

The reference's index stream is unseeded; we replace its `np_random` by a scripted stream
object so the reference consumes a known sequence (including its redraw-on-invalid loop).

Output: tests/golden/replay_<case>.npz  (inputs + the reference's slot contents + sampled batches).
Usage:  python tests/golden/make_replay_golden.py <reference checkout>
"""
from __future__ import annotations

import os
import sys
import types

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))


# ------------------------------------------------------------------------------------------
# import stubs (ours) for jax / flax / gym
# ------------------------------------------------------------------------------------------
def _install_stubs():
    jax = types.ModuleType("jax")
    jax.numpy = types.ModuleType("jax.numpy")
    jax.jit = lambda f=None, **kw: (f if f is not None else (lambda g: g))
    jax.device_put = lambda x, device=None: x
    sys.modules["jax"] = jax
    sys.modules["jax.numpy"] = jax.numpy

    class FrozenDict(dict):
        def unfreeze(self):
            return {k: (v.unfreeze() if isinstance(v, FrozenDict) else v) for k, v in self.items()}

    def freeze(d):
        return FrozenDict({k: (freeze(v) if isinstance(v, dict) else v) for k, v in d.items()})

    flax = types.ModuleType("flax")
    flax.core = types.ModuleType("flax.core")
    fd = types.ModuleType("flax.core.frozen_dict")
    fd.FrozenDict, fd.freeze = FrozenDict, freeze
    flax.core.frozen_dict = fd
    sys.modules.update({"flax": flax, "flax.core": flax.core, "flax.core.frozen_dict": fd})

    gym = types.ModuleType("gym")

    class Space:
        pass

    class Box(Space):
        def __init__(self, low, high, shape=None, dtype=np.float32):
            low = np.asarray(low)
            high = np.asarray(high)
            if shape is None:
                shape = low.shape
            self.low = np.broadcast_to(low, shape).astype(dtype)
            self.high = np.broadcast_to(high, shape).astype(dtype)
            self.shape = tuple(shape)
            self.dtype = np.dtype(dtype)

    class Dict(Space):
        def __init__(self, spaces):
            self.spaces = dict(spaces)

    gym.Space = Space
    gym.spaces = types.ModuleType("gym.spaces")
    gym.spaces.Box, gym.spaces.Dict, gym.spaces.Space = Box, Dict, Space
    gym.utils = types.ModuleType("gym.utils")
    gym.utils.seeding = types.ModuleType("gym.utils.seeding")
    gym.utils.seeding.np_random = lambda seed=None: (np.random.default_rng(seed), seed)
    sys.modules.update({"gym": gym, "gym.spaces": gym.spaces, "gym.utils": gym.utils,
                        "gym.utils.seeding": gym.utils.seeding})
    return gym


class ScriptedStream:
    """Stands in for numpy's Generator: hands out a pre-recorded index stream."""

    def __init__(self, stream):
        self.stream = list(stream)
        self.pos = 0

    def integers(self, n, size=None):
        if size is None:
            v = self.stream[self.pos] % n
            self.pos += 1
            return v
        out = np.array([self.stream[self.pos + i] % n for i in range(size)], dtype=np.int64)
        self.pos += size
        return out


def make_case(name, *, cap, T, ncam, H, W, S, A, n_insert, mean_ep, seed, n_batches, B):
    gym = _GYM
    from serl_launcher.data.memory_efficient_replay_buffer import MemoryEfficientReplayBuffer

    cams = [f"cam{i}" for i in range(ncam)]
    obs_space = gym.spaces.Dict({
        **{c: gym.spaces.Box(0, 255, shape=(T, H, W, 3), dtype=np.uint8) for c in cams},
        "state": gym.spaces.Box(-np.inf, np.inf, shape=(T, S), dtype=np.float32),
    })
    act_space = gym.spaces.Box(-1, 1, shape=(A,), dtype=np.float32)
    buf = MemoryEfficientReplayBuffer(obs_space, act_space, cap, pixel_keys=tuple(cams))

    rng = np.random.default_rng(seed)
    # transitions: consecutive observations of an episode share frames (next_obs of t == obs of t+1)
    ins = dict(frames={c: [] for c in cams}, nframes={c: [] for c in cams}, state=[], nstate=[],
               actions=[], rewards=[], masks=[], dones=[])
    cur = None
    snapshots_at = {n_insert // 3, (2 * n_insert) // 3, n_insert - 1}
    snaps = {}
    sample_out = {}
    for i in range(n_insert):
        if cur is None:
            cur = {c: rng.integers(0, 256, (T, H, W, 3), dtype=np.uint8) for c in cams}
            cur["state"] = rng.standard_normal((T, S)).astype(np.float32)
        nxt = {c: np.concatenate([cur[c][1:], rng.integers(0, 256, (1, H, W, 3), dtype=np.uint8)]) for c in cams}
        nxt["state"] = rng.standard_normal((T, S)).astype(np.float32)
        done = bool(rng.random() < 1.0 / mean_ep)
        tr = dict(observations={k: v.copy() for k, v in cur.items()},
                  next_observations={k: v.copy() for k, v in nxt.items()},
                  actions=rng.uniform(-1, 1, A).astype(np.float32),
                  rewards=np.float32(rng.random()), masks=np.float32(0.0 if (done and rng.random() < 0.5) else 1.0),
                  dones=done)
        for c in cams:
            ins["frames"][c].append(cur[c])
            ins["nframes"][c].append(nxt[c])
        ins["state"].append(cur["state"]); ins["nstate"].append(nxt["state"])
        ins["actions"].append(tr["actions"]); ins["rewards"].append(tr["rewards"])
        ins["masks"].append(tr["masks"]); ins["dones"].append(done)
        buf.insert(tr)
        cur = None if done else nxt
        if i in snapshots_at:
            tag = f"snap{len(snaps)}"
            dd = buf.dataset_dict
            snap = {"n_inserted": i + 1, "size": len(buf), "cursor": buf._insert_index,
                    "valid": buf._is_correct_index.copy(), "state": dd["observations"]["state"].copy(),
                    "next_state": dd["next_observations"]["state"].copy(), "actions": dd["actions"].copy(),
                    "rewards": dd["rewards"].copy(), "masks": dd["masks"].copy(), "dones": dd["dones"].copy()}
            for c in cams:
                snap[f"frames_{c}"] = dd["observations"][c].copy()
            snaps[tag] = snap
            # scripted sampling through the reference's own sample() (incl. its redraw loop)
            stream = rng.integers(0, 2**31, size=n_batches * B * 8)
            buf._np_random = ScriptedStream(stream)
            for b in range(n_batches):
                pos0 = buf._np_random.pos
                batch = buf.sample(B, pack_obs_and_next_obs=True).unfreeze()
                so = {"pos0": pos0, "pos1": buf._np_random.pos, "state": batch["observations"]["state"],
                      "next_state": batch["next_observations"]["state"], "actions": batch["actions"],
                      "rewards": batch["rewards"], "masks": batch["masks"], "dones": batch["dones"]}
                for c in cams:
                    so[f"pix_{c}"] = batch["observations"][c]
                assert all(c not in batch["next_observations"] for c in cams)
                sample_out[f"{tag}_b{b}"] = so
            snaps[tag]["stream"] = stream

    flat = {"meta": np.array([cap, T, ncam, H, W, S, A, n_insert, B, n_batches], dtype=np.int64)}
    for c in cams:
        flat[f"in_frames_{c}"] = np.stack(ins["frames"][c])
        flat[f"in_nframes_{c}"] = np.stack(ins["nframes"][c])
    for k in ("state", "nstate", "actions", "rewards", "masks", "dones"):
        flat[f"in_{k}"] = np.stack(ins[k])
    for tag, snap in snaps.items():
        for k, v in snap.items():
            flat[f"{tag}/{k}"] = np.asarray(v)
    for tag, so in sample_out.items():
        for k, v in so.items():
            flat[f"{tag}/{k}"] = np.asarray(v)
    path = os.path.join(HERE, f"replay_{name}.npz")
    np.savez_compressed(path, **flat)
    print("wrote", path, os.path.getsize(path), "bytes")


def make_wrap_first_case(name="wrap_first", *, cap=10, T=1, H=3, W=2, S=2, A=2, first_ep=8, second_ep=3):
    """A valid slot idx < T: an episode that ends on slot cap-2 puts the next episode's filler frame on slot cap-1 and its first
    transition on slot 0.  The reference gathers obs_pixels[indx - T] from a sliding-window view, so idx = 0 reads window -1 =
    slots cap-2, cap-1 (numpy negative index), not the ring-wrapped pair (memory_efficient_replay_buffer.py:148-151)."""
    gym = _GYM
    from serl_launcher.data.memory_efficient_replay_buffer import MemoryEfficientReplayBuffer
    obs_space = gym.spaces.Dict({"cam0": gym.spaces.Box(0, 255, shape=(T, H, W, 3), dtype=np.uint8),
                                 "state": gym.spaces.Box(-np.inf, np.inf, shape=(T, S), dtype=np.float32)})
    buf = MemoryEfficientReplayBuffer(obs_space, gym.spaces.Box(-1, 1, shape=(A,), dtype=np.float32), cap, pixel_keys=("cam0",))
    rng = np.random.default_rng(7)
    ins = dict(frames=[], nframes=[], state=[], nstate=[], actions=[], rewards=[], masks=[], dones=[])
    for n in (first_ep, second_ep):
        cur = {"cam0": rng.integers(0, 256, (T, H, W, 3), dtype=np.uint8), "state": rng.standard_normal((T, S)).astype(np.float32)}
        for i in range(n):
            nxt = {"cam0": np.concatenate([cur["cam0"][1:], rng.integers(0, 256, (1, H, W, 3), dtype=np.uint8)]),
                   "state": rng.standard_normal((T, S)).astype(np.float32)}
            tr = dict(observations={k: v.copy() for k, v in cur.items()}, next_observations={k: v.copy() for k, v in nxt.items()},
                      actions=rng.uniform(-1, 1, A).astype(np.float32), rewards=np.float32(rng.random()), masks=np.float32(1.0), dones=bool(i == n - 1))
            ins["frames"].append(cur["cam0"]); ins["nframes"].append(nxt["cam0"]); ins["state"].append(cur["state"]); ins["nstate"].append(nxt["state"])
            ins["actions"].append(tr["actions"]); ins["rewards"].append(tr["rewards"]); ins["masks"].append(tr["masks"]); ins["dones"].append(tr["dones"])
            buf.insert(tr)
            cur = nxt
    assert buf._is_correct_index[0], "the case must make slot 0 valid"
    stream = [0, 1, 2, cap - 2, 0]
    buf._np_random = ScriptedStream(stream)
    batch = buf.sample(len(stream), pack_obs_and_next_obs=True).unfreeze()
    dd = buf.dataset_dict
    flat = {"meta": np.array([cap, T, 1, H, W, S, A, first_ep + second_ep, len(stream), 1], dtype=np.int64), "stream": np.array(stream),
            "valid": buf._is_correct_index.copy(), "size": np.int64(len(buf)), "cursor": np.int64(buf._insert_index),
            "frames_cam0": dd["observations"]["cam0"].copy(), "pix_cam0": batch["observations"]["cam0"],
            "state": batch["observations"]["state"], "next_state": batch["next_observations"]["state"], "actions": batch["actions"]}
    for k in ("state", "nstate", "actions", "rewards", "masks", "dones"):
        flat[f"in_{k}"] = np.stack(ins[k])
    flat["in_frames_cam0"], flat["in_nframes_cam0"] = np.stack(ins["frames"]), np.stack(ins["nframes"])
    path = os.path.join(HERE, f"replay_{name}.npz")
    np.savez_compressed(path, **flat)
    print("wrote", path, os.path.getsize(path), "bytes")


if __name__ == "__main__":
    if len(sys.argv) != 2:
        sys.exit("usage: python tests/golden/make_replay_golden.py <reference checkout>")
    _GYM = _install_stubs()
    sys.path.insert(0, os.path.join(os.path.abspath(sys.argv[1]), "serl_launcher"))
    # T=1 single cam with several wrap-arounds; T=2 dual-cam; tiny cap stress
    make_case("t1_cam1", cap=37, T=1, ncam=1, H=6, W=5, S=3, A=2, n_insert=150, mean_ep=7, seed=1, n_batches=2, B=16)
    make_case("t2_cam2", cap=53, T=2, ncam=2, H=4, W=4, S=2, A=3, n_insert=230, mean_ep=9, seed=2, n_batches=2, B=16)
    make_case("t1_cam2_long", cap=64, T=1, ncam=2, H=4, W=6, S=7, A=4, n_insert=400, mean_ep=25, seed=3, n_batches=2, B=32)
    make_wrap_first_case()
