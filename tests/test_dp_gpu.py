"""GPU, world_size 2, NCCL (needs 2 GPUs; skipped on a single-GPU machine): the hardware data-parallel
parity test of SURVEY.md App. E - the mean of the shard gradients (ONE all-reduce of the 1/world-scaled flat gradient
segment, semantics of jax.lax.pmean(grads_and_aux), reference common/common.py:213-214) equals the single-GPU gradient on
the concatenated batch, the averaged infos equal the full-batch infos, and after Adam both replicas hold bit-identical
parameters that match the single-GPU step.  Explicit randomness (crop offsets, eps, dropout masks, subsample indices) so that
row i of the concatenated batch sees the same noise on either path."""
import os
import sys

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _rows(x, lo, hi):
    return {k: _rows(v, lo, hi) for k, v in x.items()} if isinstance(x, dict) else x[lo:hi]


def _worker(rank, world, port, out):
    sys.path.insert(0, ROOT)
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import torch.distributed as dist
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    from helpers import random_transitions
    from serl_b200.utils.launcher import make_drq_agent
    cams, B, A = ("front", "wrist"), 16, 4
    rng = np.random.default_rng(0)
    tr = random_transitions(rng, 1, cams)[0]
    batch = {"observations": {**{c: rng.integers(0, 256, (B, 2, 128, 128, 3), dtype=np.uint8) for c in cams},
                              "state": rng.standard_normal((B, 1, 7)).astype(np.float32)},
             "next_observations": {"state": rng.standard_normal((B, 1, 7)).astype(np.float32)},
             "actions": rng.uniform(-1, 1, (B, A)).astype(np.float32), "rewards": rng.random(B).astype(np.float32),
             "masks": (rng.random(B) > 0.2).astype(np.float32), "dones": np.zeros(B, bool)}
    expl = {"crop": (rng.integers(0, 9, (B, 2)).astype(np.int32), rng.integers(0, 9, (B, 2)).astype(np.int32)),
            "critic": {"eps": rng.standard_normal((B, A)).astype(np.float32),
                       "dropout": {c: (rng.random((B, 4096)) < 0.9) for c in cams}, "subsample": np.array([3, 7], np.int32)}}

    def make():
        agent = make_drq_agent(42, tr["observations"], tr["actions"], image_keys=cams, encoder_type="resnet-pretrained")
        g = torch.Generator(device="cuda").manual_seed(1)
        st = agent._store
        st.params.add_(torch.randn(st.n, device="cuda", generator=g) * 0.05)
        st.target.copy_(st.params)
        st.version += 1
        return agent

    def expl_rows(lo, hi):
        t = lambda x: torch.as_tensor(x[lo:hi]).cuda()
        return {"crop": (expl["crop"][0][lo:hi], expl["crop"][1][lo:hi]),
                "critic": {"eps": t(expl["critic"]["eps"]), "dropout": {c: t(v).to(torch.uint8) for c, v in expl["critic"]["dropout"].items()},
                           "subsample": torch.as_tensor(expl["critic"]["subsample"]).cuda()}}

    h = B // world
    dp = make()
    dp.data_parallel = True
    dp.explicit_randomness = expl_rows(rank * h, (rank + 1) * h)
    _, info = dp.update_critics(_rows(batch, rank * h, (rank + 1) * h))
    st = dp._store
    res = {"grad": st.grad[:st.info_off].cpu(), "params": st.params[:st.n_main].cpu(),
           "info": {k: float(v) for k, v in info["critic"].items()}}
    if rank == 0:
        one = make()
        one.explicit_randomness = expl_rows(0, B)
        _, info1 = one.update_critics(batch)
        s1 = one._store
        res.update(grad1=s1.grad[:s1.info_off].cpu(), params1=s1.params[:s1.n_main].cpu(),
                   info1={k: float(v) for k, v in info1["critic"].items()},
                   leaves=[(l.path, l.offset, l.size) for l in s1.spec if l.group == 0])
    torch.save(res, out.format(rank))
    dist.barrier()
    dist.destroy_process_group()


def test_reduced_shard_gradient_equals_full_batch_gradient(tmp_path):
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    import torch.multiprocessing as mp
    world, port = 2, 29500 + os.getpid() % 400
    out = str(tmp_path / "rank{}.pt")
    mp.spawn(_worker, args=(world, port, out), nprocs=world, join=True)
    r0, r1 = torch.load(out.format(0)), torch.load(out.format(1))
    assert torch.equal(r0["grad"], r1["grad"]) and torch.equal(r0["params"], r1["params"])        # replicas bit-identical
    worst = 0.0
    for path, off, size in r0["leaves"]:
        g, g1 = r0["grad"][off:off + size].double(), r0["grad1"][off:off + size].double()
        scale = float(g1.abs().max())
        assert scale > 0, path
        err = float((g - g1).abs().max()) / scale
        worst = max(worst, err)
        assert err < 2e-5, (path, err)                   # fp32 sums in a different order: 16 rows at once vs 2 x 8 rows + all-reduce
    for k, v in r0["info1"].items():
        assert abs(r0["info"][k] - v) <= 2e-6 * max(abs(v), 1.0), (k, r0["info"][k], v)
        assert r0["info"][k] == r1["info"][k]
    print(f"worst relative gradient error mean-of-shards vs full batch: {worst:.2e}")
    lr = 3e-4
    dp_, one = r0["params"].double(), r0["params1"].double()
    # Adam normalises by |g|: entries whose gradient is at fp32 noise level may move by a different sign*lr; the rest must agree
    assert float(((dp_ - one).abs() > 2.2 * lr).sum()) == 0
    assert float(((dp_ - one).abs() > 1e-2 * lr).float().mean()) < 0.02
