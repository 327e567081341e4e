"""GPU: the reward classifier (serl_b200/networks/reward_classifier.py) against the CPU restatement (oracle/classifier.py):
one train_step on a host batch (fp32 1e-5 class bars, fp16 1e-2), keyed dropout masks, the lazy device batch (one-sided sampler
crops, graph replay == eager), the one-sided sampler itself, and load_classifier_func after a checkpoint round trip."""
import numpy as np
import pytest
import torch

from helpers import fake_env, random_transitions

pytestmark = pytest.mark.gpu
KEY = np.array([0, 7], np.uint32)


def _flat(tree, prefix=""):
    out = {}
    for k, v in tree.items():
        p = f"{prefix}/{k}" if prefix else k
        out.update(_flat(v, p)) if isinstance(v, dict) else out.__setitem__(p, v)
    return out


def _state(cams, precision="fp32", perturb=True):
    from serl_b200.networks.reward_classifier import create_classifier
    sample = {c: np.zeros((2, 1, 128, 128, 3), np.uint8) for c in cams}
    st = create_classifier(KEY, sample, cams, pretrained_encoder_path=None, precision=precision)
    if perturb:                                                      # biases / scales off their init so every path is exercised
        g = torch.Generator(device="cuda").manual_seed(1)
        st._params.add_(torch.randn(st._n, device="cuda", generator=g) * 0.05)
    return st


def _params64(st):
    return {k: torch.as_tensor(np.asarray(v)).double() for k, v in _flat(st.params).items()}


def _check_step(st, oinfo, grads, newp, tol_out, tol_grad, exact_params):
    B = st._b_last
    b = st._bufs[B]
    logit, logit_e = b["logit"].cpu().double().numpy(), b["logit_e"].cpu().double().numpy()
    rl, re = oinfo["_logits"].numpy().reshape(-1), oinfo["_eval_logits"].numpy().reshape(-1)
    errs = {"logit": np.abs(logit - rl).max(), "eval_logit": np.abs(logit_e - re).max(),
            "loss": abs(float(st._info[0]) - oinfo["loss"])}
    assert errs["logit"] <= tol_out * max(np.abs(rl).max(), 1.0), errs
    assert errs["eval_logit"] <= tol_out * max(np.abs(re).max(), 1.0), errs
    assert errs["loss"] <= tol_out * max(abs(oinfo["loss"]), 1.0), errs
    keep = np.abs(re) > 1e-4
    y = b["labels"].cpu().numpy()
    acc_ref = float((((1 / (1 + np.exp(-re))) >= 0.5) == y)[keep].mean())
    acc_got = float((((1 / (1 + np.exp(-logit_e))) >= 0.5) == y)[keep].mean())
    assert acc_ref == acc_got
    if keep.all():
        assert float(st._info[1]) == pytest.approx(oinfo["accuracy"], abs=1e-7)
    leaf = {}
    for l in st._spec:
        got = st._grad[l.offset:l.offset + l.size].view(l.shape).cpu().numpy()
        ref = grads[l.path].numpy()
        assert np.abs(ref).max() > 0, l.path
        leaf[l.path] = np.abs(got - ref).max() / np.abs(ref).max()
    worst = max(leaf, key=leaf.get)
    errs["grad_rel"], errs["grad_worst_leaf"] = leaf[worst], worst
    errs["grad_median_leaf"] = float(np.median(list(leaf.values())))
    assert tol_grad is None or leaf[worst] <= tol_grad, (worst, leaf[worst], leaf)
    if exact_params:
        now = _flat(st.params)
        lr = st.learning_rate
        for l in st._spec:
            ref, got = newp[l.path].numpy(), np.asarray(now[l.path])
            gmag = np.abs(grads[l.path].numpy())
            noisy = gmag < 2e-2 * max(gmag.max(), 1e-30)
            allow = 1e-5 * max(np.abs(ref).max(), 1e-3) + lr * np.where(noisy, 2.2, 5e-3)
            assert (np.abs(got - ref) <= allow).all(), (l.path, np.abs(got - ref).max())
    return errs


def _host_batch(rng, cams, B):
    # the two classes differ (brighter positives): with indistinguishable noise images the balanced labels make every gradient a
    # near-total cancellation of per-row terms, and its max-normalised error measures that cancellation, not the kernels
    h = B // 2
    data = {c: np.concatenate([rng.integers(96, 256, (h, 1, 128, 128, 3)), rng.integers(0, 160, (B - h, 1, 128, 128, 3))]).astype(np.uint8)
            for c in cams}
    labels = np.concatenate([np.ones((B // 2, 1)), np.zeros((B - B // 2, 1))]).astype(np.float32)
    return {"data": data, "labels": labels}


def _one_host_step(cams, precision, tol_out, tol_grad):
    from oracle import classifier as OC
    from serl_b200.networks.reward_classifier import train_step
    rng = np.random.default_rng(3)
    B = 12
    st = _state(cams, precision)
    batch = _host_batch(rng, cams, B)
    masks = ({c: rng.random((B, 4096)) < 0.9 for c in cams}, rng.random((B, 256)) < 0.9)
    st.explicit_dropout = masks
    p0 = _params64(st)
    st, loss, acc = train_step(st, batch, KEY)
    st._b_last = B
    newp, opt, oinfo, grads = OC.train_step(p0, OC.new_opt(p0), cams, batch["data"], batch["labels"], masks=masks)
    if precision == "fp32":
        errs = _check_step(st, oinfo, grads, newp, tol_out, tol_grad, True)
    else:
        # 16-bit build.  The hidden layer's ReLU derivative is a branch: where its input lies within rounding of 0, TF32 / fp16 rounding
        # can take the other branch than the fp64 oracle, and with a batch of 12 one flipped entry moves a batch-summed leaf (Dense_0/bias,
        # LayerNorm_0) by several percent of its max although the arithmetic is right.  So: the flips must all sit at the kink
        # (|input| <= 1e-2 of its max), and the oracle then takes the device's branch (oracle.classifier.forward relu_pattern) for the
        # 1e-2 gradient bar - once on the device's own fp16 trunk features (the heads alone) and once through the fp64 trunk (the chain).
        b = st._bufs[B]
        sc, bi = (p0[k].numpy() for k in ("LayerNorm_0/scale", "LayerNorm_0/bias"))
        pattern = b["xhat"].cpu().double().numpy() * sc + bi > 0           # the branch ln_relu_bwd took (same predicate, exact in fp64)
        feats = {c: b["feats"][c].cpu().double() for c in cams}
        errs = {}
        for tag, fts in (("heads_", feats), ("", None)):
            _, _, info0, grads0 = OC.train_step(p0, OC.new_opt(p0), cams, batch["data"], batch["labels"], masks=masks, feats=fts)
            pre = info0["_pre_relu"].numpy()
            flips = pattern != (pre > 0)
            errs[f"{tag}relu_flips"] = int(flips.sum())
            errs[f"{tag}flip_max_input_rel"] = float(np.abs(pre[flips]).max() / np.abs(pre).max()) if flips.any() else 0.0
            assert errs[f"{tag}flip_max_input_rel"] <= 1e-2, errs
            errs[f"{tag}grad_rel_fp64_branch"] = _check_step(st, info0, grads0, None, tol_out, None, False)["grad_rel"]   # recorded only
            _, _, pinfo, pgrads = OC.train_step(p0, OC.new_opt(p0), cams, batch["data"], batch["labels"], masks=masks, feats=fts,
                                                relu_pattern=pattern)
            errs.update({f"{tag}{k}": v for k, v in _check_step(st, pinfo, pgrads, None, tol_out, tol_grad, False).items()})
    for cam in cams:                                                # frozen trunk: bit-unchanged
        for k, v in st._trunk[cam].items():
            np.testing.assert_array_equal(v.cpu().numpy(), p0[f"encoder_def/encoder_{cam}/pretrained_encoder/{k}"].float().numpy())
    assert st.opt_state["count"] == 1 and st.step == 1
    st.check_status()
    return errs


@pytest.mark.parametrize("cams", [("front",), ("front", "wrist")])
def test_fp32_train_step_matches_oracle(cams):
    _one_host_step(cams, "fp32", 1e-5, 2e-4)


@pytest.mark.parametrize("cams", [("front",), ("front", "wrist")])
def test_fp16_train_step_within_16bit_bar(cams):
    errs = _one_host_step(cams, "fp16", 1e-2, 1e-2)
    print(f"\nfp16 classifier step {cams}: " + ", ".join(f"{k} {v:.2e}" if isinstance(v, float) else f"{k} {v}" for k, v in errs.items()))


def test_keyed_dropout_masks():
    from oracle import classifier as OC
    from serl_b200.networks.reward_classifier import train_step
    cams = ("front", "wrist")
    rng = np.random.default_rng(5)
    B = 6
    st = _state(cams)
    train_step(st, _host_batch(rng, cams, B), KEY)
    b = st._bufs[B]
    sle, hid = OC.dropout_masks(KEY, cams, B)
    for j, c in enumerate(cams):
        np.testing.assert_array_equal(b["masks"][j].cpu().numpy().astype(bool), sle[c])
    np.testing.assert_array_equal(b["hmask"].cpu().numpy().astype(bool), hid)


def _rings(cams, seed, hw=128, n=2):
    from serl_b200.utils.launcher import make_replay_buffer
    out = []
    for k in range(n):
        rb = make_replay_buffer(fake_env(cams, hw=hw), capacity=64, type="memory_efficient_replay_buffer", image_keys=list(cams), seed=seed + k)
        for tr in random_transitions(np.random.default_rng(seed + 10 * k), 50, cams, hw=hw):
            rb.insert(tr)
        out.append(rb)
    return out


def _oracle_crops(batch, cams):
    """Positive rows: next frames of the positive part; negative rows: frames of the negative part; one key over the batch."""
    from oracle import jax_prng as P
    from oracle.replay import random_shift
    from serl_b200.data.replay_buffer import BatchHandle
    B, half = batch.batch_size, batch.batch_size // 2
    pos = BatchHandle([dict(batch.pos)], False).to_dict()
    neg = BatchHandle([dict(batch.neg)], False).to_dict()
    off = P.crop_offsets(batch.aug_key, B)
    out = {}
    for c in cams:
        raw = np.concatenate([pos["next_observations"][c][:, 0].cpu().numpy(), neg["observations"][c][:, 0].cpu().numpy()])
        out[c] = random_shift(raw, off)
    assert raw.shape[0] == B and half * 2 == B
    return out


def test_lazy_batch_crops_graph_replay_and_oracle_chain():
    from oracle import classifier as OC
    from serl_b200.networks.reward_classifier import sample_classifier_batch, train_step
    cams = ("front", "wrist")
    B, steps = 8, 4
    runs = []
    for graphs in (True, False):
        st = _state(cams)
        st.use_cuda_graphs = graphs
        pos, neg = _rings(cams, 20)
        _, chain = OC.example_key_chain(steps)
        hist = []
        opt = None
        for i, (aug, drop) in enumerate(chain):
            batch = sample_classifier_batch(pos, neg, B, aug)
            p0 = _params64(st)
            st, loss, acc = train_step(st, batch, drop)
            b = st._bufs[B]
            crops = _oracle_crops(batch, cams)
            for c in cams:
                np.testing.assert_array_equal(b["pix"][c].cpu().numpy(), crops[c])
            np.testing.assert_array_equal(b["labels_lazy"].cpu().numpy(), np.r_[np.ones(B // 2), np.zeros(B // 2)])
            if not graphs:                                          # the eager run against the oracle's chain (keys, Adam count)
                if opt is None:
                    opt = OC.new_opt(p0)
                newp, opt, oinfo, grads = OC.train_step(p0, opt, cams, {c: crops[c][:, None] for c in cams},
                                                        np.r_[np.ones(B // 2), np.zeros(B // 2)][:, None], key=drop)
                st._b_last = B
                b["labels"].copy_(b["labels_lazy"])
                _check_step(st, oinfo, grads, newp, 1e-5, 2e-4, True)
                assert st.opt_state["count"] == opt["count"] == i + 1
            hist.append(st._params.clone())
        st.check_status()
        runs.append(hist)
    for a, b_ in zip(*runs):                                          # graph-replayed steps 2..4 == eager steps, bit for bit
        assert torch.equal(a, b_)


# 128: sample_frames_kernel; 100 (rows not 16-byte multiples): sample_gather_crop_kernel<false>; 256 (too tall for the one-shot
# shared-memory frame): sample_gather_crop_kernel<true>
@pytest.mark.parametrize("hw", [128, 100, 256])
def test_one_sided_sampler_equals_half_of_two_sided(hw):
    from serl_b200 import _lib as L
    cams = ("front", "wrist")
    ring, = _rings(cams, 40, hw=hw, n=1)
    B, dev = 6, "cuda"
    part = ring.sample(B).parts[0]
    key = torch.from_numpy(np.array([3, 4], np.uint32).view(np.int32)).view(torch.uint32).to(dev)
    e = lambda *s, dt=torch.float32: torch.zeros(*s, dtype=dt, device=dev)

    def run(obs_on, next_on):
        pix = {(c, w): e(2 * B, hw, hw, 3, dt=torch.uint8) for c in cams for w in ("o", "n")}
        out = L.BatchOut()
        for j, c in enumerate(cams):
            out.obs_pix[j] = pix[(c, "o")].data_ptr() if obs_on else None
            out.next_pix[j] = pix[(c, "n")].data_ptr() if next_on else None
        junk = [e(2 * B, 7), e(2 * B, 7), e(2 * B, 4), e(2 * B), e(2 * B), e(2 * B, dt=torch.uint8), e(1, dt=torch.int32)]
        out.obs_state, out.next_state, out.actions, out.rewards, out.masks = [t.data_ptr() for t in junk[:5]]
        out.dones, out.status = junk[5].data_ptr(), junk[6].data_ptr()
        ring.launch_sample(part, out, crop_total=2 * B, out_row_offset=B, key_obs=key.data_ptr(), key_next=key.data_ptr())
        torch.cuda.synchronize()
        return pix

    both, only_o, only_n = run(True, True), run(True, False), run(False, True)
    for c in cams:
        assert torch.equal(only_o[(c, "o")], both[(c, "o")]) and int(only_o[(c, "n")].sum()) == 0
        assert torch.equal(only_n[(c, "n")], both[(c, "n")]) and int(only_n[(c, "o")].sum()) == 0
        assert int(both[(c, "o")][B:].sum()) > 0


@pytest.mark.parametrize("precision,tol", [("fp32", 1e-5), ("fp16", 1e-2)])
def test_load_classifier_func_after_checkpoint(tmp_path, precision, tol):
    from oracle import classifier as OC
    from serl_b200.networks.reward_classifier import load_classifier_func, train_step
    from serl_b200.utils.checkpoints import save_checkpoint
    cams = ("front", "wrist")
    rng = np.random.default_rng(9)
    st = _state(cams, precision)
    train_step(st, _host_batch(rng, cams, 4), KEY)
    save_checkpoint(str(tmp_path), st, step=1)
    sample = {c: np.zeros((1, 1, 128, 128, 3), np.uint8) for c in cams}
    func = load_classifier_func(np.array([5, 5], np.uint32), sample, cams, str(tmp_path), precision=precision)
    assert func.state.step == 1 and func.state.opt_state["count"] == 1
    p = _params64(st)
    obs5 = {c: rng.integers(0, 256, (5, 1, 128, 128, 3), dtype=np.uint8) for c in cams}
    ref = OC.eval_logits(p, cams, obs5).numpy()
    out5 = func(obs5)
    assert out5.shape == (5, 1)
    assert np.abs(out5 - ref).max() <= tol * max(np.abs(ref).max(), 1.0)
    one = {**{c: obs5[c][0] for c in cams}, "state": np.zeros((1, 7), np.float32)}     # what the actor's env returns
    out1 = func(one)
    assert out1.shape == (1,)
    assert abs(float(out1[0]) - ref[0, 0]) <= tol * max(abs(ref[0, 0]), 1.0)
    r = 1 / (1 + np.exp(-func(one).item())) >= 0.5                                    # BinaryRewardClassifierWrapper's use
    assert r in (True, False)
    n0 = torch.cuda.memory_stats()["allocation.all.allocated"]                        # repeated calls: no device allocation
    for _ in range(3):
        func(one)
        func(obs5)
    assert torch.cuda.memory_stats()["allocation.all.allocated"] == n0
