"""CPU: the reward classifier's restatement (oracle/classifier.py) - BCE against torch and the optax formula, autograd gradients
against central finite differences, the parameter tree of serl_b200.networks.reward_classifier, and the example's key chain /
crop offsets against the library's host mirrors of the device RNG."""
import numpy as np
import torch
import torch.nn.functional as F


def _params(rng, cams):
    from serl_b200.networks.reward_classifier import ENC, classifier_spec
    from serl_b200.params import init_trunk, lecun_normal
    spec, _ = classifier_spec(cams)
    p = {}
    for l in spec:
        if l.path.endswith("kernel"):
            v = lecun_normal(rng, l.shape)
        elif l.path.endswith("scale"):
            v = 1 + 0.1 * rng.standard_normal(l.shape)
        else:
            v = 0.05 * rng.standard_normal(l.shape)
        p[l.path] = torch.as_tensor(np.asarray(v, np.float64))
    for cam in cams:
        for k, v in init_trunk(rng).items():
            p[f"{ENC}/encoder_{cam}/pretrained_encoder/{k}"] = torch.as_tensor(v)
    return p


def test_bce_matches_torch_and_the_optax_formula():
    from oracle import classifier as OC
    rng = np.random.default_rng(0)
    x = torch.as_tensor(rng.standard_normal((64, 1)) * 6)
    y = torch.as_tensor((rng.random((64, 1)) < 0.5).astype(np.float64))
    ref = F.binary_cross_entropy_with_logits(x, y)
    optax = (-y * F.logsigmoid(x) - (1 - y) * F.logsigmoid(-x)).mean()       # optax.sigmoid_binary_cross_entropy
    got = OC.bce(x, y)
    assert abs(float(got - ref)) < 1e-14 and abs(float(got - optax)) < 1e-14
    assert float(OC.accuracy(torch.tensor([[0.0], [-1.0], [2.0]], dtype=torch.float64), np.array([[1.0], [0.0], [0.0]]))) == 2 / 3


def test_gradients_match_finite_differences():
    from oracle import classifier as OC
    cams = ("front", "wrist")
    rng = np.random.default_rng(1)
    params = _params(rng, cams)
    B = 4
    images = {c: rng.integers(0, 256, (B, 1, 128, 128, 3), dtype=np.uint8) for c in cams}
    labels = np.array([[1.0], [1.0], [0.0], [0.0]])
    sle_m = {c: rng.random((B, 4096)) < 0.9 for c in cams}
    hid_m = rng.random((B, 256)) < 0.9
    newp, opt, info, grads = OC.train_step(params, OC.new_opt(params), cams, images, labels, masks=(sle_m, hid_m))
    for k, g in grads.items():
        assert float(g.abs().max()) > 0.0, k                                  # no stop_gradient: every trainable leaf is reached
    assert opt["count"] == 1
    feats = {c: OC.trunk_features(params, c, images[c]) for c in cams}

    def loss(p):
        return float(OC.bce(OC.forward(p, cams, feats, sle_m, hid_m), labels))

    for path in ("Dense_0/kernel", "LayerNorm_0/scale", "Dense_1/kernel", "Dense_1/bias", "encoder_def/encoder_wrist/Dense_0/kernel",
                 "encoder_def/encoder_front/SpatialLearnedEmbeddings_0/kernel", "encoder_def/encoder_front/LayerNorm_0/bias"):
        flat = params[path].reshape(-1)
        for idx in rng.integers(0, flat.numel(), 2):
            h = 1e-6
            vals = []
            for sgn in (+1, -1):
                t = flat.clone()
                t[idx] += sgn * h
                vals.append(loss({**params, path: t.reshape(params[path].shape)}))
            fd = (vals[0] - vals[1]) / (2 * h)
            an = float(grads[path].reshape(-1)[idx])
            assert abs(fd - an) <= 1e-6 * max(abs(an), 1e-3) + 1e-9, (path, int(idx), fd, an)
    k = "Dense_0/kernel"                                                       # first Adam step moves every live entry by lr
    moved = (newp[k] - params[k]).abs()
    assert abs(float(moved.max()) - 1e-4) < 1e-7


def test_parameter_tree_matches_the_reference_layout():
    from serl_b200.networks.reward_classifier import classifier_spec
    for cams in (("front",), ("front", "wrist")):
        want = {}
        for c in cams:
            p = f"encoder_def/encoder_{c}"
            want.update({f"{p}/SpatialLearnedEmbeddings_0/kernel": (4, 4, 512, 8), f"{p}/Dense_0/kernel": (4096, 256),
                         f"{p}/Dense_0/bias": (256,), f"{p}/LayerNorm_0/scale": (256,), f"{p}/LayerNorm_0/bias": (256,)})
        want.update({"Dense_0/kernel": (256 * len(cams), 256), "Dense_0/bias": (256,), "LayerNorm_0/scale": (256,),
                     "LayerNorm_0/bias": (256,), "Dense_1/kernel": (256, 1), "Dense_1/bias": (1,)})
        spec, n = classifier_spec(cams)
        assert {l.path: tuple(l.shape) for l in spec} == want
        assert all(l.offset % 4 == 0 for l in spec) and n >= sum(l.size for l in spec)


def test_example_key_chain_and_batch_crop_offsets_match_host_mirrors():
    import __graft_entry__ as G
    G.build()
    from oracle import classifier as OC
    from oracle import jax_prng as P
    from serl_b200 import _lib as L
    L.load()

    def split(key, n=2):
        out = np.zeros((n, 2), np.uint32)
        L.call("serl_host_threefry_split", np.ascontiguousarray(key, np.uint32).ctypes.data, n, out.ctypes.data)
        return out

    init_key, epochs = OC.example_key_chain(3)
    rng = P.prng_key(0)
    rng = split(rng)[0]
    rng, key = split(rng)
    np.testing.assert_array_equal(init_key, key)
    B = 256
    for aug, drop in epochs:
        rng, a = split(rng)
        rng, d = split(rng)
        np.testing.assert_array_equal(aug, a)
        np.testing.assert_array_equal(drop, d)
        off = np.zeros((B, 2), np.int32)
        L.call("serl_host_crop_offsets", np.ascontiguousarray(a).ctypes.data, B, 4, off.ctypes.data)
        images = {"front": np.zeros((B, 1, 16, 16, 3), np.uint8)}
        _, want = OC.augment(images, aug)
        np.testing.assert_array_equal(off, want)                       # rows [0, B/2): positives, [B/2, B): negatives, one key
        # each row's offsets are split(key, B)[g] - the same for a row whether it lies in the positive or the negative half
        for g in (0, B // 2 - 1, B // 2, B - 1):
            np.testing.assert_array_equal(off[g], P.randint(P.split(aug, B)[g], (2,), 0, 9))
