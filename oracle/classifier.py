"""CPU restatement of the reference's reward classifier (test infrastructure only - never imported by serl_b200/).

Follows networks/reward_classifier.py:16-28 (BinaryClassifier: EncodingWrapper(use_proprio=False, enable_stacking=True) over
PreTrainedResNetEncoder heads -> Dense(256) -> Dropout(0.1) -> LayerNorm -> ReLU -> Dense(1)), create_classifier (:31-91:
optax.adam(1e-4)) and the training loop of examples/async_cable_route_drq/train_reward_classifier.py:84-170 (key chain,
positive next frames + negative frames, one batched_random_crop key, loss = optax.sigmoid_binary_cross_entropy(...).mean(),
accuracy of a train=False pass with the PRE-update parameters).  Trunk, LayerNorm and Adam algebra are oracle/drq.py's.
PARITY UNPINNED like oracle/drq.py (jax / flax / optax are not installable here).

Dropout keys (repo spec, DESIGN.md §4 (i)): camera j's SLE keep mask = bernoulli(fold_in(key, j), 0.9, (B, 4096)); the hidden
layer's keep mask = bernoulli(fold_in(key, ncam), 0.9, (B, 256)).

Parameters: flat {path: tensor} with the reference's tree paths:
  encoder_def/encoder_<cam>/{pretrained_encoder/..., SpatialLearnedEmbeddings_0/kernel, Dense_0/{kernel,bias}, LayerNorm_0/{scale,bias}}
  Dense_0/{kernel,bias}, LayerNorm_0/{scale,bias}, Dense_1/{kernel,bias}
"""
from __future__ import annotations

import numpy as np
import torch

from . import drq as O
from . import jax_prng as P
from .replay import random_shift

ENC = "encoder_def"
KEEP = 0.9


def trunk_features(params, cam, images_u8, dtype=torch.float64):
    """images (B, 1, H, W, 3) uint8 (enable_stacking: B T H W C -> B H W (T C)) -> (B, 4, 4, 512)."""
    img = torch.as_tensor(np.asarray(images_u8))
    if img.dim() == 4:
        img = img[:, None]
    b, t, h, w, c = img.shape
    pre = f"{ENC}/encoder_{cam}/pretrained_encoder/"
    trunk = {f"{O.ENC}/encoder_{cam}/pretrained_encoder/{k[len(pre):]}": v for k, v in params.items() if k.startswith(pre)}
    return O.trunk_forward(trunk, cam, img.permute(0, 2, 3, 1, 4).reshape(b, h, w, t * c), dtype)


def _pre_relu(params, cams, feats, sle_masks=None, hidden_mask=None):
    """The hidden ReLU's input of a pass (B, 256): LayerNorm(Dropout(Dense_0(concat_cam enc_cam))) * scale + bias."""
    outs = []
    for cam in cams:                                                       # resnet_v1.py:340-374 per camera, encoding.py:26-53
        pre = f"{ENC}/encoder_{cam}"
        k = params[f"{pre}/SpatialLearnedEmbeddings_0/kernel"]
        f = feats[cam].to(k.dtype)
        sle = torch.einsum("bhwc,hwcf->bcf", f, k).reshape(f.shape[0], -1)
        if sle_masks is not None:
            sle = torch.where(torch.as_tensor(np.asarray(sle_masks[cam])).bool(), sle / KEEP, torch.zeros_like(sle))
        z = sle @ params[f"{pre}/Dense_0/kernel"] + params[f"{pre}/Dense_0/bias"]
        outs.append(torch.tanh(O.layer_norm(z, params[f"{pre}/LayerNorm_0/scale"], params[f"{pre}/LayerNorm_0/bias"])))
    x = torch.cat(outs, dim=-1)
    x = x @ params["Dense_0/kernel"] + params["Dense_0/bias"]               # reward_classifier.py:23-27
    if hidden_mask is not None:
        x = torch.where(torch.as_tensor(np.asarray(hidden_mask)).bool(), x / KEEP, torch.zeros_like(x))
    return O.layer_norm(x, params["LayerNorm_0/scale"], params["LayerNorm_0/bias"])


def forward(params, cams, feats, sle_masks=None, hidden_mask=None, relu_pattern=None):
    """BinaryClassifier.__call__ -> logits (B, 1).  Masks given (bool keep masks) = train=True, None = train=False.
    relu_pattern (B, 256) bool: take the ReLU's branch from it instead of from the sign of its input.  Where the two agree this is
    the ReLU; where they differ the input lies at the kink (|x| at rounding level), so the forward value moves by |x| only, while
    the derivative follows the branch a lower-precision implementation chose - which lets its gradients be compared with this
    restatement's arithmetic rather than with a branch decision that rounding can flip."""
    x = _pre_relu(params, cams, feats, sle_masks, hidden_mask)
    if relu_pattern is None:
        x = torch.relu(x)
    else:
        x = torch.where(torch.as_tensor(np.asarray(relu_pattern)).bool(), x, torch.zeros_like(x))
    return x @ params["Dense_1/kernel"] + params["Dense_1/bias"]


def bce(logits, labels):
    """optax.sigmoid_binary_cross_entropy(logits, labels).mean() = mean(relu(x) - x*y + log1p(exp(-|x|)))."""
    x, y = logits, torch.as_tensor(np.asarray(labels)).to(logits.dtype).reshape(logits.shape)
    return (torch.relu(x) - x * y + torch.log1p(torch.exp(-x.abs()))).mean()


def accuracy(eval_logits, labels):
    """jnp.mean((nn.sigmoid(logits) >= 0.5) == labels)."""
    y = torch.as_tensor(np.asarray(labels)).to(eval_logits.dtype).reshape(eval_logits.shape)
    return ((torch.sigmoid(eval_logits) >= 0.5).to(y.dtype) == y).to(y.dtype).mean()


def dropout_masks(key, cams, B):
    """({cam: (B, 4096)}, (B, 256)) keep masks of one train=True pass with dropout key `key`."""
    key = np.asarray(key, np.uint32)
    sle = {cam: P.bernoulli(P.fold_in(key, j), KEEP, (B, 4096)) for j, cam in enumerate(cams)}
    return sle, P.bernoulli(P.fold_in(key, len(cams)), KEEP, (B, 256))


def example_key_chain(epochs):
    """train_reward_classifier.py:84-150: rng = PRNGKey(0); rng, key = split(rng) twice before create_classifier (the second key
    initialises it); per epoch rng, aug_key = split(rng), then rng, dropout_key = split(rng).
    Returns (init_key, [(aug_key, dropout_key)] * epochs)."""
    rng = P.prng_key(0)
    rng, _ = P.split(rng)
    rng, init_key = P.split(rng)
    out = []
    for _ in range(epochs):
        rng, aug = P.split(rng)
        rng, drop = P.split(rng)
        out.append((aug, drop))
    return init_key, out


def augment(images, aug_key):
    """data_augmentation_fn: batched_random_crop(padding=4, num_batch_dims=2) with ONE key for the whole (B, 1) batch: frame g uses
    split(aug_key, B)[g], the same offsets for every camera.  images {cam: (B, 1, H, W, 3)}."""
    cams = list(images)
    B = np.asarray(images[cams[0]]).shape[0]
    off = P.crop_offsets(np.asarray(aug_key, np.uint32), B)
    return {c: random_shift(np.asarray(images[c]).reshape(B, *np.asarray(images[c]).shape[2:]), off).reshape(np.asarray(images[c]).shape)
            for c in cams}, off


def train_step(params, opt, cams, images, labels, key=None, masks=None, lr=1e-4, dtype=torch.float64, feats=None, relu_pattern=None):
    """The example's jitted train_step on an already-augmented batch.  params: flat dict incl. the frozen trunk; opt =
    {"count", "mu", "nu"} over the trainable leaves; masks = (sle masks, hidden mask) or None -> keyed by `key`.
    feats: {cam: (B, 4, 4, 512)} trunk features to use instead of the fp64 trunk (isolates the heads of a 16-bit build).
    relu_pattern: the hidden ReLU's branch per entry of the train pass (see `forward`); info["_pre_relu"] is that pass's ReLU input.
    Returns (new_params, opt, info, grads); info: loss, accuracy, _logits (train pass), _eval_logits (train=False, pre-update)."""
    p = {k: v.detach().to(dtype) for k, v in params.items()}
    B = np.asarray(labels).shape[0]
    if feats is None:
        feats = {cam: trunk_features(p, cam, images[cam], dtype) for cam in cams}  # stop_gradient (resnet_v1.py:285-286)
    feats = {cam: torch.as_tensor(f).to(dtype) for cam, f in feats.items()}
    sle_m, hid_m = masks if masks is not None else dropout_masks(key, cams, B)
    train = {k: v.clone().requires_grad_(True) for k, v in p.items() if "pretrained_encoder" not in k}
    logits = forward({**p, **train}, cams, feats, sle_m, hid_m, relu_pattern)
    with torch.no_grad():
        pre = _pre_relu(p, cams, feats, sle_m, hid_m)
    loss = bce(logits, labels)
    gs = torch.autograd.grad(loss, list(train.values()), allow_unused=True)
    grads = {k: (torch.zeros_like(v) if g is None else g) for (k, v), g in zip(train.items(), gs)}
    with torch.no_grad():
        eval_logits = forward(p, cams, feats)
    upd = O.adam_tx_update(grads, opt, lr)
    new_params = dict(p)
    for k in train:
        new_params[k] = p[k] + upd[k]
    info = {"loss": loss.item(), "accuracy": accuracy(eval_logits, labels).item(), "_logits": logits.detach(), "_eval_logits": eval_logits,
            "_pre_relu": pre}
    return new_params, opt, info, grads


def new_opt(params, dtype=torch.float64):
    z = lambda: {k: torch.zeros_like(v, dtype=dtype) for k, v in params.items() if "pretrained_encoder" not in k}
    return {"count": 0, "mu": z(), "nu": z()}


def eval_logits(params, cams, images, dtype=torch.float64):
    """load_classifier_func's func(obs): train=False logits (B, 1)."""
    p = {k: v.detach().to(dtype) for k, v in params.items()}
    with torch.no_grad():
        return forward(p, cams, {cam: trunk_features(p, cam, images[cam], dtype) for cam in cams})
