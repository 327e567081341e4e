"""Reward classifier on the hand-written sm_100a kernels (reference networks/reward_classifier.py and the training loop of
examples/async_cable_route_drq/train_reward_classifier.py).

    logits = Dense(1)(ReLU(LayerNorm(Dropout(0.1)(Dense(256)(concat_cam enc_cam(image))))))        (reward_classifier.py:16-28)
    enc_cam = frozen ResNet-10 trunk -> SpatialLearnedEmbeddings -> Dropout(0.1) -> Dense(256) -> LayerNorm -> tanh
    loss = optax.sigmoid_binary_cross_entropy(logits_train, labels).mean(),   one optax.adam(1e-4)
    accuracy = mean((sigmoid(logits_eval) >= 0.5) == labels), logits_eval of a train=False pass with the PRE-update parameters

No stop_gradient on the image embeddings (EncodingWrapper's default): every image head, the MLP and the output layer are trained;
the trunk is frozen (resnet_v1.py:285-286).  The trunk runs ONCE per camera over the B images; the train pass (dropout masks
keyed bernoulli(fold_in(key, j)) per camera j and fold_in(key, ncam) for the hidden layer, DESIGN.md §4) and the eval pass share it.

Two builds, selected by `precision` like the agents':
  * "fp32": the 1e-5 parity build - SGEMM, ln_tanh_*, sle_*, ln_relu_* per op (the way agents/continuous/bc.py runs);
  * "fp16" / "bf16": the 16-bit tensor-core trunk and the fused heads - one SLE launch, one k-split TF32 GEMM launch and one finish
    launch for the image heads of both passes, one TF32 GEMM with the LN_RELU_HEAD epilogue (bias + dropout + LayerNorm + ReLU +
    logit) for the hidden layer of both passes, batched backward reductions.
Both share the BCE loss kernel, the LayerNorm + ReLU backward, the column reductions and the fused Adam.

A lazy batch (`sample_classifier_batch`) is trained by a CUDA graph captured once per (batch size, rings) and replayed: both
one-sided sampler launches, trunk, heads, loss, backward and Adam; keys reach the graph through device memory.
"""
from __future__ import annotations

import contextlib
import os
import pickle
from typing import Dict, Iterable, Optional

import numpy as np
import torch

from .. import _lib as L
from .. import ops
from ..agents.continuous.bc import _TrunkHost
from ..engine import AgentConfig, Engine
from ..params import Leaf, flatten, init_trunk, lecun_normal, nest

f32 = torch.float32
ENC = "encoder_def"
KEEP = 0.9


def classifier_spec(cams):
    """Trainable leaves in the reference's tree layout (trunk excluded), 16-byte aligned offsets in one flat buffer."""
    leaves = []
    for cam in cams:
        p = f"{ENC}/encoder_{cam}"
        leaves += [Leaf(f"{p}/SpatialLearnedEmbeddings_0/kernel", (4, 4, 512, 8), 0), Leaf(f"{p}/Dense_0/kernel", (4096, 256), 0),
                   Leaf(f"{p}/Dense_0/bias", (256,), 0), Leaf(f"{p}/LayerNorm_0/scale", (256,), 0), Leaf(f"{p}/LayerNorm_0/bias", (256,), 0)]
    leaves += [Leaf("Dense_0/kernel", (256 * len(cams), 256), 0), Leaf("Dense_0/bias", (256,), 0), Leaf("LayerNorm_0/scale", (256,), 0),
               Leaf("LayerNorm_0/bias", (256,), 0), Leaf("Dense_1/kernel", (256, 1), 0), Leaf("Dense_1/bias", (1,), 0)]
    off = 0
    for l in leaves:
        l.offset = off
        off += (l.size + 3) // 4 * 4
    return leaves, off


def _key_np(key):
    return np.asarray(key, dtype=np.uint32).reshape(2)


class ClassifierBatch:
    """A not-yet-materialised classifier batch: B/2 positive rows (their NEXT frames, label 1) then B/2 negative rows (their
    frames, label 0), cropped with ONE augmentation key over the whole batch (frame g: split(aug_key, B)[g])."""

    def __init__(self, pos_part, neg_part, batch_size, aug_key):
        self.pos, self.neg, self.batch_size, self.aug_key = pos_part, neg_part, int(batch_size), _key_np(aug_key)


def sample_classifier_batch(pos_buffer, neg_buffer, batch_size: int, aug_key) -> ClassifierBatch:
    """train_reward_classifier.py:153-169 as a lazy device batch (both replay rings stay in HBM)."""
    if batch_size % 2:
        raise ValueError("sample_classifier_batch: batch_size must be even (half positive, half negative)")
    pos = pos_buffer.sample(batch_size // 2).parts[0]
    neg = neg_buffer.sample(batch_size // 2).parts[0]
    return ClassifierBatch(pos, neg, batch_size, aug_key)


class ClassifierState:
    """The classifier's TrainState: `.params` (nested NumPy tree incl. the frozen trunk), `.step`, `.opt_state`, `.replace`,
    `state_dict()` / `load_state_dict()` (serl_b200/utils/checkpoints.py).  Device buffers and launch plans live here too."""

    def __init__(self, cams, hw, precision, device, spec, n, trunk):
        self.cams, self.hw, self.precision, self.device = tuple(cams), int(hw), precision, torch.device(device)
        self._spec, self._n, self._trunk = spec, n, trunk
        self._leaf = {l.path: l for l in spec}
        self._cfg = AgentConfig(cams=self.cams, state_in=1, action_dim=1, pixel=True, image_hw=self.hw, precision=precision)
        z = lambda: torch.zeros(n, dtype=f32, device=self.device)
        self._params, self._m, self._v, self._grad = z(), z(), z(), z()
        self._counts = torch.zeros(3, dtype=torch.int32, device=self.device)
        self._lr_info = torch.zeros(4, dtype=f32, device=self.device)
        self._info = torch.zeros(2, dtype=f32, device=self.device)
        self._keys = torch.zeros(4, dtype=torch.uint32, device=self.device)       # [aug key | dropout key]
        self.step = 0
        self._lr = 1e-4                       # optax.adam(1e-4) (reward_classifier.py:66)
        self.fused = precision != "fp32"
        self.explicit_dropout = None          # tests: ({cam: (B, 4096)}, (B, 256)) keep masks instead of the keyed ones
        self.use_cuda_graphs = True
        self._bufs: Dict[int, dict] = {}
        self._graphs = {}
        self._launch_adj = 0

    # ---- TrainState surface ------------------------------------------------------------------------------
    def _tree(self, buf, trunk=True):
        host = buf.detach().cpu().numpy()
        flat = {l.path: host[l.offset:l.offset + l.size].reshape(l.shape).copy() for l in self._spec}
        if trunk:
            for cam, leaves in self._trunk.items():
                for k, v in leaves.items():
                    flat[f"{ENC}/encoder_{cam}/pretrained_encoder/{k}"] = v.detach().cpu().numpy()
        return nest(flat)

    @property
    def params(self):
        return self._tree(self._params)

    @property
    def opt_state(self):
        return {"count": int(self._counts[0].item()), "mu": self._tree(self._m, False), "nu": self._tree(self._v, False)}

    def replace(self, **kw):
        """state.replace(params=tree[, step=n]): writes the trainable leaves and the frozen trunk from a tree in this layout."""
        if "params" in kw:
            flat = flatten(kw.pop("params"))
            host = self._params.detach().cpu()
            for l in self._spec:
                if l.path in flat:
                    host[l.offset:l.offset + l.size] = torch.as_tensor(np.asarray(flat[l.path], np.float32)).reshape(-1)
            self._params.copy_(host)
            for cam, leaves in self._trunk.items():
                for k in leaves:
                    key = f"{ENC}/encoder_{cam}/pretrained_encoder/{k}"
                    if key in flat:
                        leaves[k].copy_(torch.as_tensor(np.asarray(flat[key], np.float32)).to(self.device))
            self._invalidate()
        if "step" in kw:
            self.step = int(kw.pop("step"))
        if kw:
            raise TypeError(f"replace: unknown fields {sorted(kw)}")
        return self

    def state_dict(self):
        return {"step": self.step, "params": self.params, "opt_state": self.opt_state}

    def load_state_dict(self, d):
        self.replace(params=d["params"], step=d.get("step", 0))
        o = d.get("opt_state")
        if o is not None:
            for buf, tree in ((self._m, o["mu"]), (self._v, o["nu"])):
                flat, host = flatten(tree), buf.detach().cpu()
                for l in self._spec:
                    if l.path in flat:
                        host[l.offset:l.offset + l.size] = torch.as_tensor(np.asarray(flat[l.path], np.float32)).reshape(-1)
                buf.copy_(host)
            self._counts[0] = int(o["count"])
        return self

    @property
    def learning_rate(self) -> float:
        return self._lr

    @learning_rate.setter
    def learning_rate(self, lr):
        """Captured step graphs hold the learning rate as a launch argument: a new value drops them (recaptured on demand)."""
        if float(lr) != self._lr:
            self._lr = float(lr)
            self._graphs.clear()

    def _invalidate(self):
        self._graphs.clear()
        for b in self._bufs.values():                          # packed 16-bit trunk weights are derived from the fp32 ones
            b["host"].__dict__.pop("_tc_weights", None)

    @property
    def kernel_launches(self) -> int:
        """Kernels of libserl_b200 executed so far in this process (graph capture / replay corrected, like SACAgent's)."""
        return L.launch_count() + self._launch_adj

    # ---- buffers ----------------------------------------------------------------------------------------------
    def _P(self, buf, path):
        return buf.data_ptr() + 4 * self._leaf[path].offset

    def _b(self, B):
        if B not in self._bufs:
            dev, nc, F = self.device, len(self.cams), 256 * len(self.cams)
            e = lambda *s: torch.empty(*s, dtype=f32, device=dev)
            u8 = lambda *s: torch.zeros(*s, dtype=torch.uint8, device=dev)
            b = dict(host=_TrunkHost(self._cfg, self._trunk, B, dev), ws=ops.Workspace(48 << 20, dev, "f32"),
                     pix={c: u8(B, self.hw, self.hw, 3) for c in self.cams}, feats={c: e(B, 4, 4, 512) for c in self.cams},
                     masks=u8(nc, B, 4096), hmask=u8(B, 256), sle=e(nc, B, 4096), sle_e=e(nc, B, 4096), d_sle=e(nc, B, 4096),
                     X=e(B, F), Xe=e(B, F), dX=e(B, F), enc_z=e(B, 256), enc_xhat=e(nc, B, 256), enc_rstd=e(nc, B),
                     dez=e(nc, B, 256), dey=e(nc, B, 256), z=e(B, 256), h=e(B, 256), h_e=e(B, 256), xhat=e(B, 256), rstd=e(B),
                     logit=e(B), logit_e=e(B), dlogit=e(B), dz=e(B, 256), dy=e(B, 256), labels=e(B),
                     labels_lazy=torch.cat([torch.ones(B // 2), torch.zeros(B - B // 2)]).to(dev, f32),
                     status=torch.zeros(1, dtype=torch.int32, device=dev), error=torch.zeros(1, dtype=torch.int32, device=dev))
            if self.fused:
                tiles = 2 * nc * ((B + 127) // 128)
                b["S"] = ops.tgemm_splits(4096, max(1, min(148 // tiles, 32)))
                b["ws_enc"] = ops.Workspace(2 * nc * b["S"] * B * 256 * 4, dev)
            self._bufs[B] = b
        return self._bufs[B]

    # ---- forward: trunk once per camera, then the train pass (masks, saves) and / or the eval pass -----------------
    def _trunk_forward(self, b):
        for cam in self.cams:
            Engine.trunk_forward(b["host"], cam, b["pix"][cam], b["feats"][cam])

    def _heads_forward(self, b, B, train: bool, evaluate: bool):
        P, Pm, F, nc = self._P, self._params, 256 * len(self.cams), len(self.cams)
        passes = ([("train", b["X"], b["sle"], b["masks"], b["h"], b["logit"])] if train else []) + \
                 ([("eval", b["Xe"], b["sle_e"], None, b["h_e"], b["logit_e"])] if evaluate else [])
        if self.fused:
            S, ws, err = b["S"], b["ws_enc"], b["error"]
            sle, gemm, fin = [], [], []
            for pi, (kind, X, sles, masks, h, logit) in enumerate(passes):
                for j, cam in enumerate(self.cams):
                    p = f"{ENC}/encoder_{cam}"
                    i = pi * nc + j
                    sle.append((b["feats"][cam].data_ptr(), P(Pm, f"{p}/SpatialLearnedEmbeddings_0/kernel"),
                                None if masks is None else masks[j].data_ptr(), sles[j].data_ptr(), 4096))
                    gemm.append(ops.tgemm_problem(sles[j].data_ptr(), P(Pm, f"{p}/Dense_0/kernel"), sAm=4096, sAk=1, sBk=256, sBn=1))
                    fin.append(dict(partials=ws.buf.data_ptr() + 4 * i * S * B * 256, S=S, bias=P(Pm, f"{p}/Dense_0/bias"),
                                    ln_scale=P(Pm, f"{p}/LayerNorm_0/scale"), ln_bias=P(Pm, f"{p}/LayerNorm_0/bias"), out=ops.at(X, 256 * j),
                                    ld_out=F, D=256, xhat=b["enc_xhat"][j].data_ptr() if kind == "train" else None,
                                    rstd=b["enc_rstd"][j].data_ptr() if kind == "train" else None))
            ops.sle_fwd_multi(sle, KEEP, B, 16, 512)
            ops.tgemm(ws, gemm, B, 256, 4096, epilogue=L.TGEMM_PARTIAL, splits=S, error=err)
            ops.enc_finish(fin, B)
            probs = [ops.tgemm_problem(X.data_ptr(), P(Pm, "Dense_0/kernel"), sAm=F, sAk=1, sBk=256, sBn=1,
                                       C_=h.data_ptr() if kind == "train" else None, ldc=256, bias=P(Pm, "Dense_0/bias"),
                                       ln_scale=P(Pm, "LayerNorm_0/scale"), ln_bias=P(Pm, "LayerNorm_0/bias"),
                                       xhat=b["xhat"].data_ptr() if kind == "train" else None, rstd=b["rstd"].data_ptr() if kind == "train" else None,
                                       head_w=P(Pm, "Dense_1/kernel"), head_b=P(Pm, "Dense_1/bias"), head_out=logit.data_ptr(), ld_head=1,
                                       keep_mask=None if kind != "train" else b["hmask"].data_ptr(), keep=KEEP)
                     for kind, X, sles, masks, h, logit in passes]
            ops.tgemm(None, probs, B, 256, F, epilogue=L.TGEMM_LN_RELU_HEAD, head_n=1, error=err)
            return
        ws = b["ws"]
        for kind, X, sles, masks, h, logit in passes:
            for j, cam in enumerate(self.cams):
                p = f"{ENC}/encoder_{cam}"
                l = self._leaf[f"{p}/SpatialLearnedEmbeddings_0/kernel"]
                ops.sle_fwd(b["feats"][cam], Pm[l.offset:l.offset + l.size].view(l.shape), None if masks is None else masks[j], KEEP,
                            sles[j].data_ptr(), 4096)
                ops.dense_fwd(ws, sles[j].data_ptr(), 4096, P(Pm, f"{p}/Dense_0/kernel"), P(Pm, f"{p}/Dense_0/bias"), b["enc_z"].data_ptr(),
                              256, B, 4096, 256)
                save = kind == "train"
                ops.ln_tanh_fwd(b["enc_z"].data_ptr(), 256, P(Pm, f"{p}/LayerNorm_0/scale"), P(Pm, f"{p}/LayerNorm_0/bias"), B, 0,
                                ops.at(X, 256 * j), F, b["enc_xhat"][j].data_ptr() if save else None,
                                b["enc_rstd"][j].data_ptr() if save else None, B, 256)
            ops.dense_fwd(ws, X.data_ptr(), F, P(Pm, "Dense_0/kernel"), P(Pm, "Dense_0/bias"), b["z"].data_ptr(), 256, B, F, 256)
            save = kind == "train"
            ops.ln_relu_fwd(b["z"].data_ptr(), 256, b["hmask"].data_ptr() if save else None, KEEP, P(Pm, "LayerNorm_0/scale"),
                            P(Pm, "LayerNorm_0/bias"), h.data_ptr(), 256, b["xhat"].data_ptr() if save else None,
                            b["rstd"].data_ptr() if save else None, B, 256)
            ops.dense_fwd(ws, h.data_ptr(), 256, P(Pm, "Dense_1/kernel"), P(Pm, "Dense_1/bias"), logit.data_ptr(), 1, B, 256, 1)

    # ---- backward (every trainable leaf; the trunk is frozen) --------------------------------------------------
    def _backward(self, b, B):
        P, Pm, G, F, nc = self._P, self._params, self._grad, 256 * len(self.cams), len(self.cams)
        G.zero_()
        ops.ln_relu_bwd(None, 0, b["dlogit"].data_ptr(), P(Pm, "Dense_1/kernel"), b["xhat"].data_ptr(), b["rstd"].data_ptr(),
                        P(Pm, "LayerNorm_0/scale"), P(Pm, "LayerNorm_0/bias"), b["hmask"].data_ptr(), KEEP, b["dz"].data_ptr(),
                        b["dy"].data_ptr(), B, 256)
        jobs = [(L.SMALL_GRAD_HEAD, b["h"].data_ptr(), 256, b["dlogit"].data_ptr(), 1, P(G, "Dense_1/kernel"), P(G, "Dense_1/bias"), 1, B, 256),
                (L.SMALL_GRAD_LN, b["dy"].data_ptr(), 256, b["xhat"].data_ptr(), 256, P(G, "LayerNorm_0/scale"), P(G, "LayerNorm_0/bias"), 1, B, 256),
                (L.SMALL_GRAD_COLSUM, b["dz"].data_ptr(), 256, None, 0, P(G, "Dense_0/bias"), None, 1, B, 256)]
        X, dX, ws = b["X"], b["dX"], b["ws"]
        if self.fused:
            err = b["error"]
            ops.tgemm(None, [ops.tgemm_problem(X.data_ptr(), b["dz"].data_ptr(), sAm=1, sAk=F, sBk=256, sBn=1, C_=P(G, "Dense_0/kernel"), ldc=256)],
                      F, 256, B, splits=1, error=err)
            ops.tgemm(None, [ops.tgemm_problem(b["dz"].data_ptr(), P(Pm, "Dense_0/kernel"), sAm=256, sAk=1, sBk=1, sBn=256, C_=dX.data_ptr(), ldc=F)],
                      B, F, 256, splits=1, error=err)
            lnb, wg, dsle = [], [], []
            for j, cam in enumerate(self.cams):
                p = f"{ENC}/encoder_{cam}"
                dez, dey = b["dez"][j], b["dey"][j]
                lnb.append(dict(dt=ops.at(dX, 256 * j), ld_dt=F, t=ops.at(X, 256 * j), ld_t=F, xhat=b["enc_xhat"][j].data_ptr(),
                                rstd=b["enc_rstd"][j].data_ptr(), scale=P(Pm, f"{p}/LayerNorm_0/scale"), rows_per_group=B, group_stride=0,
                                dz=dez.data_ptr(), dy=dey.data_ptr(), R=B, D=256))
                wg.append(ops.tgemm_problem(b["sle"][j].data_ptr(), dez.data_ptr(), sAm=1, sAk=4096, sBk=256, sBn=1, C_=P(G, f"{p}/Dense_0/kernel"), ldc=256))
                dsle.append(ops.tgemm_problem(dez.data_ptr(), P(Pm, f"{p}/Dense_0/kernel"), sAm=256, sAk=1, sBk=1, sBn=256, C_=b["d_sle"][j].data_ptr(), ldc=4096))
                jobs.append((L.SMALL_GRAD_COLSUM, dez.data_ptr(), 256, None, 0, P(G, f"{p}/Dense_0/bias"), None, 1, B, 256))
                jobs.append((L.SMALL_GRAD_LN, dey.data_ptr(), 256, b["enc_xhat"][j].data_ptr(), 256, P(G, f"{p}/LayerNorm_0/scale"), P(G, f"{p}/LayerNorm_0/bias"), 1, B, 256))
            ops.ln_tanh_bwd_multi(lnb)
            ops.small_grads(jobs)
            ops.tgemm(None, wg, 4096, 256, B, splits=1, error=err)
            ops.tgemm(None, dsle, B, 4096, 256, splits=1, error=err)
        else:
            ops.small_grads(jobs)
            ops.dense_bwd_weight(ws, X.data_ptr(), F, b["dz"].data_ptr(), 256, P(G, "Dense_0/kernel"), B, F, 256)
            ops.dense_bwd_input(ws, b["dz"].data_ptr(), 256, P(Pm, "Dense_0/kernel"), dX.data_ptr(), F, B, F, 256)
            for j, cam in enumerate(self.cams):
                p = f"{ENC}/encoder_{cam}"
                dez, dey = b["dez"][j], b["dey"][j]
                ops.ln_tanh_bwd(ops.at(dX, 256 * j), F, ops.at(X, 256 * j), F, b["enc_xhat"][j].data_ptr(), b["enc_rstd"][j].data_ptr(),
                                P(Pm, f"{p}/LayerNorm_0/scale"), B, 0, dez.data_ptr(), dey.data_ptr(), P(G, f"{p}/LayerNorm_0/scale"),
                                P(G, f"{p}/LayerNorm_0/bias"), B, 256)
                ops.dense_bwd_weight(ws, b["sle"][j].data_ptr(), 4096, dez.data_ptr(), 256, P(G, f"{p}/Dense_0/kernel"), B, 4096, 256)
                ops.colsum(dez.data_ptr(), P(G, f"{p}/Dense_0/bias"), 1, B, 256, 256)
                ops.dense_bwd_input(ws, dez.data_ptr(), 256, P(Pm, f"{p}/Dense_0/kernel"), b["d_sle"][j].data_ptr(), 4096, B, 4096, 256)
        # SLE Dropout backward (the train pass's keep masks), then the SLE kernel gradients of every camera
        ops.dropout_bwd(b["d_sle"].data_ptr(), b["masks"].data_ptr(), KEEP, nc * B * 4096)
        ops.sle_bwd_multi(ws, [(b["feats"][cam].data_ptr(), b["d_sle"][j].data_ptr(), 4096,
                                P(G, f"{ENC}/encoder_{cam}/SpatialLearnedEmbeddings_0/kernel")) for j, cam in enumerate(self.cams)], B, 16, 512)

    def _step_body(self, b, B, labels):
        """Everything after the batch is in `pix` and the keys are in `_keys`: masks, trunk, both passes, loss, backward, Adam."""
        nc = len(self.cams)
        if self.explicit_dropout is not None:
            sle_m, hid_m = self.explicit_dropout
            for j, cam in enumerate(self.cams):
                b["masks"][j].copy_(torch.as_tensor(np.asarray(sle_m[cam])).to(self.device, torch.uint8))
            b["hmask"].copy_(torch.as_tensor(np.asarray(hid_m)).to(self.device, torch.uint8))
        else:
            kd = ops.key_ptr(self._keys, 1)
            for j in range(nc):
                ops.dropout_mask_fill(kd, j, KEEP, b["masks"][j], B * 4096)
            ops.dropout_mask_fill(kd, nc, KEEP, b["hmask"], B * 256)
        self._trunk_forward(b)
        self._heads_forward(b, B, train=True, evaluate=True)
        ops.bce_logits_loss(b["logit"].data_ptr(), b["logit_e"].data_ptr(), labels.data_ptr(), B, 1.0, b["dlogit"].data_ptr(),
                            self._info.data_ptr())
        self._backward(b, B)
        n = self._n
        ops.adam_polyak(self._params, None, self._m, self._v, self._grad, [n, n, n], [1, 0, 0], self._counts, [self.learning_rate] * 3,
                        [0, 0, 0], 0.0, False, lr_out=self._lr_info, n=n, gap=0, aux=(0, 0, 0))

    # ---- batches ------------------------------------------------------------------------------------------------
    def _ingest(self, b, data):
        for cam in self.cams:
            px = data[cam]
            px = px if isinstance(px, torch.Tensor) else torch.as_tensor(np.asarray(px))
            if px.dim() == 5:
                if px.shape[1] != 1:
                    raise NotImplementedError("reward classifier: one frame per observation (obs_horizon=1), like every SERL example")
                px = px[:, 0]
            b["pix"][cam].copy_(px.to(self.device, torch.uint8), non_blocking=True)

    def _sample(self, b, batch: ClassifierBatch, graph_mode: bool):
        """Two one-sided sampler launches: positive rows' next frames -> rows [0, B/2), negative rows' frames -> [B/2, B)."""
        B, half = batch.batch_size, batch.batch_size // 2
        for part, row, side in ((batch.pos, 0, "next"), (batch.neg, half, "obs")):
            ring = part["ring"]
            if ring.T != 1:
                raise NotImplementedError("reward classifier: one frame per observation (obs_horizon=1)")
            key = (B, ring.T * ring.S, ring.A)
            if key not in b:
                e = lambda *s: torch.empty(*s, dtype=f32, device=self.device)
                b[key] = dict(st=e(B, ring.T * ring.S), nst=e(B, ring.T * ring.S), ac=e(B, ring.A), rw=e(B), mk=e(B),
                              dn=torch.empty(B, dtype=torch.uint8, device=self.device))
            j = b[key]
            out = L.BatchOut()
            for c, cam in enumerate(self.cams):
                if side == "next":
                    out.next_pix[c] = b["pix"][cam].data_ptr()
                else:
                    out.obs_pix[c] = b["pix"][cam].data_ptr()
            out.obs_state, out.next_state, out.actions = j["st"].data_ptr(), j["nst"].data_ptr(), j["ac"].data_ptr()
            out.rewards, out.masks, out.dones, out.status = j["rw"].data_ptr(), j["mk"].data_ptr(), j["dn"].data_ptr(), b["status"].data_ptr()
            ka = ops.key_ptr(self._keys, 0)
            ring.launch_sample(part, out, crop_total=B, out_row_offset=row, key_obs=ka if side == "obs" else None,
                               key_next=ka if side == "next" else None, step_dev=ring.step_dev if graph_mode else None,
                               record_event=not graph_mode)
            if graph_mode:
                ops.counter_add(ring.step_dev, 1)

    def _set_keys(self, aug_key, drop_key):
        k = np.concatenate([_key_np(aug_key) if aug_key is not None else np.zeros(2, np.uint32), _key_np(drop_key)])
        self._keys.copy_(torch.from_numpy(k.view(np.int32)).view(torch.uint32))

    def train_step(self, batch, key):
        if isinstance(batch, ClassifierBatch):
            B = batch.batch_size
            b = self._b(B)
            self._set_keys(batch.aug_key, key)
            gkey = None
            if self.use_cuda_graphs and self.explicit_dropout is None and self.device.type == "cuda" \
                    and batch.pos.get("indx") is None and batch.neg.get("indx") is None:
                gkey = (B, id(batch.pos["ring"]), id(batch.neg["ring"]))
            self._run(gkey, batch, lambda graph_mode: (self._sample(b, batch, graph_mode), self._step_body(b, B, b["labels_lazy"])))
        else:
            labels = batch["labels"]
            labels = labels if isinstance(labels, torch.Tensor) else torch.as_tensor(np.asarray(labels))
            B = int(labels.shape[0])
            b = self._b(B)
            self._set_keys(None, key)
            self._ingest(b, batch["data"])
            b["labels"].copy_(labels.reshape(-1).to(self.device, f32))
            self._step_body(b, B, b["labels"])
        self.step += 1
        snap = self._info.clone()
        return self, snap[0], snap[1]

    def _run(self, gkey, batch, body):
        """1st call with a key: eager; 2nd: capture + replay; later: replay only (SACAgent._run_step's scheme)."""
        if gkey is None:
            return body(False)
        entry = self._graphs.get(gkey)
        if entry is None:
            self._graphs[gkey] = "warm"
            return body(False)
        for p in (batch.pos, batch.neg):                       # device draw counter := this handle's step
            ring = p["ring"]
            if ring._dev_step_mirror != p["step"]:
                ring.step_dev.fill_(p["step"])
            ring._dev_step_mirror = p["step"] + 1
        if entry == "warm":
            g = torch.cuda.CUDAGraph()
            c0 = L.launch_count()
            with contextlib.ExitStack() as stack:
                for p in (batch.pos, batch.neg):
                    stack.enter_context(p["ring"]._lock)
                with torch.cuda.graph(g, capture_error_mode="thread_local"):
                    body(True)
            recorded = L.launch_count() - c0
            self._launch_adj -= recorded
            entry = self._graphs[gkey] = (g, recorded)
        g, recorded = entry
        g.replay()
        self._launch_adj += recorded

    def check_status(self):
        for b in self._bufs.values():
            if int(b["status"].item()):
                raise L.SerlError("replay draw failed: no valid slot within the redraw budget")
            if int(b["error"].item()):
                raise L.SerlError("tgemm_tf32_kernel: pipeline barrier timeout (flagged by the kernel)")

    # ---- inference (load_classifier_func) ----------------------------------------------------------------------
    def logits(self, obs):
        """train=False logits: (B, 1, H, W, 3) | (B, H, W, 3) per camera -> (B,) device tensor (a view of a reused buffer)."""
        first = obs[self.cams[0]]
        B = int(first.shape[0])
        b = self._b(B)
        self._ingest(b, obs)
        self._trunk_forward(b)
        self._heads_forward(b, B, train=False, evaluate=True)
        return b["logit_e"]

    def logits_host(self, obs, single: bool):
        """The same from host NumPy observations, staged through pinned buffers kept per batch size: a repeated call allocates
        neither device nor pinned memory, only the returned (B,) NumPy array.  single: obs[cam] is one (1, H, W, 3) observation."""
        B = 1 if single else int(np.asarray(obs[self.cams[0]]).shape[0])
        b = self._b(B)
        if "host_pix" not in b:
            b["host_pix"] = {c: L.pin(torch.empty(B, self.hw, self.hw, 3, dtype=torch.uint8)) for c in self.cams}
            b["host_logit"] = L.pin(torch.empty(B, dtype=f32))
            b["host_evt"] = L.new_event()
        for cam in self.cams:
            stage = b["host_pix"][cam]
            np.copyto(stage.numpy(), np.asarray(obs[cam]).reshape(stage.shape))
            b["pix"][cam].copy_(stage, non_blocking=True)
        self._trunk_forward(b)
        self._heads_forward(b, B, train=False, evaluate=True)
        b["host_logit"].copy_(b["logit_e"], non_blocking=True)
        b["host_evt"].record()
        b["host_evt"].synchronize()
        return b["host_logit"].numpy().copy()


def _load_pretrained(state: ClassifierState, path):
    """create_classifier's pretrained-trunk load (reward_classifier.py:68-89); a missing file keeps the synthetic trunk (like
    utils/train_utils.py::load_resnet10_params here: there is no download)."""
    if not path or not os.path.exists(path):
        print(f"{path} not found locally: keeping synthetic ResNet-10 weights")
        return state
    with open(path, "rb") as f:
        encoder_params = pickle.load(f)
    tree = state.params
    for cam in state.cams:
        enc = tree[ENC][f"encoder_{cam}"]["pretrained_encoder"]
        for k in list(enc):
            if k in encoder_params:
                enc[k] = {kk: np.asarray(vv) for kk, vv in encoder_params[k].items()} if isinstance(encoder_params[k], dict) \
                    else np.asarray(encoder_params[k])
    return state.replace(params=tree)


def create_classifier(key, sample, image_keys: Iterable[str], pretrained_encoder_path: str = "./resnet10_params.pkl", *,
                      precision: str = "fp32", device=None) -> ClassifierState:
    """reward_classifier.py:31-91.  `sample`: an observation dict (B, 1, H, W, 3) per camera (other keys ignored: use_proprio=False).
    Initial values: the repo's NumPy stream seeded by the key (flax's init stream is not reproducible here, DESIGN.md §4 (ii))."""
    L.load()
    device = torch.device(device if device is not None else "cuda")
    L.require_cuda(device)
    if precision not in ("fp32", "fp16", "bf16"):
        raise ValueError(f"precision must be fp32, fp16 or bf16, not {precision!r}")
    cams = tuple(image_keys)
    k = _key_np(key)
    rng = np.random.default_rng((int(k[0]) << 32) | int(k[1]))
    hw = int(np.asarray(sample[cams[0]]).shape[-2])
    spec, n = classifier_spec(cams)
    trunk = {cam: {kk: torch.as_tensor(v).to(device).contiguous() for kk, v in init_trunk(rng).items()} for cam in cams}
    st = ClassifierState(cams, hw, precision, device, spec, n, trunk)
    host = torch.zeros(n, dtype=f32)
    for l in spec:                                             # flax Dense / SLE defaults: lecun_normal kernels, zero biases, unit scales
        v = lecun_normal(rng, l.shape) if l.path.endswith("kernel") else (np.ones(l.shape, np.float32) if l.path.endswith("scale")
                                                                          else np.zeros(l.shape, np.float32))
        host[l.offset:l.offset + l.size] = torch.as_tensor(v).reshape(-1)
    st._params.copy_(host)
    return _load_pretrained(st, pretrained_encoder_path)


def train_step(state: ClassifierState, batch, key):
    """The example's jitted train_step (train_reward_classifier.py:122-137) -> (state, loss, accuracy).  batch: a
    `sample_classifier_batch` handle or the host form {"data": obs dict (already augmented), "labels": (B, 1)}; key: dropout key."""
    return state.train_step(batch, key)


def load_classifier_func(key, sample, image_keys, checkpoint_path, step: Optional[int] = None, *, precision: str = "fp32", device=None,
                         pretrained_encoder_path: str = "./resnet10_params.pkl"):
    """reward_classifier.py:94-117: func(obs) -> logits.  An unbatched observation ((1, H, W, 3) per camera, as the actor's env
    returns it; other keys ignored) gives shape (1,), a batch (B, 1, H, W, 3) gives (B, 1).  Device buffers and pinned host staging
    are kept per batch size, so a repeated call with NumPy observations allocates only the returned array; torch tensors (host or
    device) are copied in directly."""
    from ..utils.checkpoints import restore_checkpoint
    state = create_classifier(key, sample, image_keys, pretrained_encoder_path, precision=precision, device=device)
    state = restore_checkpoint(checkpoint_path, target=state, step=step)
    cams = state.cams

    def func(obs):
        x = obs[cams[0]]
        single = (x.dim() if isinstance(x, torch.Tensor) else np.ndim(x)) == 4
        if isinstance(x, torch.Tensor):
            out = state.logits({c: obs[c][None] for c in cams} if single else obs).detach().cpu().numpy()
        else:
            out = state.logits_host(obs, single)
        return out if single else out[:, None]

    func.state = state
    return func
