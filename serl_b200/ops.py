"""Thin torch-tensor wrappers over the C-ABI ops (pointer + stream extraction only; no math here).

torch is plumbing: it owns device memory and the current stream.  Every function launches
hand-written kernels from libserl_b200.so and raises if the library or a launch fails.
"""
from __future__ import annotations

import ctypes as C
from typing import Optional, Sequence

import torch

from . import _lib as L


def _p(t: Optional[torch.Tensor]):
    return None if t is None else t.data_ptr()


def _s():
    return L.stream_ptr()


def _chk(t: torch.Tensor, dtype, name):
    if t.dtype != dtype:
        raise TypeError(f"{name}: expected {dtype}, got {t.dtype}")
    return t


# ---- trunk (fp32) ----------------------------------------------------------------------------------
def conv2d_nhwc(x, w, y, stride, pad_lo, pad_hi):
    """x (N,Hi,Wi,Ci) u8|f32, w (kh,kw,Ci,Co) f32 -> y (N,Ho,Wo,Co) f32."""
    N, Hi, Wi, Ci = x.shape
    kh, kw, ci2, Co = w.shape
    assert ci2 == Ci and x.is_contiguous() and w.is_contiguous() and y.is_contiguous()
    L.call("serl_conv2d_nhwc_f32", _p(x), int(x.dtype == torch.uint8), _p(w), _p(y), N, Hi, Wi, Ci, Co, kh, kw, stride,
           pad_lo, pad_hi, _s())
    return y


def groupnorm_nhwc(x, y, scale, bias, residual, groups, eps, relu):
    N, H, W, Cc = x.shape
    L.call("serl_groupnorm_nhwc_f32", _p(x), _p(y), _p(scale), _p(bias), _p(residual), N, H * W, Cc, groups, float(eps),
           int(relu), _s())
    return y


def maxpool3x3s2_nhwc(x, y):
    N, H, W, Cc = x.shape
    L.call("serl_maxpool3x3s2_nhwc_f32", _p(x), _p(y), N, H, W, Cc, _s())
    return y


# ---- GEMM -------------------------------------------------------------------------------------------
class Workspace:
    """Caller-owned scratch for split-K / batch-reduce partials."""

    GEMM_IMPLS = {"f32": "serl_gemm_f32", "tf32x3": "serl_gemm_tf32x3"}

    def __init__(self, nbytes: int, device, gemm_impl: str = "f32"):
        self.buf = torch.empty(nbytes // 4, dtype=torch.float32, device=device)
        self.nbytes = self.buf.numel() * 4
        self.gemm_fn = self.GEMM_IMPLS[gemm_impl]      # CUDA-core SGEMM (1e-5 build) or tensor-core 3xTF32 (speed builds)


def gemm(ws: Workspace, A_ptr, B_ptr, C_ptr, M, N, K, *, sAm, sAk, sBk, sBn, ldc, Z=1, sAz=0, sBz=0, sCz=0,
         bias_ptr=None, sBiasZ=0, accumulate=False, reduce_z=False):
    d = L.GemmDesc()
    d.A, d.B, d.C, d.bias = A_ptr, B_ptr, C_ptr, bias_ptr
    d.workspace, d.workspace_bytes = ws.buf.data_ptr(), ws.nbytes
    d.M, d.N, d.K, d.Z = M, N, K, Z
    d.sAz, d.sAm, d.sAk, d.sBz, d.sBk, d.sBn, d.sCz, d.sBiasZ = sAz, sAm, sAk, sBz, sBk, sBn, sCz, sBiasZ
    d.ldc, d.accumulate, d.reduce_z = ldc, int(accumulate), int(reduce_z)
    L.call(ws.gemm_fn, C.byref(d), _s())


def at(t: torch.Tensor, elem_offset: int = 0) -> int:
    """Device address of element `elem_offset` of a tensor's storage view."""
    return t.data_ptr() + elem_offset * t.element_size()


def dense_fwd(ws, x, ldx, w, b, out, ldo, M, K, N, *, Z=1, x_z=0, w_z=None, b_z=None, out_z=0):
    """out[z] (M,N) = x[z] (M,K) @ w[z] (K,N) + b[z];  x/out given as (address, ld)."""
    gemm(ws, x, w, out, M, N, K, sAm=ldx, sAk=1, sBk=N, sBn=1, ldc=ldo, Z=Z, sAz=x_z, sBz=(K * N if w_z is None else w_z),
         sCz=out_z, bias_ptr=b, sBiasZ=(N if b_z is None else b_z))


def dense_bwd_weight(ws, x, ldx, dz, lddz, dw, M, K, N, *, Z=1, x_z=0, dz_z=0, dw_z=None):
    """dw[z] (K,N) = x[z]^T (K,M) @ dz[z] (M,N)."""
    gemm(ws, x, dz, dw, K, N, M, sAm=1, sAk=ldx, sBk=lddz, sBn=1, ldc=N, Z=Z, sAz=x_z, sBz=dz_z,
         sCz=(K * N if dw_z is None else dw_z))


def dense_bwd_input(ws, dz, lddz, w, dx, lddx, M, K, N, *, Z=1, dz_z=0, w_z=None, dx_z=0, reduce_z=False, accumulate=False):
    """dx[z] (M,K) = dz[z] (M,N) @ w[z]^T (N,K)   (w stored (K,N) row-major)."""
    gemm(ws, dz, w, dx, M, K, N, sAm=lddz, sAk=1, sBk=1, sBn=N, ldc=lddx, Z=Z, sAz=dz_z, sBz=(K * N if w_z is None else w_z),
         sCz=dx_z, reduce_z=reduce_z, accumulate=accumulate)


# ---- heads -------------------------------------------------------------------------------------------
def sle_fwd(feat, kernel, keep_mask, keep, out, ld_out):
    N, Pp, Cc = feat.shape[0], feat.shape[1] * feat.shape[2], feat.shape[3]
    L.call("serl_sle_fwd", _p(feat), _p(kernel), _p(keep_mask), float(keep), out, N, Pp, Cc, kernel.shape[-1], ld_out, _s())


def sle_bwd_kernel_grad(ws, feat, dout, ld_dout, dkernel):
    N, Pp, Cc = feat.shape[0], feat.shape[1] * feat.shape[2], feat.shape[3]
    L.call("serl_sle_bwd_kernel_grad", _p(feat), dout, dkernel, ws.buf.data_ptr(), ws.nbytes, N, Pp, Cc, 8, ld_dout, _s())


def ln_tanh_fwd(z, ld_z, scale, bias, rows_per_group, group_stride, out, ld_out, xhat, rstd, R, D, eps=1e-6):
    L.call("serl_layernorm_tanh_fwd", z, ld_z, scale, bias, rows_per_group, group_stride, out, ld_out, xhat, rstd, R, D,
           float(eps), _s())


def ln_tanh_bwd(dt, ld_dt, t, ld_t, xhat, rstd, scale, rows_per_group, group_stride, dz, dy, dscale, dbias, R, D):
    L.call("serl_layernorm_tanh_bwd", dt, ld_dt, t, ld_t, xhat, rstd, scale, rows_per_group, group_stride, dz, dy, dscale,
           dbias, R, D, _s())


def ln_relu_fwd(z, ld_z, keep_mask, keep, scale, bias, out, ld_out, xhat, rstd, R, D, eps=1e-6):
    """Dense output z -> [dropout] -> LayerNorm -> ReLU (reward classifier hidden layer); addresses, keep_mask may be None."""
    L.call("serl_layernorm_relu_fwd", z, ld_z, keep_mask, float(keep), scale, bias, out, ld_out, xhat, rstd, R, D, float(eps), _s())


def ln_relu_bwd(dt, ld_dt, dlogit, head_w, xhat, rstd, scale, bias, keep_mask, keep, dz, dy, R, D):
    L.call("serl_layernorm_relu_bwd", dt, ld_dt, dlogit, head_w, xhat, rstd, scale, bias, keep_mask, float(keep), dz, dy, R, D, _s())


def dropout_bwd(x, keep_mask, keep, n):
    L.call("serl_dropout_bwd", x, keep_mask, float(keep), int(n), _s())


def bce_logits_loss(logits, eval_logits, labels, B, grad_scale, dlogit, info):
    L.call("serl_bce_logits_loss", logits, eval_logits, labels, B, float(grad_scale), dlogit, info, _s())


def ln_param_grad(dy, xhat, dscale, dbias, rows_per_group, R, D):
    L.call("serl_layernorm_param_grad", dy, xhat, dscale, dbias, rows_per_group, R, D, _s())


def colsum(x, out, groups, rows, D, ld, accumulate=False):
    L.call("serl_colsum_f32", x, out, groups, rows, D, ld, int(accumulate), _s())


def copy2d(src, ld_src, dst, ld_dst, R, D):
    L.call("serl_copy2d_f32", src, ld_src, dst, ld_dst, R, D, _s())


def fill(x, v, n):
    L.call("serl_fill_f32", x, float(v), n, _s())


# ---- rng ---------------------------------------------------------------------------------------------
def rng_schedule(rng_state, keys, do_aug, do_update):
    L.call("serl_rng_schedule", _p(_chk(rng_state, torch.uint32, "rng")), _p(keys), int(do_aug), int(do_update), _s())


def key_ptr(keys: torch.Tensor, slot: int) -> int:
    return keys.data_ptr() + 8 * slot


def normal_fill(key_addr, out, n):
    L.call("serl_normal_fill", key_addr, _p(out), n, _s())


def dropout_mask_fill(key_addr, fold, keep, mask, n):
    L.call("serl_dropout_mask_fill", key_addr, fold, float(keep), _p(mask), n, _s())


def subsample_idx(key_addr, ensemble, out, n):
    L.call("serl_subsample_idx", key_addr, ensemble, _p(out), int(n), _s())


def counter_add(counter, inc=1):
    L.call("serl_counter_add", _p(counter), inc, _s())


# ---- losses / optimizer ------------------------------------------------------------------------------
def tanh_gaussian_fwd(mu, log_std, eps, std_min, std_max, act, ld_act, logp, u, std, B, A, deterministic=False):
    L.call("serl_tanh_gaussian_fwd", _p(mu), _p(log_std), _p(eps), float(std_min), float(std_max), act, ld_act, _p(logp),
           _p(u), _p(std), B, A, int(deterministic), _s())


def critic_loss(q, q_next, sub, n_sub, rewards, masks, logp_next, lagrange, backup_entropy, gamma, grad_scale, target_q,
                dq, info, E, B):
    L.call("serl_critic_loss", _p(q), _p(q_next), _p(sub), n_sub, _p(rewards), _p(masks), _p(logp_next), lagrange,
           int(backup_entropy), float(gamma), float(grad_scale), _p(target_q), _p(dq), info, E, B, _s())


def actor_loss(q, logp, lagrange, da, ld_da, act, ld_act, std, log_std, eps, std_min, std_max, grad_scale, dmu, dlogstd,
               info, E, B, A):
    L.call("serl_actor_loss", _p(q), _p(logp), lagrange, da, ld_da, act, ld_act, _p(std), _p(log_std), _p(eps),
           float(std_min), float(std_max), float(grad_scale), _p(dmu), _p(dlogstd), info, E, B, A, _s())


def temperature_loss(logp, lagrange, target_entropy, grad_scale, dlagrange, info, B):
    L.call("serl_temperature_loss", _p(logp), lagrange, float(target_entropy), float(grad_scale), dlagrange, info, B, _s())


def adam_polyak(params, target, m, v, grad, seg_end: Sequence[int], live: Sequence[int], counts, lr, warmup, tau, polyak,
                lr_out=None, b1=0.9, b2=0.999, eps=1e-8, n=None, gap=0, aux=(0, 0, 0)):
    """aux = (aux_lo, aux_hi, aux_off): leaves with a second (actor-tx) Adam state at flat index i + aux_off."""
    d = L.AdamDesc()
    d.params, d.target, d.m, d.v, d.grad = _p(params), _p(target), _p(m), _p(v), _p(grad)
    d.n = params.numel() if n is None else int(n)
    d.gap, d.aux_lo, d.aux_hi, d.aux_off = int(gap), int(aux[0]), int(aux[1]), int(aux[2])
    for g in range(3):
        d.seg_end[g], d.live[g], d.lr[g], d.warmup[g] = int(seg_end[g]), int(live[g]), float(lr[g]), int(warmup[g])
    d.counts = _p(counts)
    d.b1, d.b2, d.eps, d.tau, d.polyak = b1, b2, eps, float(tau), int(polyak)
    d.lr_out = _p(lr_out)
    L.call("serl_adam_polyak", C.byref(d), _s())


# ---- single-pass TF32 GEMM with TMA-fed operands and fused epilogues (heads of the 16-bit builds) -------------------
def tgemm_problem(A, B, *, sAm, sAk, sBk, sBn, Z=1, sAz=0, sBz=0, C_=None, sCz=0, ldc=0, bias=None, sBiasZ=0, ln_scale=None,
                  ln_bias=None, sLnZ=0, xhat=None, rstd=None, sXhatZ=0, sRstdZ=0, head_w=None, head_b=None, sHeadWz=0, sHeadBz=0,
                  head_out=None, sHeadOutZ=0, ld_head=1, head_w2=None, head_b2=None, head_out2=None, noise=None, act=None, ld_act=0,
                  logp=None, u_out=None, std_out=None, keep_mask=None, keep=1.0):
    """One problem of a serl_tgemm_tf32 launch; every operand is a device ADDRESS (int) or None, strides in floats."""
    p = L.TgemmProblem()
    p.A, p.B, p.sAz, p.sAm, p.sAk, p.sBz, p.sBk, p.sBn, p.Z = A, B, sAz, sAm, sAk, sBz, sBk, sBn, Z
    p.C, p.sCz, p.ldc, p.bias, p.sBiasZ = C_, sCz, ldc, bias, sBiasZ
    p.ln_scale, p.ln_bias, p.sLnZ, p.xhat, p.rstd, p.sXhatZ, p.sRstdZ = ln_scale, ln_bias, sLnZ, xhat, rstd, sXhatZ, sRstdZ
    p.head_w, p.head_b, p.sHeadWz, p.sHeadBz, p.head_out, p.sHeadOutZ, p.ld_head = head_w, head_b, sHeadWz, sHeadBz, head_out, sHeadOutZ, ld_head
    p.head_w2, p.head_b2, p.head_out2 = head_w2, head_b2, head_out2
    p.noise, p.act, p.ld_act, p.logp, p.u_out, p.std_out = noise, act, ld_act, logp, u_out, std_out
    p.keep_mask, p.keep = keep_mask, float(keep)
    return p


def tgemm(ws: Optional[Workspace], problems, M, N, K, *, epilogue=L.TGEMM_STORE, head_n=0, accumulate=False, reduce_z=False, splits=0,
          ln_eps=1e-6, std_min=1e-5, std_max=5.0, deterministic=False, error=None):
    """C[z] = A[z] @ B[z] on the tensor cores (TF32, fp32 accumulate) for up to 6 problems of one shape; see include/serl_b200.h."""
    arr = (L.TgemmProblem * len(problems))(*problems)
    d = L.TgemmDesc()
    d.problems, d.num_problems, d.M, d.N, d.K = arr, len(problems), M, N, K
    d.epilogue, d.head_n, d.accumulate, d.reduce_z, d.splits = epilogue, head_n, int(accumulate), int(reduce_z), splits
    d.ln_eps, d.std_min, d.std_max, d.deterministic = float(ln_eps), float(std_min), float(std_max), int(deterministic)
    if ws is not None:
        d.workspace, d.workspace_bytes = ws.buf.data_ptr(), ws.nbytes
    d.error = _p(error)
    L.call("serl_tgemm_tf32", C.byref(d), _s())


def tgemm_splits(K: int, want: int) -> int:
    """Largest S <= want such that S k-splits of whole 32-wide k-blocks cover K with no empty split."""
    for S in range(max(want, 1), 0, -1):
        kc = -(-(-(-K // S)) // 32) * 32
        if -(-K // kc) == S:
            return S
    return 1


def sle_fwd_multi(problems, keep, N, P, C_):
    """problems: (feat, kernel, keep_mask | None, out, ld_out) device addresses; one launch."""
    arr = (L.SleProblem * len(problems))()
    for q, (feat, kern, mask, out, ld) in zip(arr, problems):
        q.feat, q.kernel, q.keep_mask, q.out, q.ld_out = feat, kern, mask, out, ld
    L.call("serl_sle_fwd_multi", arr, len(problems), float(keep), N, P, C_, 8, _s())


def sle_bwd_multi(ws: Workspace, problems, N, P, C_):
    """problems: (feat, dout, ld_dout, dkernel) device addresses; SLE kernel gradients of all cameras in two launches."""
    arr = (L.SleBwdProblem * len(problems))()
    for q, (feat, dout, ld, dk) in zip(arr, problems):
        q.feat, q.dout, q.ld_dout, q.dkernel = feat, dout, ld, dk
    L.call("serl_sle_bwd_multi", arr, len(problems), ws.buf.data_ptr(), ws.nbytes, N, P, C_, 8, _s())


def enc_finish(problems, rows, eps=1e-6):
    """problems: dicts with partials+S or x+ld_x+w+K, and bias, ln_scale, ln_bias, out, ld_out, D, optional xhat, rstd."""
    arr = (L.EncFinishProblem * len(problems))()
    for q, p in zip(arr, problems):
        q.partials, q.S, q.x, q.ld_x, q.w, q.K = p.get("partials"), p.get("S", 0), p.get("x"), p.get("ld_x", 0), p.get("w"), p.get("K", 0)
        q.bias, q.ln_scale, q.ln_bias, q.out, q.ld_out = p["bias"], p["ln_scale"], p["ln_bias"], p["out"], p["ld_out"]
        q.xhat, q.rstd, q.D = p.get("xhat"), p.get("rstd"), p["D"]
    L.call("serl_enc_finish", arr, len(problems), rows, float(eps), _s())


def ln_tanh_bwd_multi(problems):
    """problems: dicts with dt+ld_dt (or dq+head_w[+head_w_stride]), optional dt2+ld_dt2, t, ld_t, xhat, rstd, scale,
    rows_per_group, group_stride, dz, optional dy, R, D."""
    arr = (L.LnBwdProblem * len(problems))()
    for q, p in zip(arr, problems):
        q.dt, q.ld_dt, q.dt2, q.ld_dt2 = p.get("dt"), p.get("ld_dt", 0), p.get("dt2"), p.get("ld_dt2", 0)
        q.dq, q.head_w, q.head_w_stride = p.get("dq"), p.get("head_w"), p.get("head_w_stride", 0)
        q.t, q.ld_t, q.xhat, q.rstd, q.scale = p["t"], p["ld_t"], p["xhat"], p["rstd"], p["scale"]
        q.rows_per_group, q.group_stride, q.dz, q.dy, q.R, q.D = p["rows_per_group"], p.get("group_stride", 0), p["dz"], p.get("dy"), p["R"], p["D"]
        q.dt_parts, q.dt_part_stride = p.get("dt_parts", 1), p.get("dt_part_stride", 0)
    L.call("serl_layernorm_tanh_bwd_multi", arr, len(problems), _s())


def small_grads(jobs):
    """jobs: (kind, x, ld_x, y | None, ld_y, out_a, out_b | None, groups, rows, D)."""
    arr = (L.SmallGradJob * len(jobs))()
    for q, (kind, x, ld_x, y, ld_y, out_a, out_b, groups, rows, D) in zip(arr, jobs):
        q.kind, q.x, q.ld_x, q.y, q.ld_y, q.out_a, q.out_b, q.groups, q.rows, q.D = kind, x, ld_x, y, ld_y, out_a, out_b, groups, rows, D
    L.call("serl_small_grads", arr, len(jobs), _s())
