"""ctypes binding of libserl_b200.so (the C-ABI declared in include/serl_b200.h).

There is NO fallback: if the library is missing or a call fails, this raises.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "lib", "libserl_b200.so")
MAX_CAMS = 4
ABI_VERSION = 4

(KEY_CROP_OBS, KEY_CROP_NEXT, KEY_CRITIC_NEXT, KEY_CRITIC_SUBSAMPLE, KEY_ACTOR_DROPOUT, KEY_ACTOR_SAMPLE,
 KEY_TEMP_NEXT) = range(7)
NUM_KEYS = 8
FMT_BF16, FMT_FP16 = 0, 1

vp, i32, i64, u32, u64, f32 = C.c_void_p, C.c_int32, C.c_int64, C.c_uint32, C.c_uint64, C.c_float


class ReplayView(C.Structure):
    _fields_ = [("frames", vp * MAX_CAMS), ("state", vp), ("next_state", vp), ("actions", vp), ("rewards", vp),
                ("masks", vp), ("dones", vp), ("valid", vp),
                ("num_cams", i32), ("height", i32), ("width", i32), ("channels", i32), ("num_stack", i32),
                ("state_dim", i32), ("action_dim", i32), ("capacity", i32), ("size", i32)]


class SampleRequest(C.Structure):
    _fields_ = [("seed", u64), ("step", u64), ("step_dev", vp), ("size_dev", vp), ("lane_offset", u32), ("batch", i32), ("explicit_idx", vp),
                ("key_obs", vp), ("key_next", vp), ("explicit_off_obs", vp), ("explicit_off_next", vp),
                ("crop_total", i32), ("out_row_offset", i32), ("padding", i32)]


class BatchOut(C.Structure):
    _fields_ = [("obs_pix", vp * MAX_CAMS), ("next_pix", vp * MAX_CAMS), ("obs_state", vp), ("next_state", vp),
                ("actions", vp), ("rewards", vp), ("masks", vp), ("dones", vp), ("idx", vp), ("off_obs", vp),
                ("off_next", vp), ("status", vp)]


class ScatterRequest(C.Structure):
    _fields_ = [("n", i32), ("dst_slot", vp), ("src_slot", vp), ("frames", vp * MAX_CAMS), ("state", vp),
                ("next_state", vp), ("actions", vp), ("rewards", vp), ("masks", vp), ("dones", vp), ("valid", vp),
                ("row_stride", i64)]


class GemmDesc(C.Structure):
    _fields_ = [("A", vp), ("B", vp), ("C", vp), ("bias", vp), ("workspace", vp), ("workspace_bytes", C.c_size_t),
                ("M", i32), ("N", i32), ("K", i32), ("Z", i32),
                ("sAz", i64), ("sAm", i64), ("sAk", i64), ("sBz", i64), ("sBk", i64), ("sBn", i64), ("sCz", i64),
                ("sBiasZ", i64), ("ldc", i32), ("accumulate", i32), ("reduce_z", i32)]


class TgemmProblem(C.Structure):
    _fields_ = [("A", vp), ("B", vp), ("sAz", i64), ("sAm", i64), ("sAk", i64), ("sBz", i64), ("sBk", i64), ("sBn", i64), ("Z", i32),
                ("C", vp), ("sCz", i64), ("ldc", i32), ("bias", vp), ("sBiasZ", i64), ("ln_scale", vp), ("ln_bias", vp), ("sLnZ", i64),
                ("xhat", vp), ("rstd", vp), ("sXhatZ", i64), ("sRstdZ", i64), ("head_w", vp), ("head_b", vp), ("sHeadWz", i64),
                ("sHeadBz", i64), ("head_out", vp), ("sHeadOutZ", i64), ("ld_head", i32), ("head_w2", vp), ("head_b2", vp),
                ("head_out2", vp), ("noise", vp), ("act", vp), ("ld_act", i32), ("logp", vp), ("u_out", vp), ("std_out", vp),
                ("keep_mask", vp), ("keep", f32)]


class TgemmDesc(C.Structure):
    _fields_ = [("problems", C.POINTER(TgemmProblem)), ("num_problems", i32), ("M", i32), ("N", i32), ("K", i32), ("epilogue", i32),
                ("head_n", i32), ("accumulate", i32), ("reduce_z", i32), ("splits", i32), ("ln_eps", f32), ("std_min", f32),
                ("std_max", f32), ("deterministic", i32), ("workspace", vp), ("workspace_bytes", C.c_size_t), ("error", vp)]


class SleProblem(C.Structure):
    _fields_ = [("feat", vp), ("kernel", vp), ("keep_mask", vp), ("out", vp), ("ld_out", i32)]


class SleBwdProblem(C.Structure):
    _fields_ = [("feat", vp), ("dout", vp), ("ld_dout", i32), ("dkernel", vp)]


class EncFinishProblem(C.Structure):
    _fields_ = [("partials", vp), ("S", i32), ("x", vp), ("ld_x", i32), ("w", vp), ("K", i32), ("bias", vp), ("ln_scale", vp), ("ln_bias", vp),
                ("out", vp), ("ld_out", i32), ("xhat", vp), ("rstd", vp), ("D", i32)]


class LnBwdProblem(C.Structure):
    _fields_ = [("dt", vp), ("ld_dt", i32), ("dt2", vp), ("ld_dt2", i32), ("dq", vp), ("head_w", vp), ("head_w_stride", i64),
                ("t", vp), ("ld_t", i32), ("xhat", vp), ("rstd", vp), ("scale", vp), ("rows_per_group", i32), ("group_stride", i64),
                ("dz", vp), ("dy", vp), ("R", i32), ("D", i32), ("dt_parts", i32), ("dt_part_stride", i64)]


class SmallGradJob(C.Structure):
    _fields_ = [("kind", i32), ("x", vp), ("ld_x", i64), ("y", vp), ("ld_y", i64), ("out_a", vp), ("out_b", vp), ("groups", i32),
                ("rows", i32), ("D", i32)]


SMALL_GRAD_COLSUM, SMALL_GRAD_LN, SMALL_GRAD_HEAD = range(3)
TGEMM_STORE, TGEMM_LN_TANH, TGEMM_LN_TANH_HEAD, TGEMM_LN_TANH_POLICY, TGEMM_PARTIAL, TGEMM_LN_RELU_HEAD = range(6)
TGEMM_MAX_PROBLEMS = 6


class ConvTcDesc(C.Structure):
    _fields_ = [("x", vp), ("w", vp), ("y", vp), ("stats", vp), ("in_a", vp), ("in_b", vp), ("error", vp),
                ("N", i32), ("Hi", i32), ("Wi", i32), ("Ci", i32), ("Ho", i32), ("Wo", i32), ("Co", i32), ("kh", i32),
                ("kw", i32), ("stride", i32), ("pad_lo", i32), ("stem", i32), ("fmt", i32)]


class StemPoolDesc(C.Structure):
    _fields_ = [("xs", vp), ("w", vp), ("pooled", vp), ("side", vp), ("stats", vp), ("error", vp), ("neg_mask", C.c_uint64),
                ("N", i32), ("fmt", i32)]


class Conv3x3ResDesc(C.Structure):
    _fields_ = [("x", vp), ("w", vp), ("y", vp), ("out_f32", vp), ("res", vp), ("gamma", vp), ("beta", vp), ("res_stats", vp),
                ("res_gamma", vp), ("res_beta", vp), ("error", vp), ("N", i32), ("H", i32), ("W", i32), ("Ci", i32), ("Co", i32),
                ("relu", i32), ("fmt", i32), ("eps", f32)]


class Conv3x3S2ResDesc(C.Structure):
    _fields_ = [("x", vp), ("w", vp), ("w_proj", vp), ("y", vp), ("r", vp), ("gamma", vp), ("beta", vp), ("gamma_proj", vp),
                ("beta_proj", vp), ("error", vp), ("N", i32), ("Wo", i32), ("Ci", i32), ("Co", i32), ("fmt", i32), ("eps", f32)]


class AdamDesc(C.Structure):
    _fields_ = [("params", vp), ("target", vp), ("m", vp), ("v", vp), ("grad", vp), ("n", i32), ("seg_end", i32 * 3),
                ("live", i32 * 3), ("counts", vp), ("lr", f32 * 3), ("warmup", i32 * 3), ("b1", f32), ("b2", f32),
                ("eps", f32), ("tau", f32), ("polyak", i32), ("lr_out", vp), ("gap", i32), ("aux_lo", i32),
                ("aux_hi", i32), ("aux_off", i32)]


_PROTOS = {
    "serl_replay_sample_crop": [C.POINTER(ReplayView), C.POINTER(SampleRequest), C.POINTER(BatchOut), vp],
    "serl_replay_scatter": [C.POINTER(ReplayView), C.POINTER(ScatterRequest), vp],
    "serl_replay_set_valid": [vp, vp, vp, C.c_int, vp],
    "serl_replay_commit": [vp, vp, vp, C.c_int, vp, C.c_int, vp],
    "serl_counter_add": [vp, u64, vp],
    "serl_set_pdl": [C.c_int],
    "serl_rng_schedule": [vp, vp, C.c_int, C.c_int, vp],
    "serl_normal_fill": [vp, vp, C.c_int, vp],
    "serl_dropout_mask_fill": [vp, u32, f32, vp, C.c_int, vp],
    "serl_subsample_idx": [vp, C.c_int, vp, C.c_int, vp],
    "serl_host_rng_schedule": [vp, vp, C.c_int, C.c_int],
    "serl_host_crop_offsets": [vp, C.c_int, C.c_int, vp],
    "serl_host_draw_indices": [u64, u64, u32, C.c_int, C.c_int, vp, vp],
    "serl_host_threefry_split": [vp, C.c_int, vp],
    "serl_host_random_bits": [vp, C.c_int, vp],
    "serl_conv2d_nhwc_f32": [vp, C.c_int, vp, vp] + [C.c_int] * 10 + [vp],
    "serl_groupnorm_nhwc_f32": [vp, vp, vp, vp, vp, C.c_int, C.c_int, C.c_int, C.c_int, f32, C.c_int, vp],
    "serl_maxpool3x3s2_nhwc_f32": [vp, vp, C.c_int, C.c_int, C.c_int, C.c_int, vp],
    "serl_trunk_stem_prep_h16": [vp, vp, C.c_int, C.c_int, C.c_int, C.c_int, vp],
    "serl_conv2d_tc_h16": [C.POINTER(ConvTcDesc), vp],
    "serl_conv3x3s1_tc_h16": [C.POINTER(ConvTcDesc), C.c_int, vp],
    "serl_conv3x3_res_h16": [C.POINTER(Conv3x3ResDesc), vp],
    "serl_conv3x3s2_res_h16": [C.POINTER(Conv3x3S2ResDesc), vp],
    "serl_gn_finalize": [vp, vp, vp, vp, vp, C.c_int, C.c_int, C.c_int, f32, vp],
    "serl_affine_relu_h16": [vp, vp, vp, C.c_int, C.c_int, C.c_int, C.c_int, vp],
    "serl_stem_conv_pool_tc_h16": [C.POINTER(StemPoolDesc), vp],
    "serl_pool_finish_h16": [vp, vp, vp, vp, vp, C.c_int, C.c_int, vp],
    "serl_pool_finish_gn_h16": [vp, vp, vp, vp, vp, vp, C.c_int, C.c_float, C.c_int, vp],
    "serl_affine_relu_gn_h16": [vp, vp, vp, vp, C.c_int, C.c_int, C.c_int, C.c_float, C.c_int, vp],
    "serl_block_combine_gn_h16": [vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, C.c_int, C.c_int, C.c_int, C.c_float, C.c_int, vp],
    "serl_maxpool_affine_h16": [vp, vp, vp, vp, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, vp],
    "serl_block_combine_h16": [vp, vp, vp, vp, vp, vp, vp, vp, C.c_int, C.c_int, C.c_int, C.c_int, vp],
    "serl_gemm_f32": [C.POINTER(GemmDesc), vp],
    "serl_gemm_tf32x3": [C.POINTER(GemmDesc), vp],
    "serl_tgemm_tf32": [C.POINTER(TgemmDesc), vp],
    "serl_sle_fwd_multi": [C.POINTER(SleProblem), C.c_int, f32, C.c_int, C.c_int, C.c_int, C.c_int, vp],
    "serl_sle_bwd_multi": [C.POINTER(SleBwdProblem), C.c_int, vp, C.c_size_t, C.c_int, C.c_int, C.c_int, C.c_int, vp],
    "serl_enc_finish": [C.POINTER(EncFinishProblem), C.c_int, C.c_int, f32, vp],
    "serl_layernorm_tanh_bwd_multi": [C.POINTER(LnBwdProblem), C.c_int, vp],
    "serl_small_grads": [C.POINTER(SmallGradJob), C.c_int, vp],
    "serl_sle_fwd": [vp, vp, vp, f32, vp, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, vp],
    "serl_sle_bwd_kernel_grad": [vp, vp, vp, vp, C.c_size_t, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, vp],
    "serl_layernorm_tanh_fwd": [vp, C.c_int, vp, vp, C.c_int, C.c_int, vp, C.c_int, vp, vp, C.c_int, C.c_int, f32, vp],
    "serl_layernorm_tanh_bwd": [vp, C.c_int, vp, C.c_int, vp, vp, vp, C.c_int, C.c_int, vp, vp, vp, vp, C.c_int, C.c_int, vp],
    "serl_layernorm_param_grad": [vp, vp, vp, vp, C.c_int, C.c_int, C.c_int, vp],
    "serl_layernorm_relu_fwd": [vp, C.c_int, vp, f32, vp, vp, vp, C.c_int, vp, vp, C.c_int, C.c_int, f32, vp],
    "serl_layernorm_relu_bwd": [vp, C.c_int, vp, vp, vp, vp, vp, vp, vp, f32, vp, vp, C.c_int, C.c_int, vp],
    "serl_colsum_f32": [vp, vp, C.c_int, C.c_int, C.c_int, C.c_longlong, C.c_int, vp],
    "serl_copy2d_f32": [vp, C.c_longlong, vp, C.c_longlong, C.c_int, C.c_int, vp],
    "serl_fill_f32": [vp, f32, C.c_int, vp],
    "serl_tanh_gaussian_fwd": [vp, vp, vp, f32, f32, vp, C.c_int, vp, vp, vp, C.c_int, C.c_int, C.c_int, vp],
    "serl_critic_loss": [vp, vp, vp, C.c_int, vp, vp, vp, vp, C.c_int, f32, f32, vp, vp, vp, C.c_int, C.c_int, vp],
    "serl_actor_loss": [vp, vp, vp, vp, C.c_int, vp, C.c_int, vp, vp, vp, f32, f32, f32, vp, vp, vp, C.c_int, C.c_int,
                        C.c_int, vp],
    "serl_tanh_fwd": [vp, vp, C.c_int, vp],
    "serl_tanh_bwd": [vp, vp, vp, C.c_int, vp],
    "serl_bc_loss": [vp, vp, vp, f32, f32, f32, vp, vp, vp, C.c_int, C.c_int, vp],
    "serl_temperature_loss": [vp, vp, f32, f32, vp, vp, C.c_int, vp],
    "serl_dropout_bwd": [vp, vp, f32, C.c_longlong, vp],
    "serl_bce_logits_loss": [vp, vp, vp, C.c_int, f32, vp, vp, vp],
    "serl_adam_polyak": [C.POINTER(AdamDesc), vp],
}
EXPORTS = sorted(list(_PROTOS) + ["serl_last_error", "serl_version", "serl_device_sm_count", "serl_launch_count", "serl_stem_v2_active", "serl_balanced_grid"])

_lib = None


class SerlError(RuntimeError):
    pass


def load():
    """Loads the shared library; raises (no CPU fallback) if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise SerlError(f"{LIB_PATH} not found - run `python -m serl_b200.build` (or __graft_entry__.build()). "
                        "serl_b200 has no fallback path.")
    lib = C.CDLL(LIB_PATH)
    lib.serl_last_error.restype = C.c_char_p
    lib.serl_last_error.argtypes = []
    lib.serl_version.restype = C.c_int
    lib.serl_launch_count.restype = C.c_ulonglong
    lib.serl_launch_count.argtypes = []
    lib.serl_device_sm_count.argtypes = [C.c_int]
    for name, args in _PROTOS.items():
        fn = getattr(lib, name)
        fn.argtypes = args
        fn.restype = C.c_int
    if lib.serl_version() != ABI_VERSION:
        raise SerlError(f"libserl_b200 ABI {lib.serl_version()} != binding {ABI_VERSION}; rebuild")
    _lib = lib
    return lib


def call(name: str, *args):
    lib = load()
    rc = getattr(lib, name)(*args)
    if rc != 0:
        raise SerlError(f"{name} failed ({rc}): {lib.serl_last_error().decode()}")
    return rc


def launch_count() -> int:
    """Kernels libserl_b200 has enqueued in this process so far (launches recorded into a CUDA graph count once, at capture)."""
    return int(load().serl_launch_count())


# ---- torch plumbing indirections (device memory / streams / events); tests may patch these for dry runs -------
def require_cuda(device):
    if device.type != "cuda":
        raise SerlError("serl_b200 runs on a CUDA device only (HBM-resident replay and sm_100a kernels; no CPU fallback)")


_stream_objs = {}


def _raw_stream():
    """Raw cudaStream_t of the CURRENT stream.  torch.cuda.current_stream() costs ~15 us of Python per call, which is real
    time in a loop that synchronises every step; the C getter is ~0.3 us."""
    import torch
    get = getattr(torch._C, "_cuda_getCurrentRawStream", None)
    if get is None:
        return torch.cuda.current_stream().cuda_stream
    return get(torch._C._cuda_getDevice())


def _stream_obj():
    import torch
    raw = _raw_stream()
    s = _stream_objs.get(raw)
    if s is None:
        s = _stream_objs[raw] = torch.cuda.current_stream()
    return s


def stream_ptr():
    return _raw_stream()


class _Event:
    def __init__(self):
        import torch
        self.e = torch.cuda.Event()

    def record(self):
        self.e.record(_stream_obj())

    def synchronize(self):
        self.e.synchronize()

    def make_current_stream_wait(self):
        _stream_obj().wait_event(self.e)


def new_event():
    return _Event()


class _Side:
    """A side stream with fork / join against the CURRENT stream (works eagerly and under CUDA-graph capture, where the
    event dependencies become fork / join edges of the captured graph).  Entering it makes it the current stream."""

    def __init__(self, device, priority: int = 0):
        import torch
        self.s = torch.cuda.Stream(device, priority=priority)
        self._ctx = None

    def fork(self):                 # side stream waits for everything enqueued on the current stream so far
        import torch
        e = torch.cuda.Event()
        e.record()
        self.s.wait_event(e)

    def join(self):                 # current stream waits for everything enqueued on the side stream so far
        import torch
        e = torch.cuda.Event()
        e.record(self.s)
        torch.cuda.current_stream().wait_event(e)

    def __enter__(self):
        import torch
        self._ctx = torch.cuda.stream(self.s)
        self._ctx.__enter__()
        return self

    def __exit__(self, *a):
        ctx, self._ctx = self._ctx, None
        return ctx.__exit__(*a)


class _NoSide:
    """Serial stand-in (dry runs on a CPU device, or SERL_STREAMS=0): same call sites, everything stays on one stream."""

    def fork(self): pass
    def join(self): pass
    def __enter__(self): return self
    def __exit__(self, *a): return False


def new_side_stream(device, enabled=True, priority: int = 0):
    """priority < 0: a high-priority stream (its kernels' CTAs are placed before those of default-priority streams whenever an SM
    frees up; captured into CUDA-graph kernel nodes)."""
    return _Side(device, priority) if enabled and device.type == "cuda" else _NoSide()


def pin(t):
    return t.pin_memory()
