"""ctypes binding of the C-ABI library (include/keisei_b200.h).

There is NO CPU fallback: if ``libkeisei_b200.so`` is missing or a CUDA device is not available the
product path raises.  torch is used for device memory and streams only."""
from __future__ import annotations

import ctypes as C
import os
from typing import Optional

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("KZ_LIB_PATH") or os.path.join(_HERE, "libkeisei_b200.so")  # override: kernel tuning only

NUM_ACTIONS = 13527
OBS_FLOATS = 46 * 81
MASK_PAD_STRIDE = 13536
BITMAP_WORDS = 448
REASONS = {0: None, 1: "Tsumi", 2: "stalemate", 3: "Max moves reached", 4: "Sennichite"}
TSUMI = 1  # KZ_TSUMI
ERR_KING_CAPTURE = 4  # KZ_ERR_KING_CAPTURE

EXPORTS = [
    "kz_abi_version", "kz_last_cuda_error", "kz_build_info", "kz_init_tables", "kz_state_layout", "kz_reset", "kz_load_positions",
    "kz_export_positions", "kz_piece_targets", "kz_refresh", "kz_step", "kz_legal_mask", "kz_observe", "kz_errors", "kz_sample_masked",
    "kz_gae", "kz_gae_exact", "kz_eval_masked_fwd", "kz_eval_masked_bwd", "kz_obs_conv_fwd", "kz_obs_conv_wgrad_ctas",
    "kz_obs_conv_wgrad", "kz_ppo_loss", "kz_eval_masked_bwd_bias", "kz_adam_clip_workspace", "kz_adam_clip_step",
    "kz_step_rollout", "kz_legal_bitmap", "kz_bitmap_expand", "kz_sample_bitmap",
    "kz_eval_bitmap_fwd", "kz_eval_bitmap_bwd", "kz_step_range", "kz_cobs_conv_fwd", "kz_cobs_conv_wgrad_ctas",
    "kz_cobs_conv_wgrad", "kz_heuristic_actions", "kz_pool_records", "kz_step_pool", "kz_reset_pool", "kz_legal_list",
    "kz_expand", "kz_check_bitmap",
]
COBS_WORDS = 40
POOL_RECORD_WORDS = 512
ABI_VERSION = 3


class NativeError(RuntimeError):
    pass


_lib: Optional[C.CDLL] = None
_tables_ready = set()


def lib() -> C.CDLL:
    """Load the shared library (never builds implicitly on a GPU box: the .so ships in-tree)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise NativeError(
            f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(nvcc, sm_100a).  shogidrl_b200 has no CPU fallback.")
    L = C.CDLL(LIB_PATH)
    vp, i32, i64, u64, u32, f32, f64 = C.c_void_p, C.c_int, C.c_int64, C.c_uint64, C.c_uint32, C.c_float, C.c_double
    L.kz_abi_version.restype = i32
    L.kz_last_cuda_error.restype = C.c_char_p
    L.kz_build_info.restype = C.c_char_p
    L.kz_init_tables.argtypes = [vp]
    L.kz_state_layout.argtypes = [i32, i32, C.POINTER(i64), C.POINTER(i64)]
    L.kz_reset.argtypes = [vp, i32, i32, vp, i32, vp]
    L.kz_load_positions.argtypes = [vp, i32, i32, vp, vp, vp, vp, vp, vp]
    L.kz_export_positions.argtypes = [vp, i32, i32, vp, vp, vp, vp]
    L.kz_refresh.argtypes = [vp, i32, i32, vp, i64, vp, i64, vp, vp, i32, u64, u32, u32, i32, vp, vp]
    L.kz_step.argtypes = [vp, i32, i32, vp, i32, vp, i64, vp, i64, vp, vp, vp, vp, vp, vp, vp, u64, u32, u32, i32, vp]
    L.kz_step_rollout.argtypes = [vp, i32, i32, vp, i32, vp, i64, vp, i64, vp, vp, vp, vp, vp, vp, vp, vp, u64, u32, u32, i32, vp]
    L.kz_step_range.argtypes = [vp, i32, i32, i32, i32, i32, vp, i32, vp, i64, vp, i64, vp, i64, vp, vp, vp, vp, vp, vp, vp, vp,
                                u64, u32, u32, i32, vp]
    L.kz_legal_bitmap.argtypes = [vp, i32, i32, vp, i64, vp, i64, vp, vp, vp]
    L.kz_cobs_conv_fwd.argtypes = [vp, vp, vp, vp, i32, i32, i32, vp, vp]
    L.kz_cobs_conv_wgrad_ctas.argtypes = [i32]
    L.kz_cobs_conv_wgrad.argtypes = [vp, vp, vp, vp, i32, i32, i32, vp, i32, vp, vp, vp]
    L.kz_bitmap_expand.argtypes = [vp, i64, vp, i32, vp, i64, vp]
    L.kz_sample_bitmap.argtypes = [vp, i32, i64, vp, i64, i32, u64, u64, vp, vp, i32, vp, vp, i32, vp]
    L.kz_eval_bitmap_fwd.argtypes = [vp, i32, i64, vp, i64, vp, vp, i32, vp, vp, vp, vp]
    L.kz_eval_bitmap_bwd.argtypes = [vp, i32, i64, vp, i64, vp, vp, i32, vp, vp, vp, vp, i64, vp, vp]
    L.kz_heuristic_actions.argtypes = [vp, i32, i32, vp, i64, vp, i64, vp, i32, vp, vp, u64, u32, u32, vp]
    L.kz_pool_records.argtypes = [vp, i32, i32, vp, i64, vp, vp, vp, vp]
    L.kz_step_pool.argtypes = [vp, i32, i32, i32, i32, i32, vp, i32, vp, i64, vp, i64, vp, i64, vp, vp, vp, vp, vp, vp, vp, vp,
                               u64, u32, u32, vp, i32, vp, u64, vp, vp]
    L.kz_reset_pool.argtypes = [vp, i32, i32, vp, i32, vp, i32, vp, u64, u32, vp, vp]
    L.kz_legal_list.argtypes = [vp, i64, i32, vp, vp, vp, i32, vp]
    L.kz_expand.argtypes = [vp, i32, i32, i32, vp, vp, i32, i32, vp, i64, vp, i64, vp, vp, vp, vp, vp, vp, vp, vp, vp, i32, vp]
    L.kz_check_bitmap.argtypes = [vp, i32, i32, vp, i64, vp, i64, vp, vp]
    L.kz_legal_mask.argtypes = [vp, i32, i32, vp, i64, vp, vp]
    L.kz_observe.argtypes = [vp, i32, i32, vp, i64, vp]
    L.kz_errors.argtypes = [vp, i32, i32, vp, i32, vp]
    L.kz_piece_targets.argtypes = [vp, i32, i32, vp, vp, vp]
    L.kz_sample_masked.argtypes = [vp, i32, i64, vp, i64, i32, u64, u64, vp, vp, i32, vp, vp, i32, vp]
    L.kz_gae.argtypes = [vp, vp, vp, vp, i32, i32, f32, f32, vp, vp, vp]
    L.kz_gae_exact.argtypes = [vp, vp, vp, vp, i32, i32, f32, f32, vp, vp, vp]
    L.kz_eval_masked_fwd.argtypes = [vp, i32, i64, vp, i64, vp, vp, i32, vp, vp, vp, vp]
    L.kz_eval_masked_bwd.argtypes = [vp, i32, i64, vp, i64, vp, vp, i32, vp, vp, vp, vp, i64, vp]
    L.kz_eval_masked_bwd_bias.argtypes = [vp, i32, i64, vp, i64, vp, vp, i32, vp, vp, vp, vp, i64, vp, vp]
    L.kz_adam_clip_workspace.argtypes = [i32, vp]
    L.kz_adam_clip_step.argtypes = [i32, vp, vp, vp, vp, vp, vp, f64, f64, f64, f64, f64, f64, vp, i64, vp, vp]
    L.kz_obs_conv_fwd.argtypes = [vp, vp, vp, vp, i32, i32, i32, vp, vp]
    L.kz_ppo_loss.argtypes = [vp, vp, vp, vp, vp, vp, i32, f32, f32, f32, f32, vp, vp, vp, vp, vp]
    L.kz_obs_conv_wgrad_ctas.argtypes = [i32]
    L.kz_obs_conv_wgrad.argtypes = [vp, vp, vp, vp, i32, i32, i32, vp, i32, vp, vp, vp]
    for name in EXPORTS:
        fn = getattr(L, name)
        if name not in ("kz_last_cuda_error", "kz_build_info"):
            fn.restype = i64 if name == "kz_adam_clip_workspace" else i32
    if L.kz_abi_version() != ABI_VERSION:
        raise NativeError(f"{LIB_PATH} has ABI version {L.kz_abi_version()}, this package binds version {ABI_VERSION}: "
                          "rebuild it (python -c 'import __graft_entry__ as g; g.build()')")
    _lib = L
    return L


def build_info() -> dict:
    """{"src_sha": hash of the sources the loaded library was built from, "built": ..., "src_sha_now": hash of the
    sources in the tree, "match": whether they agree, "lib": path}."""
    import re
    from . import _build
    m = re.match(r"src_sha=(\S+) built=(.*) arch=(\S+)", lib().kz_build_info().decode())
    info = {"src_sha": m.group(1), "built": m.group(2), "arch": m.group(3)} if m else {"src_sha": None}
    try:
        now = _build.source_sha()
    except OSError:
        now = None
    info.update(src_sha_now=now, match=(now == info.get("src_sha")), lib=LIB_PATH)
    return info


def check(rc: int, what: str) -> None:
    if rc != 0:
        msg = {-1: "invalid argument", -2: "CUDA error: " + (lib().kz_last_cuda_error() or b"").decode(),
               -3: "kz_init_tables has not run"}.get(rc, f"error {rc}")
        raise NativeError(f"{what} failed: {msg}")


def require(cond: bool, what: str) -> None:
    """Argument validation in front of the raw-pointer C ABI (kept under ``python -O``, unlike ``assert``)."""
    if not cond:
        raise ValueError(what)


def stream_ptr(device: torch.device) -> int:
    """torch's current stream on ``device`` -- the last argument of every launch.  The library launches on the CALLING
    THREAD's current CUDA device (one process per GPU with torch.cuda.set_device(local_rank) is the supported layout), so
    tensors on another device are refused here instead of failing inside the launch with "invalid resource handle"."""
    idx = device.index if device.index is not None else torch.cuda.current_device()
    if idx != torch.cuda.current_device():
        raise NativeError(f"tensors live on cuda:{idx} but the current CUDA device is cuda:{torch.cuda.current_device()}: call "
                          f"torch.cuda.set_device({idx}) (or wrap the call in `with torch.cuda.device({idx}):`) first")
    return torch.cuda.current_stream(device).cuda_stream


def require_cuda(device) -> torch.device:
    device = torch.device(device)
    if device.type != "cuda":
        raise NativeError(f"shogidrl_b200 runs on CUDA devices only (got {device}); there is no CPU fallback")
    if not torch.cuda.is_available():
        raise NativeError("no CUDA device is available; shogidrl_b200 has no CPU fallback")
    if device.index is None:
        device = torch.device("cuda", torch.cuda.current_device())
    return device


def init_tables(device: torch.device) -> None:
    """kz_init_tables once per device (ray / step tables, start-position bitmap)."""
    device = require_cuda(device)
    if device.index in _tables_ready:
        return
    with torch.cuda.device(device):
        check(lib().kz_init_tables(stream_ptr(device)), "kz_init_tables")
        torch.cuda.current_stream(device).synchronize()
    _tables_ready.add(device.index)


def ptr(t: Optional[torch.Tensor]) -> Optional[int]:
    return None if t is None else t.data_ptr()
