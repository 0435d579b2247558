"""CPU-only checks of the C-ABI library: it loads without a GPU and exports every symbol that
include/keisei_b200.h declares (no compute calls here)."""
import ctypes as C
import os
import re

import pytest

from shogidrl_b200 import _native as nv

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _declared():
    src = open(os.path.join(ROOT, "include", "keisei_b200.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(kz_[a-z0-9_]+)\s*\(", src)))


def test_header_symbols_exported():
    L = nv.lib()
    names = _declared()
    assert len(names) >= 14
    for n in names:
        assert hasattr(L, n), f"{n} declared in include/keisei_b200.h but not exported"
    assert sorted(nv.EXPORTS) == names


def test_abi_version_and_layout():
    L = nv.lib()
    assert L.kz_abi_version() == 3
    offs = (C.c_int64 * 3)()
    total = C.c_int64()
    assert L.kz_state_layout(65536, 500, offs, C.byref(total)) == 0
    assert offs[0] == 0 and offs[1] == 65536 * 96 and offs[2] % 256 == 0
    # boards + meta + 1024-slot repetition table of 16-byte slots: ~16.5 kB per game
    per_game = total.value / 65536
    assert 96 + 32 + 1024 * 16 <= per_game <= 96 + 32 + 1024 * 16 + 1
    assert L.kz_state_layout(0, 500, offs, C.byref(total)) == -1  # KZ_E_ARG


def test_no_cpu_fallback():
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    from shogidrl_b200 import VecShogiEnv, NativeError
    with pytest.raises(NativeError):
        VecShogiEnv(4)
    with pytest.raises(NativeError):
        VecShogiEnv(4, device="cpu")


def test_product_does_not_import_oracle():
    """The oracle is test infrastructure: nothing under shogidrl_b200/ may reference it."""
    pkg = os.path.join(ROOT, "shogidrl_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                txt = open(os.path.join(dirpath, f)).read()
                assert "oracle" not in txt.lower() or f == "_never_", (dirpath, f)


def test_output_storage_validation_rejects_short_or_misshapen_rows():
    """The C ABI sees raw pointers, so VecShogiEnv validates caller storage before every launch."""
    import types

    import pytest
    import torch

    from shogidrl_b200.vec_env import VecShogiEnv

    env = types.SimpleNamespace(device=torch.device("cpu"), n=4)
    rows = lambda t, what="obs", dt=(torch.float32,), k=3726: VecShogiEnv._rows_arg(env, t, what, dt, k)
    assert rows(None) == (None, 0)
    ok = torch.zeros((4, 46, 9, 9))
    assert rows(ok) == (ok.data_ptr(), 3726)
    ring = torch.zeros((3, 4, 46, 9, 9))
    assert rows(ring[1])[1] == 3726
    padded = torch.zeros((4, 13536), dtype=torch.uint8)[:, :13527]
    assert rows(padded, "mask", (torch.uint8, torch.bool), 13527) == (padded.data_ptr(), 13536)
    for bad in (torch.zeros((3, 46, 9, 9)), torch.zeros((4, 46, 9, 8)), torch.zeros((4, 46, 9, 9), dtype=torch.float64),
                torch.zeros((4, 9, 9, 46)).permute(0, 3, 1, 2), torch.zeros((46, 9, 9))):
        with pytest.raises(ValueError):
            rows(bad)


def test_invalid_arguments_are_rejected_before_any_device_work():
    """Every entry point returns KZ_E_ARG (-1) -- or KZ_E_NOT_INIT (-3) where the tables come first -- for null
    pointers and out-of-range sizes, without touching the device (so this runs without a GPU)."""
    L = nv.lib()
    z = None
    bad = (-1, -3)
    assert L.kz_reset(z, 4, 500, z, 500, z) in bad
    assert L.kz_load_positions(z, 4, 500, z, z, z, z, z, z) in bad
    assert L.kz_export_positions(z, 4, 500, z, z, z, z) in bad
    assert L.kz_refresh(z, 4, 500, z, 0, z, 0, z, z, 1, 0, 0, 0, 0, z, z) in bad
    assert L.kz_step(z, 4, 500, z, 1, z, 0, z, 0, z, z, z, z, z, z, z, 0, 0, 0, 1, z) == -1
    assert L.kz_step_rollout(z, 4, 500, z, 1, z, 0, z, 448, z, z, z, z, z, z, z, z, 0, 0, 0, 1, z) == -1
    assert L.kz_legal_bitmap(z, 4, 500, z, 0, z, 448, z, z, z) == -1
    assert L.kz_step_range(z, 4, 500, 0, 2, 0, z, 1, z, 0, z, 0, z, 0, z, z, z, z, z, z, z, z, 0, 0, 0, 1, z) == -1
    assert L.kz_bitmap_expand(z, 448, z, 4, z, 13536, z) == -1
    assert L.kz_sample_bitmap(z, 0, 13527, z, 448, 4, 0, 0, z, z, 1, z, z, 0, z) == -1
    assert L.kz_eval_bitmap_fwd(z, 0, 13527, z, 448, z, z, 4, z, z, z, z) == -1
    assert L.kz_eval_bitmap_bwd(z, 0, 13527, z, 448, z, z, 4, z, z, z, z, 13536, z, z) == -1
    assert L.kz_legal_mask(z, 4, 500, z, 0, z, z) == -1
    assert L.kz_observe(z, 4, 500, z, 0, z) == -1
    assert L.kz_piece_targets(z, 4, 500, z, z, z) in bad
    assert L.kz_errors(z, 4, 500, z, 0, z) in bad
    assert L.kz_sample_masked(z, 0, 13527, z, 13527, 4, 0, 0, z, z, 1, z, z, 0, z) == -1
    assert L.kz_gae(z, z, z, z, 8, 4, 0.99, 0.94, z, z, z) == -1
    assert L.kz_gae_exact(z, z, z, z, 8, 4, 0.99, 0.94, z, z, z) == -1
    assert L.kz_eval_masked_fwd(z, 0, 13527, z, 13527, z, z, 4, z, z, z, z) == -1
    assert L.kz_eval_masked_bwd(z, 0, 13527, z, 13527, z, z, 4, z, z, z, z, 13536, z) == -1
    assert L.kz_eval_masked_bwd_bias(z, 0, 13527, z, 13527, z, z, 4, z, z, z, z, 13536, z, z) == -1
    assert L.kz_ppo_loss(z, z, z, z, z, z, 4, 0.2, 0.5, 0.01, 1.0, z, z, z, z, z) == -1
    assert L.kz_obs_conv_fwd(z, z, z, z, 16, 4, 1, z, z) == -1
    assert L.kz_obs_conv_wgrad(z, z, z, z, 1, 16, 4, z, 1, z, z, z) == -1
    assert L.kz_adam_clip_step(0, z, z, z, z, z, z, 3e-4, 0.9, 0.999, 1e-8, 0.0, 0.5, z, 0, z, z) == -1
    assert L.kz_cobs_conv_fwd(z, z, z, z, 16, 4, 1, z, z) == -1
    assert L.kz_cobs_conv_wgrad(z, z, z, z, 1, 16, 4, z, 1, z, z, z) == -1
    assert L.kz_obs_conv_wgrad_ctas(0) <= 0 or L.kz_obs_conv_wgrad_ctas(1) >= 1
