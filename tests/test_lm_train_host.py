"""CPU: argument validation and workspace queries of the decoder-layer training entries (attention forward with lse,
attention backward, RMSNorm / RoPE backward).  Validation happens before any CUDA call, so it is testable without a GPU."""
import ctypes

import pytest


@pytest.fixture(scope="module")
def lib():
    from aria_b200 import build, _lib
    build.build()
    return _lib.load()


FAKE = ctypes.c_void_p(0x1000)   # never dereferenced: validation fails first


def _bwd(lib, B=1, H=2, T=256, head_dim=128, causal=1, ws=FAKE, ws_bytes=None, ptr=FAKE):
    if ws_bytes is None:
        ws_bytes = lib.aria_attention_bwd_workspace_bytes(B, H, T)
    return lib.aria_attention_bwd(ptr, FAKE, FAKE, FAKE, FAKE, FAKE, FAKE, FAKE, FAKE, None, B, H, T, H * T * 128, T * 128,
                                  H * T * 128, T * 128, 0.088, head_dim, causal, ws, ws_bytes, None)


def test_attention_bwd_workspace_bytes(lib):
    assert lib.aria_attention_bwd_workspace_bytes(8, 20, 2048) == 8 * 20 * 2048 * 4
    assert lib.aria_attention_bwd_workspace_bytes(2, 3, 300) == (2 * 3 * 300 * 4 + 255) // 256 * 256
    assert lib.aria_attention_bwd_workspace_bytes(0, 3, 300) == -1


def test_attention_bwd_rejects_bad_arguments(lib):
    assert _bwd(lib, ptr=None) == -1                          # null pointer
    assert _bwd(lib, ws=None) == -1                           # no workspace
    assert _bwd(lib, causal=0) == -2                          # non-causal backward: not implemented
    assert _bwd(lib, head_dim=72) == -2                       # only head_dim 128
    assert _bwd(lib, ws_bytes=lib.aria_attention_bwd_workspace_bytes(1, 2, 256) - 1) == -1   # workspace too small
    assert _bwd(lib, T=0) == -1


def test_attention_fwd_lse_rejects_bad_arguments(lib):
    def fwd(ptr=FAKE, lse=FAKE, head_dim=128, causal=1, T=256):
        return lib.aria_attention_fwd_lse(ptr, FAKE, FAKE, FAKE, lse, None, 1, 2, T, 2 * T * 128, T * 128, 2 * T * 128, T * 128,
                                          0.088, head_dim, causal, None)
    assert fwd(ptr=None) == -1
    assert fwd(lse=None) == -1
    assert fwd(causal=0) == -2
    assert fwd(head_dim=80) == -2
    assert fwd(T=-1) == -1


def test_rmsnorm_bwd_workspace_and_validation(lib):
    assert lib.aria_rmsnorm_bwd_workspace_bytes(1000, 2560) == 256 * 2560 * 4
    assert lib.aria_rmsnorm_bwd_workspace_bytes(100, 2560) == 100 * 2560 * 4
    assert lib.aria_rmsnorm_bwd_workspace_bytes(100, 12) == -1
    nb = lib.aria_rmsnorm_bwd_workspace_bytes(1000, 2560)
    args = [FAKE, FAKE, FAKE, None, FAKE, FAKE, 1000, 2560, 1e-6, FAKE, nb, None]
    bad = list(args)
    bad[0] = None
    assert lib.aria_rmsnorm_bwd(*bad) == -1                   # null x
    bad = list(args)
    bad[10] = nb - 4
    assert lib.aria_rmsnorm_bwd(*bad) == -1                   # workspace too small
    bad = list(args)
    bad[7] = 2564
    assert lib.aria_rmsnorm_bwd(*bad) == -1                   # d not a multiple of 8


def test_rope_bwd_validation(lib):
    assert lib.aria_rope_bwd(None, FAKE, FAKE, None, 10, 2, 10, None) == -1
    assert lib.aria_rope_bwd(FAKE, FAKE, FAKE, None, 10, 2, 0, None) == -1     # neither positions nor rows_per_batch
    assert lib.aria_rope_bwd(FAKE, FAKE, FAKE, None, 0, 2, 10, None) == 0      # nothing to do


def test_lm_train_refuses_cpu_tensors():
    import torch
    from aria_b200 import ops
    x = torch.zeros(4, 256, dtype=torch.bfloat16)
    with pytest.raises(RuntimeError):
        ops.rmsnorm_bwd(x, torch.ones(256, dtype=torch.bfloat16), x, 1e-6)
    q = torch.zeros(1, 2, 128, 128, dtype=torch.bfloat16)
    with pytest.raises(RuntimeError):
        ops.attention_fwd_lse(q, q, q, 0.088)
