"""CPU: workspace queries and argument validation of the fused lm_head + cross-entropy and embedding-backward entries (checked
before any CUDA call), and the shifted targets the loss is built from."""
import ctypes

import pytest
import torch

FAKE = ctypes.c_void_p(0x1000)   # never dereferenced: validation fails first


@pytest.fixture(scope="module")
def lib():
    from aria_b200 import build, _lib
    build.build()
    return _lib.load()


def _al(n):
    return (n + 255) // 256 * 256


def test_xent_fwd_workspace_bytes(lib):
    M, V = 300, 32000
    assert lib.aria_lm_xent_fwd_workspace_bytes(M, V) == _al(500 * M * 8) + _al(M * 4) + 2 * _al(3 * 4)
    assert lib.aria_lm_xent_fwd_workspace_bytes(37, 1000) == _al(16 * 37 * 8) + _al(37 * 4) + 2 * _al(4)
    assert lib.aria_lm_xent_fwd_workspace_bytes(10, 1004) == -1        # V % 8
    assert lib.aria_lm_xent_fwd_workspace_bytes(-1, 1000) == -1
    assert lib.aria_lm_xent_fwd_workspace_bytes(10, 0) == -1


def test_xent_bwd_workspace_bytes(lib):
    # small problems: the whole (256-padded) vocabulary in one chunk
    assert lib.aria_lm_xent_bwd_workspace_bytes(37, 1000, 256) == 256 + _al(37 * 256 * 4) + _al(37 * 1024 * 2)
    # recipe shape: a 512 MiB chunk budget -> 16384 columns at M = 16384
    M, V, d = 16384, 100352, 2560
    assert lib.aria_lm_xent_bwd_workspace_bytes(M, V, d) == 256 + M * d * 4 + M * 16384 * 2
    assert lib.aria_lm_xent_bwd_workspace_bytes(M, V, 2568) == -1      # d % 64
    assert lib.aria_lm_xent_bwd_workspace_bytes(M, 100353, d) == -1    # V % 8


def test_embedding_bwd_workspace_bytes(lib):
    assert lib.aria_embedding_bwd_workspace_bytes(16384, 100352) == (_al(100353 * 4) + _al(100354 * 4) + _al(100353 * 4)
                                                                     + _al(16384 * 4))
    assert lib.aria_embedding_bwd_workspace_bytes(-1, 1000) == -1
    assert lib.aria_embedding_bwd_workspace_bytes(10, 0) == -1


def _fwd(lib, h=FAKE, ws=FAKE, M=300, V=32000, d=512, nb=None):
    if nb is None:
        nb = lib.aria_lm_xent_fwd_workspace_bytes(M, V)
    return lib.aria_lm_xent_fwd(h, FAKE, FAKE, FAKE, FAKE, FAKE, M, V, d, ws, nb, None)


def _bwd(lib, h=FAKE, dw=FAKE, ws=FAKE, M=300, V=32000, d=512, nb=None):
    if nb is None:
        nb = lib.aria_lm_xent_bwd_workspace_bytes(M, V, 512)
    return lib.aria_lm_xent_bwd(h, FAKE, FAKE, FAKE, FAKE, FAKE, FAKE, dw, M, V, d, ws, nb, None)


def test_xent_fwd_rejects_bad_arguments(lib):
    assert _fwd(lib, h=None) == -1
    assert _fwd(lib, ws=None) == -1
    assert _fwd(lib, d=500) == -1                                       # d % 8
    assert _fwd(lib, V=32004) == -1                                     # V % 8
    assert _fwd(lib, nb=lib.aria_lm_xent_fwd_workspace_bytes(300, 32000) - 1) == -1
    assert _fwd(lib, M=0, nb=0) == 0                                    # nothing to do


def test_xent_bwd_rejects_bad_arguments(lib):
    assert _bwd(lib, h=None) == -1
    assert _bwd(lib, ws=None) == -1
    assert _bwd(lib, d=520) == -1                                       # d % 64
    assert _bwd(lib, V=31999) == -1
    assert _bwd(lib, nb=256 + 300 * 512 * 4 + 300 * 255 * 2) == -1      # not even one 256-column chunk
    assert _bwd(lib, M=0, nb=256) == 0


def test_embedding_bwd_rejects_bad_arguments(lib):
    nb = lib.aria_embedding_bwd_workspace_bytes(64, 1000)
    assert lib.aria_embedding_bwd(None, FAKE, FAKE, 64, 256, 1000, -1, FAKE, nb, None) == -1
    assert lib.aria_embedding_bwd(FAKE, FAKE, FAKE, 64, 250, 1000, -1, FAKE, nb, None) == -1     # d % 8
    assert lib.aria_embedding_bwd(FAKE, FAKE, FAKE, 64, 256, 1000, -1, FAKE, nb - 1, None) == -1
    assert lib.aria_embedding_bwd(FAKE, FAKE, FAKE, 64, 256, 1000, -1, None, nb, None) == -1
    assert lib.aria_embedding_bwd(FAKE, FAKE, FAKE, 0, 256, 1000, -1, FAKE, nb, None) == 0


def _mirror_targets(labels, attention_mask):
    """The positions and labels modeling_aria._shifted_cross_entropy keeps, as a [B, T-1] int tensor with -1 elsewhere."""
    B, T = labels.shape
    keep = torch.ones(B, T - 1, dtype=torch.bool) if attention_mask is None else attention_mask[:, -(T - 1):] != 0
    want = torch.full((B, T - 1), -1, dtype=torch.int64)
    sel = labels[..., 1:][keep]
    want[keep] = torch.where(sel == -100, torch.full_like(sel, -1), sel)
    return want


@pytest.mark.parametrize("masked", [False, True])
def test_shifted_targets_match_the_mirror(masked):
    from aria_b200.lm_train import shifted_targets
    g = torch.Generator().manual_seed(0)
    B, T = 3, 11
    labels = torch.randint(0, 50, (B, T), generator=g)
    labels[0, 4] = labels[2, 10] = labels[1, 1] = -100
    mask = None
    if masked:
        mask = torch.ones(B, T, dtype=torch.int64)
        mask[1, :3] = 0            # left padding
        mask[2, :1] = 0
    got = shifted_targets(labels, mask).view(B, T)
    assert got.dtype == torch.int32
    assert (got[:, -1] == -1).all()                                     # the last position predicts nothing
    assert torch.equal(got[:, :-1].long(), _mirror_targets(labels, mask))
    # the reference's loss over the kept rows equals the mean over our valid rows
    logits = torch.randn(B, T, 50, generator=g)
    from aria_b200.modeling_aria import AriaForConditionalGeneration
    want = AriaForConditionalGeneration._shifted_cross_entropy(logits, labels, mask)
    t = got.view(-1).long()
    ok = t >= 0
    ours = torch.nn.functional.cross_entropy(logits.view(-1, 50)[ok], t[ok])
    assert torch.allclose(ours, want)


def test_lm_loss_ops_refuse_cpu_tensors():
    from aria_b200 import ops
    h = torch.zeros(4, 256, dtype=torch.bfloat16)
    with pytest.raises(RuntimeError):
        ops.lm_xent_fwd(h, torch.zeros(64, 256, dtype=torch.bfloat16), torch.zeros(4, dtype=torch.int32))
    with pytest.raises(RuntimeError):
        ops.embedding_bwd(torch.zeros(4, dtype=torch.int64), h, 64)
