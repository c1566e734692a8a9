"""CPU: the oracle against the UNMODIFIED reference modules.  The numerical cases compare with the reference's outputs on the
same seeded inputs, captured by oracle/make_golden.py (section 3) into tests/golden/; the two seam-wiring checks instantiate the
reference's own classes and run only where oracle/ref_loader.py finds the reference files."""
import os

import pytest
import torch

from oracle import aria_oracle as O
from oracle import configs as C
from oracle.ref_loader import load_reference, reference_available

GOLD = os.path.join(os.path.dirname(__file__), "golden")
needs_reference = pytest.mark.skipif(not reference_available(), reason="reference files not staged (oracle/build_ref.py)")
torch.set_grad_enabled(False)


def _load(name):
    return torch.load(os.path.join(GOLD, name), weights_only=False)


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("T,E,k", [(1, 8, 2), (7, 8, 2), (64, 16, 6), (33, 64, 6)])
def test_moe_layer_live(dtype, T, E, k):
    gold = _load("moe_layer_live.pt")[f"{'fp32' if dtype == torch.float32 else 'bf16'}_T{T}_E{E}_k{k}"]
    tc = dict(hidden_size=128, moe_num_experts=E, moe_topk=k, moe_intermediate_size=64, moe_num_shared_experts=2)
    gen = torch.Generator().manual_seed(T * 131 + E)
    sd = {n: v.to(dtype) for n, v in C.moe_layer_state(tc, gen).items()}
    x = torch.randn(1, T, 128, generator=gen).to(dtype)
    assert C.state_checksum(sd) == pytest.approx(gold["checksum"], rel=1e-9), "seeded weights drifted"
    assert float(x.double().sum()) == pytest.approx(gold["x_checksum"], rel=1e-9), "seeded input drifted"
    want, ridx = gold["out"], gold["top_idx"]      # the reference MoELayer's output and its router's expert choice
    got, parts = O.moe_layer(x, sd, k, return_parts=True)
    if torch.equal(ridx.sort(1).values, parts["top_idx"].sort(1).values):
        tol = 1e-6 if dtype == torch.float32 else 0.0
        assert (want.float() - got.float()).abs().max() <= tol
    else:  # a bf16 tie resolved differently by torch.topk: only tied rows may differ
        vals = parts["logits"].float().sort(1, descending=True).values
        tied = vals[:, k - 1] == vals[:, k]
        bad = (want.float() - got.float()).abs().amax(-1).view(-1) > 0
        assert not (bad & ~tied).any()


@needs_reference
def test_installer_rebinds_reference_seams():
    """aria_b200.install.install() patches the reference MoELayer.forward and the `experts_gemm` global (no GPU needed to
    check the wiring; executing the patched path needs CUDA)."""
    from aria_b200 import install, moe_lm as ours
    ref = load_reference()
    cfg = ref.moe_lm.AriaMoELMConfig(hidden_size=128, moe_num_experts=8, moe_topk=2, moe_intermediate_size=64,
                                     moe_num_shared_experts=2, num_hidden_layers=2, num_attention_heads=1, vocab_size=64)
    model = ref.moe_lm.AriaMoELMForCausalLM(cfg)
    saved = ref.moe_lm.experts_gemm
    try:
        assert install.install(model, ref.moe_lm) == 2
        assert ref.moe_lm.experts_gemm is ours.experts_gemm
        layer = model.model.layers[0].mlp
        assert layer.forward.__func__ is install._moe_forward
        with pytest.raises(RuntimeError):   # no CPU fallback
            layer(torch.zeros(1, 4, 128, dtype=torch.bfloat16))
    finally:
        ref.moe_lm.experts_gemm = saved


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("scale", [1.0, 64.0])
def test_moe_layer_training_losses_backward_live(dtype, scale):
    """Training-mode routing (z-loss + load-balancing loss injected through MoEAuxLossAutoScaler, moe_lm.py:84-166,
    203-241): gradients of the unmodified reference vs the oracle's restatement, and vs the closed form the CUDA kernel
    implements (O.router_loss_grad).  The reference gradients are a strided sample per parameter (oracle/make_golden.py)."""
    gold = _load("moe_layer_train_live.pt")["fp32" if dtype == torch.float32 else "bf16"]
    T, E, k, d = 48, 16, 4, 128
    # large coefficients so the loss terms are well above bf16 noise of the main gradient
    tc = dict(hidden_size=d, moe_num_experts=E, moe_topk=k, moe_intermediate_size=64, moe_num_shared_experts=2,
              moe_z_loss_coeff=0.5, moe_aux_loss_coeff=2.0)
    gen = torch.Generator().manual_seed(5)
    sd = {n: v.to(dtype) for n, v in C.moe_layer_state(tc, gen).items()}
    sd["router.weight"] = (sd["router.weight"].float() * 20).to(dtype)   # spread the logits
    x0 = torch.randn(1, T, d, generator=gen).to(dtype)
    dout = torch.randn(1, T, d, generator=gen).to(dtype)
    assert C.state_checksum(sd) == pytest.approx(gold["checksum"], rel=1e-9), "seeded weights drifted"
    assert float(x0.double().sum()) + float(dout.double().sum()) == pytest.approx(gold["x_checksum"], rel=1e-9)
    ref_grads = gold[scale]
    with torch.enable_grad():
        w = {n: v.clone().requires_grad_(True) for n, v in sd.items()}
        xo = x0.clone().requires_grad_(True)
        O._LossGradInjector.scale = scale
        try:
            O.moe_layer(xo, w, k, loss_coeffs=(0.5, 2.0)).backward(dout)
        finally:
            O._LossGradInjector.scale = 1.0
        # eval-mode oracle (no losses): the difference of the router gradients is the loss contribution
        w0 = {n: v.clone().requires_grad_(True) for n, v in sd.items()}
        x1 = x0.clone().requires_grad_(True)
        O.moe_layer(x1, w0, k).backward(dout)
    tol = 1e-6 if dtype == torch.float32 else 0.0
    for n, want in ref_grads["grads"].items():
        got = w[n].grad.reshape(-1)[::ref_grads["grad_strides"][n]]
        assert (want.float() - got.float()).abs().max() <= tol * max(1.0, ref_grads["grad_absmax"][n]), n
    # dx sums three branches (router, dispatch, shared expert); autograd's bf16 accumulation order is an engine detail,
    # so in bf16 it is only checked to an ulp-level tolerance (the parameter gradients above are bit-exact)
    xtol = 1e-6 if dtype == torch.float32 else 1e-2
    dx = ref_grads["dx"]
    assert (dx.float() - xo.grad.float()).abs().max() <= xtol * max(1.0, float(dx.float().abs().max()))
    # closed form: d_router(train) - d_router(eval) == router_loss_grad^T @ x
    x2 = x0.reshape(T, d)
    logits = O.router_gating(x2, sd["router.weight"])
    _, _, counts = O.router_routing(logits, k)
    dl = O.router_loss_grad(logits, counts, k, 0.5, 2.0, scale)
    assert float(dl.abs().max()) > 0
    delta = w["router.weight"].grad.float() - w0["router.weight"].grad.float()
    closed = dl.t() @ x2.float()
    rel = (delta - closed).abs().max() / closed.abs().max()
    assert rel <= (1e-4 if dtype == torch.float32 else 4e-2), float(rel)


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_grouped_gemm_lora_layer_live(dtype):
    """LoRA on the grouped GEMM: the unmodified `aria/lora/layers.py` (run under a stand-in for the two peft symbols it
    imports, see oracle/ref_loader.py; outputs in tests/golden/lora_layer_live.pt) vs the oracle's restatement — forward and the
    gradients of A, B and x."""
    gold = _load("lora_layer_live.pt")["fp32" if dtype == torch.float32 else "bf16"]
    g = torch.Generator().manual_seed(4)
    E, K, N, r, alpha = 4, 64, 96, 8, 32
    counts = torch.tensor([16, 0, 40, 24])
    rows = int(counts.sum())
    w = (torch.randn(E, K, N, generator=g) * 0.05).to(dtype)
    a = (torch.randn(E, K, r, generator=g) * 0.05).to(dtype)
    b = (torch.randn(E, r, N, generator=g) * 0.05).to(dtype)
    x0 = torch.randn(rows, K, generator=g).to(dtype)
    dy = torch.randn(rows, N, generator=g).to(dtype)
    assert float(x0.double().sum()) == pytest.approx(gold["x_checksum"], rel=1e-9), "seeded input drifted"
    assert gold["scaling"] == alpha / r
    want = gold["out"]
    with torch.enable_grad():
        ao, bo, xo = a.clone().requires_grad_(True), b.clone().requires_grad_(True), x0.clone().requires_grad_(True)
        got = O.grouped_gemm_lora(xo, w, ao, bo, counts, alpha / r)
        got.backward(dy)
    assert torch.equal(got.detach(), want)
    assert torch.equal(ao.grad, gold["d_a"])
    assert torch.equal(bo.grad, gold["d_b"])
    tol = 1e-6 if dtype == torch.float32 else 1e-2   # dx sums two autograd branches (accumulation order, see above)
    assert (xo.grad.float() - gold["dx"].float()).abs().max() <= tol * float(gold["dx"].float().abs().max())
    # merged weights (layers.py:154-213: W += A @ B * scaling) give the same function as the adapter path
    if dtype == torch.float32:
        assert (O.sequential_gemm(x0, w + torch.matmul(a, b) * (alpha / r), counts) - gold["merged_out"]).abs().max() <= 1e-5
        merged_w = (w + torch.matmul(a, b) * (alpha / r)).reshape(-1)[::gold["merged_weight_stride"]]
        assert (gold["merged_weight"] - merged_w).abs().max() <= 1e-7


@needs_reference
def test_install_vit_rebinds_the_reference_vision_layers():
    """Seam 3 wiring (executing the patched layers needs CUDA): every Idefics2EncoderLayer of the reference vision tower is
    patched, the tuple/tensor return convention of the host transformers version is detected, and CPU input fails loudly."""
    from aria_b200 import install
    ref = load_reference()
    vc = ref.vision_encoder.AriaVisionConfig(hidden_size=144, num_attention_heads=2, num_hidden_layers=2, intermediate_size=256,
                                             patch_size=14, image_size=56, hidden_act="gelu_pytorch_tanh")
    vc._attn_implementation = "eager"
    tower = ref.vision_encoder.AriaVisionModel(vc)
    assert install.install_vit(tower) == 2
    layer = tower.vision_model.encoder.layers[0]
    assert layer.forward.__func__ is install._vit_layer_forward and layer._aria_returns_tuple is False   # transformers 5.x here
    with pytest.raises(RuntimeError):
        layer(torch.zeros(1, 16, 144, dtype=torch.bfloat16), None)
