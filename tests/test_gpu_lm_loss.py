"""GPU: the fused lm_head + cross-entropy (forward stats epilogue, chunked backward), the embedding backward and the whole-model
training loss (`lm_train.causal_lm_loss`, `AriaForConditionalGeneration.training_loss`) against torch / the fp32 oracle."""
import os

import pytest
import torch
import torch.nn.functional as F

import test_gpu_lm_train as layer_tests

pytestmark = pytest.mark.gpu
DEV = "cuda"
GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
_rel_l2 = layer_tests._rel_l2


def _problem(M, V, d, seed, ignore=0.1):
    g = torch.Generator().manual_seed(seed)
    h = torch.randn(M, d, generator=g).bfloat16()
    w = (torch.randn(V, d, generator=g) * d ** -0.5).bfloat16()
    t = torch.randint(0, V, (M,), generator=g)
    t[torch.rand(M, generator=g) < ignore] = -1
    return h.to(DEV), w.to(DEV), t.to(DEV, torch.int32)


def _fused(h, w, t, need_dw=True, workspace_bytes=None):
    from aria_b200 import ops
    loss, lse, nv = ops.lm_xent_fwd(h, w, t)
    dh, dw = ops.lm_xent_bwd(h, w, t, lse, nv, torch.ones(1, device=DEV), need_dw=need_dw, workspace_bytes=workspace_bytes)
    torch.cuda.synchronize()
    return loss, lse, nv, dh, dw


@pytest.mark.parametrize("M,V,d", [(1, 1000, 256), (37, 1000, 256), (300, 32000, 512), (4096, 100352, 2560)])
def test_loss_and_lse_match_torch(M, V, d):
    from aria_b200 import ops
    h, w, t = _problem(M, V, d, seed=M)
    loss, lse, nv, _, _ = _fused(h, w, t)
    z = ops.linear(h, w).float()                       # the bf16 logits the unfused path sees
    tl = t.long()
    want = F.cross_entropy(z, tl.clamp_min(0), reduction="none")[tl >= 0].mean() if (tl >= 0).any() else z.new_tensor(float("nan"))
    assert int(nv) == int((tl >= 0).sum())
    assert abs(float(loss) - float(want)) <= 1e-3 * abs(float(want)), (float(loss), float(want))
    assert float((lse - torch.logsumexp(z, -1)).abs().max()) <= 2e-3


def _torch_grads(h, w, t):
    h32, w32 = h.float().requires_grad_(True), w.float().requires_grad_(True)
    with torch.enable_grad():
        F.cross_entropy(h32 @ w32.t(), t.long(), ignore_index=-1).backward()
    return h32.grad, w32.grad


@pytest.mark.parametrize("M,V,d", [(37, 1000, 256), (300, 32000, 512)])
def test_backward_matches_fp32_autograd(M, V, d):
    h, w, t = _problem(M, V, d, seed=M + 1)
    want_dh, want_dw = _torch_grads(h, w, t)
    _, _, _, dh, dw = _fused(h, w, t)
    assert _rel_l2(dh, want_dh) <= 2e-2
    assert _rel_l2(dw, want_dw) <= 2e-2
    _, _, _, dh2, dw2 = _fused(h, w, t, need_dw=False)    # frozen lm_head: dW skipped, dh unchanged
    assert dw2 is None and torch.equal(dh, dh2)


def test_chunked_backward_matches_one_chunk():
    from aria_b200 import _lib as L
    M, V, d = 300, 32000, 512
    h, w, t = _problem(M, V, d, seed=5)
    _, _, _, dh, dw = _fused(h, w, t)
    assert L.load().aria_lm_xent_bwd_workspace_bytes(M, V, d) >= 256 + M * d * 4 + M * 32000 * 2   # default: one chunk
    ws = 256 + M * d * 4 + M * 3840 * 2                 # 3840-column chunks: 9 of them, the last one partial
    _, _, _, dh8, dw8 = _fused(h, w, t, workspace_bytes=ws)
    assert _rel_l2(dh8, dh) <= 1e-3 and _rel_l2(dw8, dw) <= 1e-3
    assert torch.equal(dw8, dw)                          # dW rows do not depend on the chunking at all


def test_fused_loss_is_deterministic():
    h, w, t = _problem(4096, 32000, 512, seed=6)
    a, b = _fused(h, w, t), _fused(h, w, t)
    for x, y in zip(a, b):
        assert torch.equal(x, y)


def test_edge_cases():
    h, w, t = _problem(77, 1000, 256, seed=7)
    loss, _, nv, dh, dw = _fused(h, w, torch.full_like(t, -1))      # nothing to predict
    assert torch.isnan(loss) and int(nv) == 0
    assert float(dh.abs().max()) == 0.0 and float(dw.abs().max()) == 0.0
    bad = t.clone()
    bad[3] = 1000                                                     # target >= V: NaN, not a fault
    loss, lse, *_ = _fused(h, w, bad)
    assert torch.isnan(loss) and torch.isfinite(lse).all()


def test_lm_head_loss_memory():
    """At the recipe shape the fused forward + backward needs well under 1 GiB beyond inputs and gradients (the unfused path
    keeps M*V*6 bytes: bf16 logits, their fp32 copy and its gradient)."""
    from aria_b200 import lm_train
    M, V, d = 16384, 100352, 2560
    h, w, t = _problem(M, V, d, seed=8)
    h.requires_grad_(True)
    w.requires_grad_(True)
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    base = torch.cuda.memory_allocated()
    with torch.enable_grad():
        loss = lm_train.LMHeadCrossEntropyFunction.apply(h, w, t)
        loss.backward()
    torch.cuda.synchronize()
    grads = h.grad.numel() * 2 + w.grad.numel() * 2
    growth = torch.cuda.max_memory_allocated() - base - grads
    assert growth < 2 ** 30, growth / 2 ** 30
    assert torch.isfinite(h.grad).all() and torch.isfinite(w.grad).all()


# ------------------------------------------------------------------------------------------------ embedding backward
def test_embedding_backward():
    from aria_b200 import _lib as L, ops
    g = torch.Generator().manual_seed(9)
    n, vocab, d, skip = 4096, 1000, 256, 7
    ids = torch.randint(0, vocab, (n,), generator=g)
    ids[::50] = skip
    ids[5], ids[6] = -3, vocab + 4                      # out of range: ignored, no fault
    dout = torch.randn(n, d, generator=g).bfloat16()
    keep = (ids != skip) & (ids >= 0) & (ids < vocab)
    want = torch.zeros(vocab, d).index_add_(0, ids[keep], dout[keep].float())
    got = ops.embedding_bwd(ids.to(DEV), dout.to(DEV), vocab, skip)
    assert torch.allclose(got.float().cpu(), want.bfloat16().float(), rtol=1e-2, atol=1e-2)
    assert float(got[skip].abs().max()) == 0.0
    assert torch.equal(got, ops.embedding_bwd(ids.to(DEV), dout.to(DEV), vocab, skip))     # bit-reproducible
    # untouched rows keep whatever the caller put there
    lib = L.load()
    table = torch.full((vocab, d), 3.0, dtype=torch.bfloat16, device=DEV)
    nb = lib.aria_embedding_bwd_workspace_bytes(n, vocab)
    ws = torch.empty(nb, dtype=torch.uint8, device=DEV)
    idd, dd = ids.to(DEV), dout.to(DEV)
    L.check(lib.aria_embedding_bwd(idd.data_ptr(), dd.data_ptr(), table.data_ptr(), n, d, vocab, skip, ws.data_ptr(), nb,
                                   torch.cuda.current_stream().cuda_stream), "embedding_bwd")
    used = torch.zeros(vocab, dtype=torch.bool)
    used[ids[keep]] = True
    assert (table.cpu()[~used] == 3.0).all()
    assert torch.equal(table[used.to(DEV)], got[used.to(DEV)])


def test_embedding_backward_one_hot_id():
    from aria_b200 import ops
    g = torch.Generator().manual_seed(10)
    n, vocab, d = 16384, 100352, 2560
    ids = torch.full((n,), 4242, dtype=torch.int64)
    dout = torch.randn(n, d, generator=g).bfloat16()
    got = ops.embedding_bwd(ids.to(DEV), dout.to(DEV), vocab)
    want = dout.float().sum(0)                         # fp32 sum, rounded once: equal up to the summation order
    assert torch.allclose(got[4242].float().cpu(), want.bfloat16().float(), rtol=1e-2, atol=1e-2)
    assert int((got.float().abs().sum(1) > 0).sum()) == 1


# ------------------------------------------------------------------------------------------------ whole model
def _lm_cfg():
    return dict(hidden_size=256, num_attention_heads=2, num_hidden_layers=2, moe_num_experts=8, moe_topk=2,
                moe_intermediate_size=128, moe_num_shared_experts=2, vocab_size=1000, rms_norm_eps=1e-5, rope_theta=5e6)


def _lm(tc, sd):
    from aria_b200 import moe_lm
    lm = moe_lm.AriaMoELMForCausalLM(moe_lm.AriaMoELMConfig(**tc), device=DEV)
    lm.load_state_dict({n: v.to(DEV) for n, v in sd.items()}, strict=True)
    for p_ in lm.parameters():
        p_.requires_grad_(True)
    return lm


def _layer_sd(sd, i):
    p = f"model.layers.{i}."
    return {n[len(p):]: v for n, v in sd.items() if n.startswith(p)}


def _oracle_loss(ids, labels, mask, sd32, tc, capture=None):
    from oracle import aria_oracle as O
    x = F.embedding(ids, sd32["model.embed_tokens.weight"])
    orig = O.moe_layer
    if capture is not None:
        def spy(h, w_, k, prefix="", **kw):
            capture.append(h.detach())
            return orig(h, w_, k, prefix, **kw)
        O.moe_layer = spy
    try:
        for i in range(tc["num_hidden_layers"]):
            x, _ = layer_tests._oracle_layer(x, _layer_sd(sd32, i), tc, mask)
    finally:
        O.moe_layer = orig
    h = O.rms_norm(x, sd32["model.norm.weight"], tc["rms_norm_eps"])
    logits = F.linear(h, sd32["lm_head.weight"])
    from aria_b200.modeling_aria import AriaForConditionalGeneration
    return AriaForConditionalGeneration._shifted_cross_entropy(logits, labels, mask)


def _whole_model_inputs(tc, sd32):
    """B = 2, T = 160, row 1 left-padded by 37, some labels -100; token ids with a near-tie top-k in any layer are redrawn."""
    from oracle import aria_oracle as O
    B, T, pad, V = 2, 160, 37, tc["vocab_size"]
    g = torch.Generator().manual_seed(11)
    ids = torch.randint(0, V, (B, T), generator=g)
    mask = torch.ones(B, T, dtype=torch.int64)
    mask[1, :pad] = 0
    real = mask.bool().view(-1)
    for _ in range(30):
        cap = []
        with torch.no_grad():
            _oracle_loss(ids, ids, mask, sd32, tc, capture=cap)
        bad = torch.zeros(B * T, dtype=torch.bool)
        for i, hcap in enumerate(cap):
            lg = O.router_gating(hcap.reshape(-1, tc["hidden_size"]),
                                 sd32[f"model.layers.{i}.mlp.router.weight"]).sort(1, descending=True).values
            k = tc["moe_topk"]
            bad |= (lg[:, k - 1] - lg[:, k]) / lg.abs().amax(1) <= 2 ** -6
        bad &= real
        if not bool(bad.any()):
            break
        ids.view(-1)[bad] = torch.randint(0, V, (int(bad.sum()),), generator=g)
    assert not bool(bad.any())
    labels = ids.clone()
    labels[0, 10:20] = -100
    labels[1, :pad + 1] = -100        # the last pad position would predict the first real token from a row that sees no key
    return ids, labels, mask


def _our_grads(lm):
    return {n: p_.grad.clone() for n, p_ in lm.named_parameters()}


def test_whole_model_loss_and_gradients_vs_oracle():
    from aria_b200 import lm_train
    from oracle import configs as C
    tc = _lm_cfg()
    sd = {n: v.bfloat16() for n, v in C.lm_state(tc, torch.Generator().manual_seed(12), prefix="").items()}
    sd32 = {n: v.float().requires_grad_(True) for n, v in sd.items()}
    ids, labels, mask = _whole_model_inputs(tc, sd32)
    with torch.enable_grad():
        want = _oracle_loss(ids, labels, mask, sd32, tc)
        want.backward()
    lm = _lm(tc, sd)
    with torch.enable_grad():
        loss = lm_train.causal_lm_loss(lm, labels.to(DEV), input_ids=ids.to(DEV), attention_mask=mask.to(DEV))
        loss.backward()
    assert abs(float(loss.detach()) - float(want.detach())) <= 5e-3 * abs(float(want.detach())), (float(loss), float(want))
    got = _our_grads(lm)
    assert sorted(got) == sorted(sd32)
    for n in sd32:
        assert _rel_l2(got[n], sd32[n].grad) <= 2e-2, (n, _rel_l2(got[n], sd32[n].grad))


@pytest.mark.parametrize("router_losses", [False, True])
def test_gradient_checkpointing_is_bit_identical(router_losses):
    from aria_b200 import lm_train
    from oracle import configs as C
    tc = _lm_cfg()
    sd = {n: v.bfloat16() for n, v in C.lm_state(tc, torch.Generator().manual_seed(13), prefix="").items()}
    lm = _lm(tc, sd)
    g = torch.Generator().manual_seed(14)
    ids = torch.randint(0, 1000, (2, 160), generator=g).to(DEV)
    mask = torch.ones(2, 160, dtype=torch.int64, device=DEV)
    mask[0, :20] = 0
    runs = []
    for ckpt in (False, True):
        lm.zero_grad(set_to_none=True)
        with torch.enable_grad():
            loss = lm_train.causal_lm_loss(lm, ids, input_ids=ids, attention_mask=mask, router_losses=router_losses,
                                           gradient_checkpointing=ckpt)
            loss.backward()
        runs.append([loss.detach().clone()] + [p_.grad.clone() for p_ in lm.parameters()])
    for a, b in zip(*runs):
        assert torch.equal(a, b)


def test_training_loss_matches_inference_loss():
    from oracle import configs as C
    from aria_b200.modeling_aria import AriaConfig, AriaForConditionalGeneration
    gold = torch.load(os.path.join(GOLD, "aria_tiny_bf16_full.pt"), weights_only=False)
    m = AriaForConditionalGeneration(AriaConfig.from_dict(C.TINY), device=DEV)
    m.load_state_dict({k: v.to(DEV) for k, v in C.aria_state(C.TINY, seed=0, dtype=torch.bfloat16).items()}, strict=True)
    for p_ in m.language_model.parameters():
        p_.requires_grad_(True)
    ids, pv = gold["input_ids"], gold["pixel_values"]
    labels = ids.clone()
    labels[0, :3] = -100
    want = m(ids, pv, None, labels=labels).loss
    with torch.enable_grad():
        loss = m.training_loss(ids, labels, pixel_values=pv)
        assert loss.grad_fn is not None
        loss.backward()
    assert abs(float(loss) - float(want)) <= 1e-2 * abs(float(want)), (float(loss), float(want))
    emb = m.get_input_embeddings().weight.grad
    assert emb is not None and float(emb[C.TINY["image_token_index"]].abs().max()) == 0.0
    assert torch.isfinite(m.get_output_embeddings().weight.grad).all()
    for p_ in m.multi_modal_projector.parameters():
        p_.requires_grad_(True)
    with pytest.raises(NotImplementedError):
        m.training_loss(ids, labels, pixel_values=pv)


def test_full_width_two_layer_step_is_finite():
    from aria_b200 import lm_train, moe_lm
    from aria_b200.modeling_aria import init_random_
    tc = dict(hidden_size=2560, num_attention_heads=20, num_hidden_layers=2, moe_num_experts=64, moe_topk=6,
              moe_intermediate_size=1664, moe_num_shared_experts=2, vocab_size=100352, rms_norm_eps=1e-5, rope_theta=5e6)
    lm = moe_lm.AriaMoELMForCausalLM(moe_lm.AriaMoELMConfig(**tc), device=DEV)
    with torch.no_grad():
        init_random_(lm, seed=3)
    for p_ in lm.parameters():
        p_.requires_grad_(True)
    g = torch.Generator().manual_seed(15)
    ids = torch.randint(0, 100352, (1, 2048), generator=g).to(DEV)
    with torch.enable_grad():
        loss = lm_train.causal_lm_loss(lm, ids, input_ids=ids, gradient_checkpointing=True)
        loss.backward()
    assert torch.isfinite(loss)
    for n, p_ in lm.named_parameters():
        assert p_.grad is not None and torch.isfinite(p_.grad).all(), n
