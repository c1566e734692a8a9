"""Host-side mirror of `aria/model/modeling_aria.py`: AriaForConditionalGeneration.forward()/generate() with the
Hugging Face state-dict layout, running entirely on the B200-native kernels.

forward() follows modeling_aria.py:194-335: embed -> vision tower -> projector -> masked_scatter merge -> LM, with the
reference's argument list (attention_mask, position_ids, labels -> loss, ...).  Differences that are deliberate: no
autograd through this class (inference hot path; training = moe_train / lora), the KV cache is our static `KVCache`
(HF layout [B,H,T,hd] per layer), integer index tensors stay int32 on the device.  The drop-in surface for an
*unmodified* HF / reference model is aria_b200.install + aria_b200.hf_attention (tests/test_gpu_dropin.py).
"""
from __future__ import annotations

from typing import Optional

import torch
import torch.nn as nn

from . import ops
from .moe_lm import AriaMoELMConfig, AriaMoELMForCausalLM, KVCache, bf16
from .projector import AriaProjector
from .vision_encoder import AriaVisionConfig, AriaVisionModel


class AriaConfig:
    """configuration_aria.py:31-114 (attributes used on the hot path)."""

    def __init__(self, vision_config, text_config, projector_patch_to_query_dict=None, image_token_index=32000,
                 ignore_index=-100, **_ignored):
        self.vision_config = vision_config if not isinstance(vision_config, dict) else AriaVisionConfig(**vision_config)
        self.text_config = text_config if not isinstance(text_config, dict) else AriaMoELMConfig(**text_config)
        self.projector_patch_to_query_dict = {int(k): int(v) for k, v in
                                              (projector_patch_to_query_dict or {1225: 128, 4900: 256}).items()}
        self.image_token_index = image_token_index
        self.ignore_index = ignore_index

    @classmethod
    def from_dict(cls, cfg: dict):
        """From the plain-dict configs used by oracle/configs.py and bench.py."""
        return cls(cfg["vision_config"], cfg["text_config"], cfg["projector"]["patch_to_query_dict"],
                   cfg["image_token_index"])


class AriaCausalLMOutputWithPast:
    def __init__(self, logits, past_key_values):
        self.logits = logits
        self.past_key_values = past_key_values
        self.loss = None


class AriaForConditionalGeneration(nn.Module):
    """modeling_aria.py:125-365."""

    def __init__(self, config: AriaConfig, device=None):
        super().__init__()
        self.config = config
        v, t = config.vision_config, config.text_config
        self.vision_tower = AriaVisionModel(v, device)
        self.multi_modal_projector = AriaProjector(  # build_mm_projector, modeling_aria.py:102-122
            config.projector_patch_to_query_dict, v.hidden_size, v.num_attention_heads, v.hidden_size, t.hidden_size,
            t.hidden_size, device)
        self.vocab_size = t.vocab_size
        self.language_model = AriaMoELMForCausalLM(t, device)

    # ---- modeling_aria.py:145-192: the helpers aria/train.py:70-75 and the recipes call on the model
    def freeze_vit(self):
        for p in self.vision_tower.parameters():
            p.requires_grad = False

    def freeze_projector(self):
        for p in self.multi_modal_projector.parameters():
            p.requires_grad = False

    def freeze_llm(self):
        for p in self.language_model.parameters():
            p.requires_grad = False

    def get_input_embeddings(self):
        return self.language_model.get_input_embeddings()

    def set_input_embeddings(self, value):
        self.language_model.set_input_embeddings(value)

    def get_output_embeddings(self):
        return self.language_model.get_output_embeddings()

    def set_output_embeddings(self, value):
        self.language_model.set_output_embeddings(value)

    def set_moe_z_loss_coeff(self, value):
        self.language_model.set_z_loss_coeff(value)

    def set_moe_aux_loss_coeff(self, value):
        self.language_model.set_aux_loss_coeff(value)

    def enable_expert_parallel(self, max_tokens: int, group=None):
        """Shard the routed experts of every MoE layer over the ranks of `group` (rank r serves experts
        [r*E/W, (r+1)*E/W), a dim-0 view of the HF weights) and exchange token rows over NVLink peer memory
        (aria_b200.expert_parallel.FusedPeerTransport: dispatch fused into the permute kernel, return path fused into the fc2
        GEMM epilogue).  Every rank must then call forward() in lock-step with its own tokens."""
        import torch.distributed as dist
        from .expert_parallel import ExpertParallelMoE, FusedPeerTransport
        t = self.config.text_config
        W, r = dist.get_world_size(group), dist.get_rank(group)
        tr = FusedPeerTransport(max_tokens, t.hidden_size, t.moe_intermediate_size, t.moe_num_experts, t.moe_topk, self.device, group)
        lo, hi = r * t.moe_num_experts // W, (r + 1) * t.moe_num_experts // W
        for layer in self.language_model.model.layers:
            m = layer.mlp
            w = {"router.weight": m.router.weight, "experts.fc1.weight": m.experts.fc1.weight[lo:hi],
                 "experts.fc2.weight": m.experts.fc2.weight[lo:hi],
                 "shared_experts.gate_proj.weight": m.shared_experts.gate_proj.weight,
                 "shared_experts.up_proj.weight": m.shared_experts.up_proj.weight,
                 "shared_experts.down_proj.weight": m.shared_experts.down_proj.weight}
            m.expert_parallel = ExpertParallelMoE(w, t.moe_num_experts, t.moe_topk, group=group, transport=tr)
        self._ep_transport = tr
        return tr

    @property
    def device(self):
        return self.language_model.lm_head.weight.device

    @torch.no_grad()
    def forward(self, input_ids: torch.Tensor = None, pixel_values: Optional[torch.Tensor] = None,
                pixel_mask: Optional[torch.Tensor] = None, attention_mask: Optional[torch.Tensor] = None,
                position_ids: Optional[torch.Tensor] = None, past_key_values: Optional[KVCache] = None,
                inputs_embeds: Optional[torch.Tensor] = None, labels: Optional[torch.Tensor] = None,
                use_cache: Optional[bool] = None, output_attentions: Optional[bool] = None,
                output_hidden_states: Optional[bool] = None, return_dict: Optional[bool] = None,
                cache_position: Optional[torch.Tensor] = None, num_logits_to_keep: int = 0,
                max_cache_len: Optional[int] = None, input_ids_host: Optional[torch.Tensor] = None) -> AriaCausalLMOutputWithPast:
        """Same arguments as the reference forward (modeling_aria.py:194-210); `max_cache_len` / `input_ids_host` are ours.

        input_ids / pixel_values / pixel_mask may be HOST tensors (pinned for async copies): they are copied to
        the device on the current stream; image-token bookkeeping is then done on the host copy (no device sync).
        Device-resident input_ids cost one sync for the image-token count check, like the reference's `.item()`
        (modeling_aria.py:265).

        attention_mask: the HF 2-D padding mask [B, past + T] (1 = real token).  Padded keys are masked inside the attention
        kernels (prefill and decode).  position_ids [B, T]: RoPE positions (default: cache positions, as in LlamaModel).
        labels: shifted cross-entropy exactly as modeling_aria.py:300-323 (the loss itself is torch glue on our logits;
        this class is the inference path, so it carries no grad_fn — training goes through aria_b200.moe_train / lora).
        Not supported, and rejected loudly: output_attentions / output_hidden_states (no such tensors exist in the fused
        path), return_dict=False."""
        if output_attentions or output_hidden_states:
            raise NotImplementedError("aria_b200: attention weights / per-layer hidden states are not materialised by the fused path")
        if return_dict is False:
            raise NotImplementedError("aria_b200: tuple outputs are not supported (return_dict=False)")
        if cache_position is not None and past_key_values is not None and int(cache_position.reshape(-1)[0]) != past_key_values.seq_len:
            raise NotImplementedError("aria_b200: cache_position must continue the KV cache (static cache, append-only)")
        dev = self.device
        ids_host = input_ids_host  # optional host copy of device-resident ids (bookkeeping without a sync)
        if input_ids is not None and not input_ids.is_cuda:
            ids_host = input_ids
            input_ids = input_ids.to(dev, non_blocking=True)
        if pixel_values is not None and not pixel_values.is_cuda:
            pixel_values = pixel_values.to(dev, non_blocking=True)
        if inputs_embeds is None:
            inputs_embeds = ops.embedding(input_ids.contiguous(), self.get_input_embeddings().weight)
        elif pixel_values is not None:
            inputs_embeds = inputs_embeds.clone()   # the merge below writes in place; the reference's masked_scatter does not

        if pixel_values is not None:
            feats, image_attn_mask = self.vision_tower(pixel_values.to(bf16), pixel_mask)
            image_features = self.multi_modal_projector(feats, image_attn_mask)
            n_image_features = image_features.shape[0] * image_features.shape[1]
            src = ids_host if ids_host is not None else input_ids
            n_image_tokens = int((src == self.config.image_token_index).sum())
            if n_image_tokens != n_image_features:
                raise ValueError(  # modeling_aria.py:268-271
                    f"Image features and image tokens do not match: tokens: {n_image_tokens}, features {n_image_features}")
            ops.merge_image_features(input_ids.reshape(-1).contiguous(), self.config.image_token_index,
                                     image_features.reshape(-1, image_features.shape[-1]),
                                     inputs_embeds.view(-1, inputs_embeds.shape[-1]))

        B, T, _ = inputs_embeds.shape
        cache = past_key_values
        if cache is None:
            cache = self.language_model.new_cache(B, max_cache_len or T, dev)
        key_mask = None
        if attention_mask is not None:
            if attention_mask.shape != (B, cache.seq_len + T):
                raise ValueError(f"attention_mask must be [B, past + T] = {(B, cache.seq_len + T)}, got {tuple(attention_mask.shape)}")
            if not bool((attention_mask != 0).all()):      # host tensor: free; device tensor: one sync, only when a mask is given
                key_mask = (attention_mask == 0).to(device=dev, dtype=torch.uint8).contiguous()
        pos = None
        if position_ids is not None:
            if position_ids.shape != (B, T):
                raise ValueError(f"position_ids must be [B, T] = {(B, T)}, got {tuple(position_ids.shape)}")
            pos = position_ids.to(device=dev, dtype=torch.int32).reshape(-1).contiguous()
        logits, cache = self.language_model(inputs_embeds, cache, num_logits_to_keep, key_mask=key_mask, position_ids=pos)
        out = AriaCausalLMOutputWithPast(logits, cache)
        if labels is not None:
            out.loss = self._shifted_cross_entropy(logits, labels, attention_mask)
        return out

    def training_loss(self, input_ids: torch.Tensor, labels: torch.Tensor, pixel_values: Optional[torch.Tensor] = None,
                      pixel_mask: Optional[torch.Tensor] = None, attention_mask: Optional[torch.Tensor] = None,
                      position_ids: Optional[torch.Tensor] = None, router_losses: bool = False,
                      gradient_checkpointing: bool = False) -> torch.Tensor:
        """The loss of forward(..., labels=labels) as a tensor with a grad_fn, for fine-tuning the language model (the recipes'
        freeze_vit; aria_b200.lm_train.causal_lm_loss does the work).  The vision tower and projector run without grad and
        their features replace the image-token embeddings as in forward(); the image-token row of the embedding table gets no
        gradient.  Their backward is not built: a vision-tower or projector parameter that requires grad raises
        NotImplementedError (call freeze_vit() / freeze_projector())."""
        from .lm_train import _MergeImageFunction, causal_lm_loss
        if any(p.requires_grad for m in (self.vision_tower, self.multi_modal_projector) for p in m.parameters()):
            raise NotImplementedError("aria_b200: the vision tower / projector backward is not implemented; freeze them "
                                      "(freeze_vit(), freeze_projector()) to train the language model")
        dev = self.device
        input_ids = input_ids.to(dev)
        lm = self.language_model
        embeds = None
        if pixel_values is not None:
            from .lm_train import EmbeddingFunction
            with torch.no_grad():
                feats, image_attn_mask = self.vision_tower(pixel_values.to(dev, bf16), pixel_mask)
                image_features = self.multi_modal_projector(feats, image_attn_mask)
            n_image_tokens = int((input_ids == self.config.image_token_index).sum())
            if n_image_tokens != image_features.shape[0] * image_features.shape[1]:
                raise ValueError(f"Image features and image tokens do not match: tokens: {n_image_tokens}, "
                                 f"features {image_features.shape[0] * image_features.shape[1]}")
            embeds = EmbeddingFunction.apply(input_ids, lm.model.embed_tokens.weight, self.config.image_token_index)
            embeds = _MergeImageFunction.apply(embeds, input_ids, self.config.image_token_index, image_features)
        return causal_lm_loss(lm, labels, input_ids=None if embeds is not None else input_ids, inputs_embeds=embeds,
                              attention_mask=attention_mask, position_ids=position_ids, router_losses=router_losses,
                              gradient_checkpointing=gradient_checkpointing, skip_embed_id=self.config.image_token_index)

    @staticmethod
    def _shifted_cross_entropy(logits, labels, attention_mask):
        """modeling_aria.py:300-323, verbatim semantics: tokens < n predict n; padded positions dropped through the 2-D mask."""
        labels = labels.to(logits.device)
        if attention_mask is not None:
            shift_mask = attention_mask[:, -(logits.shape[1] - 1):].to(logits.device)
            shift_logits = logits[..., :-1, :][shift_mask != 0].contiguous()
            shift_labels = labels[..., 1:][shift_mask != 0].contiguous()
        else:
            shift_logits = logits[..., :-1, :].contiguous()
            shift_labels = labels[..., 1:].contiguous()
        return nn.functional.cross_entropy(shift_logits.view(-1, shift_logits.size(-1)).float(), shift_labels.view(-1))

    def prepare_inputs_for_generation(self, input_ids, past_key_values=None, inputs_embeds=None, pixel_values=None,
                                      pixel_mask=None, attention_mask=None, cache_position=None, num_logits_to_keep=None,
                                      **kwargs):
        """modeling_aria.py:337-365: with a non-empty cache only the new token ids go in; pixel inputs only at step 0;
        position ids from the padding mask (what LlamaForCausalLM.prepare_inputs_for_generation derives)."""
        past = 0 if past_key_values is None else past_key_values.seq_len
        model_inputs = {"input_ids": input_ids[:, past:] if past else input_ids, "past_key_values": past_key_values,
                        "attention_mask": attention_mask}
        if inputs_embeds is not None and not past:
            model_inputs = {"inputs_embeds": inputs_embeds, "input_ids": input_ids, "past_key_values": past_key_values,
                            "attention_mask": attention_mask}
        if attention_mask is not None:
            pos = (attention_mask.long().cumsum(-1) - 1).clamp_min(0)
            model_inputs["position_ids"] = pos[:, past:] if past else pos
        if num_logits_to_keep is not None:
            model_inputs["num_logits_to_keep"] = num_logits_to_keep
        if not past:
            model_inputs["pixel_values"] = pixel_values
            model_inputs["pixel_mask"] = pixel_mask
        return model_inputs

    @torch.no_grad()
    def generate(self, input_ids, pixel_values=None, pixel_mask=None, max_new_tokens: int = 16, attention_mask=None):
        """Greedy decoding (the reference goes through HF GenerationMixin, modeling_aria.py:125,337-365):
        prefill with the image, then one token per step against the KV cache (pixel inputs only at step 0).
        attention_mask [B, T]: LEFT-padded batches of ragged prompts (the HF generation convention); positions are derived
        from it as GenerationMixin does."""
        B, T = input_ids.shape
        mask = None if attention_mask is None else attention_mask.to("cpu", torch.long)
        inputs = self.prepare_inputs_for_generation(input_ids, None, pixel_values=pixel_values, pixel_mask=pixel_mask,
                                                    attention_mask=mask, num_logits_to_keep=1)
        out = self.forward(**inputs, max_cache_len=T + max_new_tokens)
        cache = out.past_key_values
        tokens = [out.logits[:, -1].float().argmax(-1)]
        all_ids = input_ids.to(tokens[0].device)
        for _ in range(max_new_tokens - 1):
            all_ids = torch.cat([all_ids, tokens[-1].view(B, 1)], dim=1)
            if mask is not None:
                mask = torch.cat([mask, torch.ones(B, 1, dtype=torch.long)], dim=1)
            inputs = self.prepare_inputs_for_generation(all_ids, cache, attention_mask=mask, num_logits_to_keep=1)
            step = self.forward(**inputs)
            tokens.append(step.logits[:, -1].float().argmax(-1))
        return torch.cat([input_ids.to(tokens[0].device), torch.stack(tokens, 1)], dim=1)


class GraphedPrefill:
    """CUDA-graph capture of one prefill `forward()` for fixed shapes (streams + graphs instead of a tracing
    compiler): the whole ViT -> projector -> merge -> LM chain has no host sync, so it is captured once and replayed.

        g = GraphedPrefill(model, input_ids_host, pixel_values_host)      # warm-up + capture
        logits = g(input_ids_host, pixel_values_host)                      # H2D copies + replay; logits on device
        logits = g.replay()                                                # inputs already resident in HBM
    """

    def __init__(self, model: "AriaForConditionalGeneration", input_ids: torch.Tensor, pixel_values: torch.Tensor,
                 num_logits_to_keep: int = 1):
        self.model = model
        dev = model.device
        self.ids_dev = torch.empty(input_ids.shape, dtype=torch.int64, device=dev)
        self.pv_dev = torch.empty(pixel_values.shape, dtype=bf16, device=dev)
        self.ids_dev.copy_(input_ids)
        self.pv_dev.copy_(pixel_values)
        self.n_image_tokens = int((input_ids == model.config.image_token_index).sum())
        ids_host = input_ids.cpu()
        kw = dict(num_logits_to_keep=num_logits_to_keep, input_ids_host=ids_host)
        side = torch.cuda.Stream(device=dev)
        side.wait_stream(torch.cuda.current_stream(dev))
        with torch.cuda.stream(side):
            for _ in range(2):
                model(self.ids_dev, self.pv_dev, None, **kw)
        torch.cuda.current_stream(dev).wait_stream(side)
        self.graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(self.graph):
            self.logits = model(self.ids_dev, self.pv_dev, None, **kw).logits

    def replay(self) -> torch.Tensor:
        self.graph.replay()
        return self.logits

    def __call__(self, input_ids: torch.Tensor, pixel_values: torch.Tensor) -> torch.Tensor:
        if not input_ids.is_cuda:  # same ValueError contract as forward() (modeling_aria.py:268-271), checked on the host
            n = int((input_ids == self.model.config.image_token_index).sum())
            if n != self.n_image_tokens:
                raise ValueError(f"Image features and image tokens do not match: tokens: {n}, features {self.n_image_tokens}")
        self.ids_dev.copy_(input_ids, non_blocking=True)
        self.pv_dev.copy_(pixel_values, non_blocking=True)
        return self.replay()


def init_random_(model: nn.Module, seed: int = 0, std: float = 0.02):
    """Random-init (no checkpoint offline): N(0, std^2) for matrices / embeddings / biases / queries, 1 for the
    norm scales (the only 1-D parameters named `weight`)."""
    g = torch.Generator(device=next(model.parameters()).device).manual_seed(seed)
    for name, p in model.named_parameters():
        if p.dim() == 1 and name.endswith("weight"):
            p.fill_(1.0)
        else:
            p.normal_(0.0, std, generator=g)
    return model
