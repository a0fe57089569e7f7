"""Client-side model shells shared by every family (reference: src/petals/models/*/model.py,
src/petals/client/from_pretrained.py:17-84).

A shell holds only what the reference keeps on the client — token embeddings (+ BLOOM's embedding LayerNorm), the
final norm, the LM / classification head and the trainable prompt-tuning parameters — while ``self.layers`` is a
:class:`RemoteSequential` over the stage workers. Nothing subclasses Hugging Face modeling classes (they moved
under the reference's feet, SURVEY.md §7.4 Q13); outputs are small HF-shaped dataclasses and generation is
provided by :mod:`petals_b200.client.remote_generation`.

``from_pretrained`` reads *only* the client tensors: it consults ``model.safetensors.index.json`` and opens just the
shards that contain them (the reference patches HF's shard resolver to the same effect).

On a CUDA client in bf16 the shell runs on the GPU with the engine's kernels (embedding gather, final norm fused
into the weight-streaming LM-head GEMV, arg-max) — the reference defaults these to the client CPU (Q12).
"""
from __future__ import annotations

import dataclasses
import json
import os
from typing import Dict, Optional, Tuple

import torch
import torch.nn as nn
import torch.nn.functional as F

from petals_b200.client.lm_head import LMHead
from petals_b200.client.ptune import PTuneMixin
from petals_b200.client.remote_generation import RemoteGenerationMixin, RemotePastKeyValues
from petals_b200.client.remote_sequential import RemoteSequential
from petals_b200.models.base import DistributedConfig
from petals_b200.utils.paths import resolve_model_path
from petals_b200.utils.logging import get_logger
from petals_b200.utils.misc import DUMMY, is_dummy
from petals_b200.utils.safetensors_io import SafetensorsFile

logger = get_logger(__name__)


@dataclasses.dataclass
class ModelOutput:
    last_hidden_state: Optional[torch.Tensor] = None
    logits: Optional[torch.Tensor] = None
    loss: Optional[torch.Tensor] = None
    past_key_values: Optional[RemotePastKeyValues] = None
    hidden_states: Optional[Tuple[torch.Tensor, ...]] = None
    attentions: Optional[Tuple[torch.Tensor, ...]] = None

    def __getitem__(self, i):
        vals = [v for v in (self.loss, self.logits if self.logits is not None else self.last_hidden_state, self.past_key_values) if v is not None]
        return vals[i]


def load_client_tensors(model_name_or_path: str, names: Dict[str, str]) -> Dict[str, torch.Tensor]:
    """canonical key -> tensor for the non-block parameters, opening only the shards that hold them."""
    path = resolve_model_path(str(model_name_or_path))
    index = os.path.join(path, "model.safetensors.index.json")
    wanted = {hf: key for key, hf in names.items()}
    out: Dict[str, torch.Tensor] = {}
    if os.path.exists(index):
        with open(index) as f:
            weight_map = json.load(f)["weight_map"]
        files = sorted({fn for hf, fn in weight_map.items() if hf in wanted})
    else:
        files = ["model.safetensors"]
    for fn in files:
        with SafetensorsFile(os.path.join(path, fn)) as f:
            for hf in f.keys():
                if hf in wanted:
                    out[wanted[hf]] = f.get_tensor(hf)
    return out


# Trainable client-side state that a fine-tuning run adds on top of the checkpoint's own tensors: canonical key ->
# name in the saved file (the reference stores them as ordinary parameters of the HF module, src/petals/client/ptune.py:24-39,
# models/llama/model.py:157-174; they "may be missing at load", ptune.py:22).
TRAINABLE_STATE_NAMES = {"prompts": "prompt_embeddings.weight", "deep_prompts": "intermediate_prompt_embeddings.weight",
                         "score": "score.weight"}


def client_state_names(config) -> Dict[str, str]:
    """Checkpoint names of everything the client owns: the family's embeddings / final norm / head plus the trainable
    prompt-tuning and classifier tensors (stored under the backbone's own prefix, e.g. ``model.prompt_embeddings.weight``)."""
    names = dict(type(config).client_weight_names)
    embed = names.get("embed", "")
    prefix = embed.split(".")[0] + "." if embed.count(".") >= 2 else ""
    names["prompts"] = prefix + TRAINABLE_STATE_NAMES["prompts"]
    names["deep_prompts"] = prefix + TRAINABLE_STATE_NAMES["deep_prompts"]
    names["score"] = TRAINABLE_STATE_NAMES["score"]
    return names


def _load_trainable(param: torch.Tensor, t: Dict[str, torch.Tensor], key: str) -> None:
    if key in t:
        if tuple(t[key].shape) != tuple(param.shape):
            raise ValueError(f"checkpoint tensor {key!r} has shape {tuple(t[key].shape)}, the model expects {tuple(param.shape)} "
                             f"(was it saved with another pre_seq_len / tuning_mode / num_labels?)")
        with torch.no_grad():
            param.copy_(t[key].to(param.dtype))


class FromPretrainedMixin:
    def save_pretrained(self, path: str) -> None:
        """Write ``config.json`` + ``model.safetensors`` with the *client* tensors only (embeddings, final norm, head,
        trained prompts / classifier); ``from_pretrained(path)`` resumes from it while the blocks stay remote
        (SURVEY.md §5.4: trainable state is ordinary client parameters saved with save_pretrained)."""
        from petals_b200.utils.safetensors_io import save_file

        os.makedirs(path, exist_ok=True)
        self.config.save_pretrained(path)
        names = client_state_names(self.config)
        state = {names[k]: v.detach().to("cpu").contiguous() for k, v in self.client_state().items()}
        save_file(state, os.path.join(path, "model.safetensors"), metadata={"format": "pt"})

    @classmethod
    def from_pretrained(cls, model_name_or_path, *args, torch_dtype=None, dht=None, device=None, **kwargs):
        config = cls.config_class.from_pretrained(model_name_or_path, **kwargs)
        if torch_dtype is None or torch_dtype == "auto":
            torch_dtype = config.torch_dtype if isinstance(getattr(config, "torch_dtype", None), torch.dtype) else torch.float32
        model = cls(config, dht=dht)
        tensors = load_client_tensors(model_name_or_path, client_state_names(config))
        missing = model.load_client_state(tensors)
        if missing:
            logger.warning(f"Client parameters initialised randomly (not in checkpoint): {sorted(missing)}")
        model = model.to(torch_dtype)
        model.float_trainable_()
        model.load_trainable_state(tensors)  # again, now in fp32: the cast to the model dtype above must not round them
        if device is not None:
            model = model.to(device)
        model.eval()
        return model


class DistributedModelBase(nn.Module, PTuneMixin, FromPretrainedMixin):
    """Embeddings + RemoteSequential + final norm."""

    config_class = DistributedConfig
    has_embedding_layernorm = False

    def __init__(self, config: DistributedConfig, *, dht=None):
        super().__init__()
        assert config.dht_prefix, "config.dht_prefix must be set (from_pretrained derives it from the model name)"
        self.config = config
        spec = config.block_spec()
        self.spec = spec
        H = config.hidden_size
        self.embed_tokens = nn.Embedding(config.vocab_size, H)
        if self.has_embedding_layernorm:
            self.embed_layernorm = nn.LayerNorm(H, eps=spec.norm_eps)
        if getattr(config, "fabric_address", None):  # a client on the stages' box: become a member of their landing-ring fabric
            from petals_b200.parallel.fabric import join_fabric

            join_fabric(config.fabric_address, config.fabric_rank, config.fabric_world, H, max_tokens=int(getattr(config, "fabric_max_tokens", 8192)),
                        device=getattr(config, "fabric_device", None))
        self.layers = RemoteSequential(config, dht=dht)
        self.norm_weight = nn.Parameter(torch.ones(H), requires_grad=False)
        self.norm_bias = nn.Parameter(torch.zeros(H), requires_grad=False) if spec.norm == "layer" else None
        self.embed_tokens.weight.requires_grad_(False)
        self.init_prompts(config)

    # ---- parameters -------------------------------------------------------------------------------------------
    def get_input_embeddings(self) -> nn.Embedding:
        return self.embed_tokens

    def load_client_state(self, t: Dict[str, torch.Tensor]) -> set:
        missing = set()
        H, V = self.config.hidden_size, self.config.vocab_size
        for key, want in (("embed", (V, H)), ("norm_w", (H,)), ("norm_b", (H,)), ("embed_ln_w", (H,)), ("embed_ln_b", (H,)), ("head", (V, H))):
            if key in t and tuple(t[key].shape) != want:  # lookups and GEMMs are sized from the config: refuse a checkpoint that disagrees with it
                raise ValueError(f"checkpoint tensor {key!r} has shape {tuple(t[key].shape)}, config.json implies {want}")
        with torch.no_grad():
            if "embed" in t:
                self.embed_tokens.weight.data = t["embed"].clone()
            else:
                missing.add("embed")
            if "norm_w" in t:
                self.norm_weight.data = t["norm_w"].clone()
            else:
                missing.add("norm_w")
            if self.norm_bias is not None and "norm_b" in t:
                self.norm_bias.data = t["norm_b"].clone()
            if self.has_embedding_layernorm:
                if "embed_ln_w" in t:
                    self.embed_layernorm.weight.data = t["embed_ln_w"].clone()
                    self.embed_layernorm.bias.data = t["embed_ln_b"].clone()
                    self.embed_layernorm.requires_grad_(False)
                else:
                    missing.add("embed_ln")
        self.load_trainable_state(t)
        return missing

    def load_trainable_state(self, t: Dict[str, torch.Tensor]) -> None:
        if hasattr(self, "prompt_embeddings"):
            _load_trainable(self.prompt_embeddings.weight, t, "prompts")
        if hasattr(self, "intermediate_prompt_embeddings"):
            _load_trainable(self.intermediate_prompt_embeddings.weight, t, "deep_prompts")

    def client_state(self) -> Dict[str, torch.Tensor]:
        out = {"embed": self.embed_tokens.weight, "norm_w": self.norm_weight}
        if self.norm_bias is not None:
            out["norm_b"] = self.norm_bias
        if self.has_embedding_layernorm:
            out["embed_ln_w"], out["embed_ln_b"] = self.embed_layernorm.weight, self.embed_layernorm.bias
        if hasattr(self, "prompt_embeddings"):
            out["prompts"] = self.prompt_embeddings.weight
        if hasattr(self, "intermediate_prompt_embeddings"):
            out["deep_prompts"] = self.intermediate_prompt_embeddings.weight
        names = type(self.config).client_weight_names
        return {k: v for k, v in out.items() if k in names or k in TRAINABLE_STATE_NAMES}

    def float_trainable_(self) -> None:
        """Prompt-tuning parameters stay fp32 regardless of the model dtype (reference ptune.py:24-39)."""
        for name in ("prompt_embeddings", "intermediate_prompt_embeddings"):
            if hasattr(self, name):
                getattr(self, name).float()

    # ---- pieces -----------------------------------------------------------------------------------------------------
    def _fast(self, t: torch.Tensor) -> bool:
        return t.is_cuda and self.embed_tokens.weight.dtype == torch.bfloat16 and not torch.is_grad_enabled()

    def embed(self, input_ids: torch.Tensor) -> torch.Tensor:
        w = self.embed_tokens.weight
        if self._fast(w) and w.shape[1] % 8 == 0:
            from petals_b200.ops import functional as Fn

            h = Fn.embedding(w, input_ids.to(w.device))
        else:
            h = self.embed_tokens(input_ids)
        if self.has_embedding_layernorm:
            h = self.embed_layernorm(h)
        return h

    def final_norm(self, h: torch.Tensor) -> torch.Tensor:
        if self.spec.norm == "rms":
            xf = h.float()
            xf = xf * torch.rsqrt(xf.pow(2).mean(-1, keepdim=True) + self.spec.norm_eps)
            return self.norm_weight * xf.to(h.dtype)
        return F.layer_norm(h, (h.shape[-1],), self.norm_weight, self.norm_bias, self.spec.norm_eps)

    def forward_hidden(self, input_ids=None, inputs_embeds=None, past_key_values: Optional[RemotePastKeyValues] = None,
                       apply_final_norm: bool = True) -> torch.Tensor:
        """Everything up to (and optionally including) the final norm."""
        if (input_ids is None) == (inputs_embeds is None):
            raise ValueError("You must specify exactly one of input_ids or inputs_embeds")
        if inputs_embeds is None:
            inputs_embeds = self.embed(input_ids.view(-1, input_ids.shape[-1]))
        B = inputs_embeds.shape[0]
        session = self.layers.active_session
        use_prompts = bool(self.config.tuning_mode and "ptune" in self.config.tuning_mode and (session is None or session.position == 0))
        intermediate_prompts = DUMMY
        if use_prompts:
            prompts, intermediate_prompts = self.get_prompt(B)
            inputs_embeds = torch.cat([prompts.to(inputs_embeds.device, inputs_embeds.dtype), inputs_embeds], dim=1)
            if not is_dummy(intermediate_prompts):
                intermediate_prompts = intermediate_prompts.to(inputs_embeds.device, inputs_embeds.dtype)
        hypo_ids = past_key_values.hypo_ids if past_key_values is not None else None
        if session is not None:
            hidden = self.layers(inputs_embeds, prompts=intermediate_prompts, hypo_ids=hypo_ids)
        else:
            hidden = self.layers(inputs_embeds, prompts=intermediate_prompts)
        if past_key_values is not None:
            past_key_values.update_seen(hidden.shape[1])
        if use_prompts:
            hidden = hidden[:, self.pre_seq_len:]
        return self.final_norm(hidden) if apply_final_norm else hidden

    def forward(self, input_ids=None, past_key_values=None, attention_mask=None, position_ids=None, inputs_embeds=None,
                use_cache=None, output_attentions=None, output_hidden_states=None, return_dict=None, **_) -> ModelOutput:
        _check_unsupported(attention_mask, position_ids, output_attentions, output_hidden_states)
        hidden = self.forward_hidden(input_ids, inputs_embeds, past_key_values)
        return ModelOutput(last_hidden_state=hidden, past_key_values=past_key_values)


def _check_unsupported(attention_mask, position_ids, output_attentions, output_hidden_states) -> None:
    """Custom masks / positions / attention dumps cannot be honoured by remote blocks (reference llama/model.py:63-74)."""
    if attention_mask is not None and not bool((attention_mask == 1).all()):
        raise ValueError("Custom attention masks are not supported")
    if position_ids is not None:
        first = position_ids[..., :-1] + 1
        if position_ids.shape[-1] > 1 and not bool((first == position_ids[..., 1:]).all()):
            raise ValueError("Non-consecutive position_ids are not supported")
    if output_attentions:
        raise ValueError("output_attentions=True is not supported")
    if output_hidden_states:
        raise ValueError("output_hidden_states=True is not supported")


class DistributedModelForCausalLM(nn.Module, RemoteGenerationMixin, FromPretrainedMixin):
    """Backbone shell + LM head + generation."""

    base_model_class = DistributedModelBase
    config_class = DistributedConfig

    def __init__(self, config: DistributedConfig, *, dht=None):
        super().__init__()
        self.config = config
        self.model = self.base_model_class(config, dht=dht)
        self.lm_head = LMHead(config)
        if self.lm_head.weight is None:
            self.lm_head.weight = self.model.embed_tokens.weight  # tied

    # ---- plumbing --------------------------------------------------------------------------------------------------
    def load_client_state(self, t: Dict[str, torch.Tensor]) -> set:
        missing = self.model.load_client_state(t)
        if getattr(self.config, "tie_word_embeddings", False) or "head" not in t:
            if not getattr(self.config, "tie_word_embeddings", False):
                missing.add("head")
            else:
                self.lm_head.weight = self.model.embed_tokens.weight
        else:
            self.lm_head.weight.data = t["head"].clone()
        return missing

    def load_trainable_state(self, t: Dict[str, torch.Tensor]) -> None:
        self.model.load_trainable_state(t)

    def client_state(self) -> Dict[str, torch.Tensor]:
        out = self.model.client_state()
        if not getattr(self.config, "tie_word_embeddings", False) and "head" in type(self.config).client_weight_names:
            out["head"] = self.lm_head.weight
        return out

    def float_trainable_(self) -> None:
        self.model.float_trainable_()

    def to(self, *args, **kwargs):
        out = super().to(*args, **kwargs)
        if getattr(self.config, "tie_word_embeddings", False):
            self.lm_head.weight = self.model.embed_tokens.weight
        return out

    def get_input_embeddings(self):
        return self.model.embed_tokens

    def get_output_embeddings(self):
        return self.lm_head

    @property
    def layers(self) -> RemoteSequential:
        return self.model.layers

    @property
    def device(self) -> torch.device:
        return self.model.embed_tokens.weight.device

    @property
    def dtype(self) -> torch.dtype:
        return self.model.embed_tokens.weight.dtype

    # ---- forward --------------------------------------------------------------------------------------------------------
    def logits_from_hidden(self, hidden_prenorm: torch.Tensor) -> torch.Tensor:
        """Final norm + LM head; decode shapes fuse both into one weight-streaming kernel on the GPU."""
        w = self.lm_head.weight
        m = self.model
        rows = hidden_prenorm.numel() // hidden_prenorm.shape[-1]
        if (m._fast(w) and hidden_prenorm.dtype == torch.bfloat16 and rows <= 8 and w.shape[0] % 2 == 0 and w.shape[1] % 8 == 0
                and w.shape[1] * rows * 2 <= 200 * 1024):
            from petals_b200.ops import functional as Fn

            return Fn.linear_decode(hidden_prenorm.contiguous(), w, norm_weight=m.norm_weight, norm_bias=m.norm_bias,
                                    norm_kind=Fn.NORM_RMS if m.spec.norm == "rms" else Fn.NORM_LAYER, eps=m.spec.norm_eps)
        return self.lm_head(m.final_norm(hidden_prenorm))

    def forward(self, input_ids=None, past_key_values=None, attention_mask=None, position_ids=None, inputs_embeds=None, labels=None,
                use_cache=None, output_attentions=None, output_hidden_states=None, return_dict=None, **_) -> ModelOutput:
        _check_unsupported(attention_mask, position_ids, output_attentions, output_hidden_states)
        hidden = self.model.forward_hidden(input_ids, inputs_embeds, past_key_values, apply_final_norm=False)
        logits = self.logits_from_hidden(hidden)
        loss = None
        if labels is not None:
            shift_logits = logits[..., :-1, :].float().contiguous()
            shift_labels = labels[..., 1:].contiguous().to(shift_logits.device)
            loss = F.cross_entropy(shift_logits.view(-1, shift_logits.size(-1)), shift_labels.view(-1), ignore_index=-100)
        return ModelOutput(logits=logits, loss=loss, past_key_values=past_key_values)

    def prepare_inputs_for_generation(self, input_ids, past_key_values=None, **kwargs):
        return dict(input_ids=input_ids, past_key_values=past_key_values)


class DistributedModelForSequenceClassification(nn.Module, FromPretrainedMixin):
    """Backbone shell + a trainable linear ``score`` head on the last non-padding token
    (reference: src/petals/models/llama/model.py:157-174, bloom/model.py:161-197)."""

    base_model_class = DistributedModelBase
    config_class = DistributedConfig

    def __init__(self, config: DistributedConfig, *, dht=None):
        super().__init__()
        self.config = config
        self.num_labels = int(getattr(config, "num_labels", 2))
        self.model = self.base_model_class(config, dht=dht)
        self.score = nn.Linear(config.hidden_size, self.num_labels, bias=False)

    def load_client_state(self, t):
        missing = self.model.load_client_state(t)
        _load_trainable(self.score.weight, t, "score")
        return missing

    def load_trainable_state(self, t: Dict[str, torch.Tensor]) -> None:
        self.model.load_trainable_state(t)
        _load_trainable(self.score.weight, t, "score")

    def client_state(self) -> Dict[str, torch.Tensor]:
        return dict(self.model.client_state(), score=self.score.weight)

    def float_trainable_(self) -> None:
        self.model.float_trainable_()
        self.score.float()

    @property
    def layers(self) -> RemoteSequential:
        return self.model.layers

    def forward(self, input_ids=None, attention_mask=None, inputs_embeds=None, labels=None, **kwargs) -> ModelOutput:
        hidden = self.model.forward_hidden(input_ids, inputs_embeds, None)
        logits = self.score(hidden.to(self.score.weight.dtype))
        B = logits.shape[0]
        pad = getattr(self.config, "pad_token_id", None)
        if input_ids is not None and pad is not None:
            lengths = (input_ids != pad).long().sum(-1) - 1
        else:
            lengths = torch.full((B,), logits.shape[1] - 1, dtype=torch.long)
        pooled = logits[torch.arange(B, device=logits.device), lengths.to(logits.device)]
        loss = None
        if labels is not None:
            labels = labels.to(pooled.device)
            problem = getattr(self.config, "problem_type", None)
            if problem is None:
                problem = "regression" if self.num_labels == 1 else ("single_label_classification" if labels.dtype in (torch.long, torch.int) else "multi_label_classification")
            if problem == "regression":
                loss = F.mse_loss(pooled.squeeze(-1) if self.num_labels == 1 else pooled, labels.to(pooled.dtype))
            elif problem == "single_label_classification":
                loss = F.cross_entropy(pooled.float().view(-1, self.num_labels), labels.view(-1))
            else:
                loss = F.binary_cross_entropy_with_logits(pooled.float(), labels.float())
        return ModelOutput(logits=pooled, loss=loss)
