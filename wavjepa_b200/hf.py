"""Hugging-Face-shaped entry point (SURVEY.md 8a-H5): the reference recommends
`AutoModel / AutoFeatureExtractor.from_pretrained("labhamlet/wavjepa-base", trust_remote_code=True)` and
`model(extractor(audio, return_tensors="pt")["input_values"]) -> (embeddings, timestamps)` (README.md:72-108,
hear_configs/WavJEPA_huggingface.py:1-39).  The remote code lives on the hub, not in the reference checkout, and cannot be
fetched here, so the NUMERICAL behaviour of this pair follows the HEAR runtime of the checkout (hear_api/runtime.py,
runtime_natjepa.py: loudness to -14 dBFS, 2.01 s windows, per-window normalisation, padded frames key-masked and cut) --
parity with the hub code is unpinned by necessity (DESIGN.md).  What is mirrored exactly is the CALL SHAPE:

    extractor = WavJEPAFeatureExtractor.from_pretrained(path_or_name)         # AutoFeatureExtractor stand-in
    model     = WavJEPAModel.from_pretrained(checkpoint_path_or_dict).to(dev)   # AutoModel stand-in
    feats = extractor(audio, return_tensors="pt")["input_values"]             # [B, L] (Nat: [B, 2, L]) fp32
    emb, ts = model(feats)                                                    # [B, frames, 768], [B, frames] (ms)

plus the three module-level functions of hear_configs/WavJEPA_huggingface.py (`load_model`, `get_scene_embeddings`,
`get_timestamp_embeddings`).  If `transformers` is importable the two classes register as `PreTrainedModel`-free plain
objects on purpose: no hub access, no config download -- `from_pretrained` takes a LOCAL Lightning checkpoint.
"""
from __future__ import annotations

from typing import Dict, Optional, Sequence, Union

import torch
from torch import nn

from . import hear

SAMPLING_RATE = 16000


class BatchFeature(dict):
    """Minimal `transformers.BatchFeature`: a dict with attribute access and .to()."""
    __getattr__ = dict.__getitem__

    def to(self, *args, **kwargs) -> "BatchFeature":
        return BatchFeature({k: (v.to(*args, **kwargs) if torch.is_tensor(v) else v) for k, v in self.items()})


class WavJEPAFeatureExtractor:
    """`AutoFeatureExtractor` stand-in: batches raw 16 kHz waveforms into `input_values` (fp32, zero-padded to the longest
    clip).  No numerical preprocessing happens here -- loudness / window normalisation are part of the model call, where
    they run as kernels (hear.RuntimeJEPA.to_feature / embed_chunks)."""
    model_input_names = ["input_values"]

    def __init__(self, sampling_rate: int = SAMPLING_RATE, in_channels: int = 1):
        self.sampling_rate, self.in_channels = sampling_rate, in_channels

    @classmethod
    def from_pretrained(cls, name_or_path: str = "labhamlet/wavjepa-base", **kwargs) -> "WavJEPAFeatureExtractor":
        kwargs.pop("trust_remote_code", None)
        return cls(in_channels=2 if "nat" in str(name_or_path).lower() else 1, **{k: v for k, v in kwargs.items() if k in ("sampling_rate",)})

    def __call__(self, raw_speech: Union[torch.Tensor, Sequence], sampling_rate: Optional[int] = None,
                 return_tensors: Optional[str] = "pt", **kwargs) -> BatchFeature:
        if sampling_rate is not None and sampling_rate != self.sampling_rate:
            raise ValueError(f"WavJEPA expects {self.sampling_rate} Hz audio, got {sampling_rate} Hz")
        if return_tensors not in (None, "pt"):
            raise ValueError("only return_tensors='pt' is supported")
        if torch.is_tensor(raw_speech):
            x = raw_speech.to(torch.float32)
            if x.dim() == 1:
                x = x.unsqueeze(0)
        else:
            clips = [torch.as_tensor(c, dtype=torch.float32) for c in raw_speech]
            L = max(c.shape[-1] for c in clips)
            x = torch.stack([torch.nn.functional.pad(c, (0, L - c.shape[-1])) for c in clips])
        return BatchFeature({"input_values": x})


class WavJEPAModel(nn.Module):
    """`AutoModel` stand-in over the HEAR runtime: forward(input_values) -> (embeddings, timestamps).

    Like HF's `from_pretrained`, `from_pretrained` returns the model in eval mode, where forward runs under no_grad.
    Fine-tuning is opt-in: after `model.train()`, forward in grad mode (precision "bf16") is differentiable --
    `emb, _ = model(input_values); loss.backward()` fills `.grad` of the trainable feature-path parameters (model
    parameters under `runtime.model.`) and, when input_values requires grad, `input_values.grad` (hear.RuntimeJEPA,
    DESIGN.md 2.5)."""

    def __init__(self, runtime: hear.RuntimeJEPA):
        super().__init__()
        self.runtime = runtime
        self.train(runtime.training)   # the runtime's mode (eval when it comes from a loader)
        self.sample_rate = runtime.sample_rate
        self.embedding_size = runtime.embedding_size

    @classmethod
    def from_pretrained(cls, checkpoint: Union[str, Dict], nat: Optional[bool] = None, precision: str = "bf16",
                        **kwargs) -> "WavJEPAModel":
        """checkpoint: path to (or dict of) a Lightning checkpoint with 'state_dict' (hub names cannot be resolved here:
        there is no network).  nat: build the binaural WavJEPA-Nat runtime (default: inferred from the state-dict keys).
        precision: "bf16" (default) or "tf32" (reference-precision features, wavjepa_b200.hear).  Other keyword
        arguments go to the HEAR loader, e.g. layer=k: embed encoder hidden state k instead of the final features
        (hear.load_model, JEPA.get_hidden_states)."""
        for k in ("trust_remote_code", "force_download"):
            kwargs.pop(k, None)
        ck = hear._load_weights((checkpoint,))
        if nat is None:
            nat = any(k.startswith("extract_audio.cnns.") for k in ck["state_dict"])
        rt = hear.load_model_nat(ck, precision=precision, **kwargs) if nat else hear.load_model(ck, precision=precision, **kwargs)
        return cls(rt)

    def forward(self, input_values: torch.Tensor):
        return self.runtime.get_timestamp_embeddings(input_values)


# ---- hear_configs/WavJEPA_huggingface.py:9-39 --------------------------------------------------------------------------
extractor = WavJEPAFeatureExtractor()


def load_model(*args, precision: str = "bf16", **kwargs) -> WavJEPAModel:
    """hear_configs/WavJEPA_huggingface.py:19-24 (there: the hub model; here: args[0] = local checkpoint path / dict).
    precision: "bf16" (default) or "tf32"; other keyword arguments (e.g. layer=k) as in WavJEPAModel.from_pretrained."""
    model = WavJEPAModel.from_pretrained(args[0], precision=precision, **kwargs)
    model.sample_rate = SAMPLING_RATE
    return model


def get_scene_embeddings(audio, model: WavJEPAModel) -> torch.Tensor:
    x, _ = model(extractor(audio, return_tensors="pt")["input_values"])     # :27-32
    return torch.mean(x, dim=1)


def get_timestamp_embeddings(audio, model: WavJEPAModel):
    return model(extractor(audio, return_tensors="pt")["input_values"])     # :35-39
