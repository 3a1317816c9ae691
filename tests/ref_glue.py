"""Run the REFERENCE'S OWN code for the hot path on the CPU (test infrastructure for tests/golden/make_ref_golden.py; never shipped).

The original project's `src/slam_llm` (a checkout named by the SLAM_LLM_REFERENCE environment variable) imports third-party
packages that are absent offline (peft, openai-whisper, soundfile, deepspeed, omegaconf).  This module installs small stand-ins
for exactly the names the reference reaches for, puts its `src` first on sys.path and imports the reference's modules UNMODIFIED:

    slam_llm.models.slam_model      (setup_encoder / setup_llm / setup_encoder_projector / slam_model.forward, :68-407)
    slam_llm.models.encoder         (WhisperWrappedEncoder.load -> extract_variable_length_features, :13-45)
    slam_llm.models.projector       (EncoderProjectorConcat / Cov1d, :5-49)
    slam_llm.utils.metric           (compute_accuracy, :3-20)
    slam_llm.utils.config_utils     (generate_peft_config, :46-65)
    slam_llm.datasets.speech_dataset / speech_dataset_large   (__getitem__ + collator)

The stand-ins restate the PUBLISHED third-party behaviour the reference pins:
  peft 0.6.0     LoraConfig, get_peft_model, PeftModel, tuners/lora/layer.py Linear (forward + reset_lora_parameters)
  openai-whisper model.py AudioEncoder / ResidualAttentionBlock / MultiHeadAttention / LayerNorm / Linear / Conv1d,
                 audio.py load_audio (WAV via scipy; no ffmpeg offline) / pad_or_trim / log_mel_spectrogram
  omegaconf      the repo's own shim (src/slam_llm/_compat/omegaconf_shim.py), loaded by file path
The repo's `src/slam_llm` mirror must NOT be importable as `slam_llm` in the same process: use this module only from a
dedicated process (tests/golden/make_ref_golden.py) or through `run_in_subprocess`.
"""
from __future__ import annotations

import importlib
import importlib.machinery
import importlib.util
import math
import os
import sys
import types
from dataclasses import dataclass, field
from typing import Dict, Iterable, List, Optional

import numpy as np
import torch
import torch.nn as nn
import torch.nn.functional as F

REFERENCE = os.environ.get("SLAM_LLM_REFERENCE", "")                          # checkout of the original SLAM-LLM project
REFERENCE_SRC = os.path.join(os.path.abspath(REFERENCE), "src") if REFERENCE else ""
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def reference_available() -> bool:
    return bool(REFERENCE_SRC) and os.path.isdir(os.path.join(REFERENCE_SRC, "slam_llm"))


# =====================================================================================================================
# peft 0.6.0 stand-in
# =====================================================================================================================
@dataclass
class LoraConfig:
    r: int = 8
    lora_alpha: int = 8
    target_modules: Optional[List[str]] = None
    lora_dropout: float = 0.0
    bias: str = "none"
    task_type: Optional[str] = None
    inference_mode: bool = False
    fan_in_fan_out: bool = False
    modules_to_save: Optional[List[str]] = None
    peft_type: str = "LORA"


class _Unsupported:
    def __init__(self, *a, **kw):
        raise NotImplementedError("only LoRA is restated in the peft stand-in")


class TaskType:
    CAUSAL_LM = "CAUSAL_LM"
    SEQ_2_SEQ_LM = "SEQ_2_SEQ_LM"


class LoraLinear(nn.Module):
    """peft 0.6.0 tuners/lora/layer.py `Linear`: result = F.linear(x, W, b) + lora_B(lora_A(dropout(x))) * alpha / r."""

    def __init__(self, base: nn.Linear, r: int, lora_alpha: int, lora_dropout: float, adapter: str = "default"):
        super().__init__()
        self.in_features, self.out_features = base.in_features, base.out_features
        self.weight, self.bias = base.weight, base.bias
        self.weight.requires_grad = False
        self.r = {adapter: r}
        self.scaling = {adapter: lora_alpha / r}
        self.lora_dropout = nn.ModuleDict({adapter: nn.Dropout(p=lora_dropout) if lora_dropout > 0.0 else nn.Identity()})
        self.lora_A = nn.ModuleDict({adapter: nn.Linear(self.in_features, r, bias=False)})
        self.lora_B = nn.ModuleDict({adapter: nn.Linear(r, self.out_features, bias=False)})
        nn.init.kaiming_uniform_(self.lora_A[adapter].weight, a=math.sqrt(5))        # reset_lora_parameters
        nn.init.zeros_(self.lora_B[adapter].weight)
        self.active_adapter = adapter

    def forward(self, x: torch.Tensor) -> torch.Tensor:
        previous_dtype = x.dtype
        result = F.linear(x, self.weight, bias=self.bias)
        a = self.active_adapter
        x = x.to(self.lora_A[a].weight.dtype)
        result = result + self.lora_B[a](self.lora_A[a](self.lora_dropout[a](x))) * self.scaling[a]
        return result.to(previous_dtype)


class LoraModel(nn.Module):
    def __init__(self, model: nn.Module, config: LoraConfig):
        super().__init__()
        self.model = model
        targets = list(config.target_modules)
        for name, mod in list(model.named_modules()):
            if isinstance(mod, nn.Linear) and any(name == t or name.endswith("." + t) for t in targets):
                parent = model.get_submodule(name.rsplit(".", 1)[0]) if "." in name else model
                setattr(parent, name.rsplit(".", 1)[-1], LoraLinear(mod, config.r, config.lora_alpha, config.lora_dropout))
        for n, p in model.named_parameters():                                          # mark_only_lora_as_trainable (bias="none")
            if "lora_" not in n:
                p.requires_grad = False

    def forward(self, *a, **kw):
        return self.model(*a, **kw)


class PeftModel(nn.Module):
    """PeftModelForCausalLM surface the reference touches: forward(**kw), generate, print_trainable_parameters, and
    __getattr__ forwarding to base_model (so `llm.model` is the HF causal LM, slam_model.py:375-380)."""

    def __init__(self, model: nn.Module, peft_config: LoraConfig):
        super().__init__()
        self.base_model = LoraModel(model, peft_config)
        self.peft_config = {"default": peft_config}

    def __getattr__(self, name: str):
        try:
            return super().__getattr__(name)
        except AttributeError:
            return getattr(self.base_model, name)

    def forward(self, *a, **kw):
        return self.base_model(*a, **kw)

    def generate(self, *a, **kw):
        return self.base_model.model.generate(*a, **kw)

    def print_trainable_parameters(self):
        t = sum(p.numel() for p in self.parameters() if p.requires_grad)
        n = sum(p.numel() for p in self.parameters())
        print(f"trainable params: {t:,d} || all params: {n:,d} || trainable%: {100 * t / n}")

    @classmethod
    def from_pretrained(cls, model, model_id, is_trainable=False, **kw):
        """peft directory layout: adapter_config.json + adapter_model.bin (keys without the adapter name)."""
        import json
        with open(os.path.join(model_id, "adapter_config.json")) as f:
            c = json.load(f)
        cfg = LoraConfig(r=c["r"], lora_alpha=c["lora_alpha"], target_modules=c["target_modules"], lora_dropout=c.get("lora_dropout", 0.0))
        self = cls(model, cfg)
        sd = torch.load(os.path.join(model_id, "adapter_model.bin"), map_location="cpu")
        sd = {k.replace("lora_A.weight", "lora_A.default.weight").replace("lora_B.weight", "lora_B.default.weight"): v for k, v in sd.items()}
        missing, unexpected = self.load_state_dict(sd, strict=False)
        assert not unexpected, unexpected
        return self


def get_peft_model(model, peft_config):
    return PeftModel(model, peft_config)


def _peft_module() -> types.ModuleType:
    m = types.ModuleType("peft")
    m.LoraConfig, m.TaskType, m.get_peft_model, m.PeftModel = LoraConfig, TaskType, get_peft_model, PeftModel
    m.PeftConfig = LoraConfig
    m.AdaptionPromptConfig = m.PrefixTuningConfig = _Unsupported
    m.prepare_model_for_kbit_training = lambda model: model
    return m


# =====================================================================================================================
# openai-whisper stand-in (model.py AudioEncoder + audio.py helpers)
# =====================================================================================================================
class _WLayerNorm(nn.LayerNorm):
    def forward(self, x):
        return super().forward(x.float()).type(x.dtype)


class _WLinear(nn.Linear):
    def forward(self, x):
        return F.linear(x, self.weight.to(x.dtype), None if self.bias is None else self.bias.to(x.dtype))


class _WConv1d(nn.Conv1d):
    def _conv_forward(self, x, weight, bias):
        return super()._conv_forward(x, weight.to(x.dtype), None if bias is None else bias.to(x.dtype))


class _MultiHeadAttention(nn.Module):
    def __init__(self, n_state: int, n_head: int):
        super().__init__()
        self.n_head = n_head
        self.query = _WLinear(n_state, n_state)
        self.key = _WLinear(n_state, n_state, bias=False)
        self.value = _WLinear(n_state, n_state)
        self.out = _WLinear(n_state, n_state)

    def forward(self, x, xa=None, mask=None, kv_cache=None):
        q, k, v = self.query(x), self.key(x), self.value(x)
        n_batch, n_ctx, n_state = q.shape
        scale = (n_state // self.n_head) ** -0.25
        q = q.view(*q.shape[:2], self.n_head, -1).permute(0, 2, 1, 3) * scale
        k = k.view(*k.shape[:2], self.n_head, -1).permute(0, 2, 3, 1) * scale
        v = v.view(*v.shape[:2], self.n_head, -1).permute(0, 2, 1, 3)
        qk = (q @ k).float()
        w = F.softmax(qk, dim=-1).to(q.dtype)
        return self.out((w @ v).permute(0, 2, 1, 3).flatten(start_dim=2)), qk.detach()


class _ResidualAttentionBlock(nn.Module):
    def __init__(self, n_state: int, n_head: int):
        super().__init__()
        self.attn = _MultiHeadAttention(n_state, n_head)
        self.attn_ln = _WLayerNorm(n_state)
        self.mlp = nn.Sequential(_WLinear(n_state, 4 * n_state), nn.GELU(), _WLinear(4 * n_state, n_state))
        self.mlp_ln = _WLayerNorm(n_state)

    def forward(self, x, xa=None, mask=None, kv_cache=None):
        x = x + self.attn(self.attn_ln(x), mask=mask, kv_cache=kv_cache)[0]
        return x + self.mlp(self.mlp_ln(x))


def _sinusoids(length, channels, max_timescale=10000):
    inc = np.log(max_timescale) / (channels // 2 - 1)
    inv = torch.exp(-inc * torch.arange(channels // 2))
    t = torch.arange(length)[:, np.newaxis] * inv[np.newaxis, :]
    return torch.cat([torch.sin(t), torch.cos(t)], dim=1)


class AudioEncoder(nn.Module):
    def __init__(self, n_mels: int, n_ctx: int, n_state: int, n_head: int, n_layer: int):
        super().__init__()
        self.conv1 = _WConv1d(n_mels, n_state, kernel_size=3, padding=1)
        self.conv2 = _WConv1d(n_state, n_state, kernel_size=3, stride=2, padding=1)
        self.register_buffer("positional_embedding", _sinusoids(n_ctx, n_state))
        self.blocks = nn.ModuleList([_ResidualAttentionBlock(n_state, n_head) for _ in range(n_layer)])
        self.ln_post = _WLayerNorm(n_state)

    def forward(self, x):
        x = F.gelu(self.conv1(x))
        x = F.gelu(self.conv2(x))
        x = x.permute(0, 2, 1)
        assert x.shape[1:] == self.positional_embedding.shape, "incorrect audio shape"
        x = (x + self.positional_embedding).to(x.dtype)
        for block in self.blocks:
            x = block(x)
        return self.ln_post(x)


class _Whisper(nn.Module):
    def __init__(self, dims: dict):
        super().__init__()
        self.dims = types.SimpleNamespace(**dims)
        self.encoder = AudioEncoder(dims["n_mels"], dims["n_audio_ctx"], dims["n_audio_state"], dims["n_audio_head"], dims["n_audio_layer"])


def _whisper_load_model(name: str, device=None, download_root=None, in_memory: bool = False):
    """whisper.load_model on a checkpoint path: {'dims': {...}, 'model_state_dict': {...}} (the official .pt layout)."""
    ck = torch.load(name, map_location="cpu")
    model = _Whisper(ck["dims"])
    sd = {k: v for k, v in ck["model_state_dict"].items() if k.startswith("encoder.")}
    model.load_state_dict(sd, strict=True)
    return model.to(device) if device else model


def _whisper_load_audio(path: str, sr: int = 16000):
    from scipy.io import wavfile
    rate, data = wavfile.read(path)
    assert rate == sr and data.dtype == np.int16, "the stand-in reads 16 kHz int16 WAV only (whisper: ffmpeg -> s16le / 32768)"
    return data.flatten().astype(np.float32) / 32768.0


def _whisper_pad_or_trim(array, length: int = 480000, *, axis: int = -1):
    if torch.is_tensor(array):
        if array.shape[axis] > length:
            array = array.index_select(dim=axis, index=torch.arange(length, device=array.device))
        if array.shape[axis] < length:
            pad = [(0, 0)] * array.ndim
            pad[axis] = (0, length - array.shape[axis])
            array = F.pad(array, [p for sizes in pad[::-1] for p in sizes])
        return array
    if array.shape[axis] > length:
        array = array.take(indices=range(length), axis=axis)
    if array.shape[axis] < length:
        pad = [(0, 0)] * array.ndim
        pad[axis] = (0, length - array.shape[axis])
        array = np.pad(array, pad)
    return array


def _mel_filters_librosa(n_mels: int) -> torch.Tensor:
    """librosa.filters.mel(sr=16000, n_fft=400, n_mels) as shipped in whisper/assets/mel_filters.npz — taken from
    transformers.audio_utils.mel_filter_bank (slaney/slaney), an implementation independent of the oracle's."""
    from transformers.audio_utils import mel_filter_bank
    return torch.from_numpy(mel_filter_bank(201, n_mels, 0.0, 8000.0, 16000, norm="slaney", mel_scale="slaney")).float().t().contiguous()


def _whisper_log_mel_spectrogram(audio, n_mels: int = 80, padding: int = 0, device=None):
    if not torch.is_tensor(audio):
        audio = torch.from_numpy(audio)
    if device is not None:
        audio = audio.to(device)
    if padding > 0:
        audio = F.pad(audio, (0, padding))
    window = torch.hann_window(400).to(audio.device)
    stft = torch.stft(audio, 400, 160, window=window, return_complex=True)
    magnitudes = stft[..., :-1].abs() ** 2
    mel_spec = _mel_filters_librosa(n_mels).to(audio.device) @ magnitudes
    log_spec = torch.clamp(mel_spec, min=1e-10).log10()
    log_spec = torch.maximum(log_spec, log_spec.max() - 8.0)
    return (log_spec + 4.0) / 4.0


def _kaldiio_module() -> types.ModuleType:
    """kaldiio.load_mat(path) -> (rate, int16 samples): the stand-in reads a 16 kHz int16 WAV instead of an ark entry."""
    m = types.ModuleType("kaldiio")

    def load_mat(path):
        from scipy.io import wavfile
        rate, data = wavfile.read(path)
        return rate, data
    m.load_mat = load_mat
    return m


def _whisper_module() -> types.ModuleType:
    m = types.ModuleType("whisper")
    m.load_model, m.load_audio, m.pad_or_trim, m.log_mel_spectrogram = (_whisper_load_model, _whisper_load_audio, _whisper_pad_or_trim,
                                                                       _whisper_log_mel_spectrogram)
    m.model = types.ModuleType("whisper.model")
    m.model.AudioEncoder = AudioEncoder
    return m


# =====================================================================================================================
def _load_by_path(name: str, path: str) -> types.ModuleType:
    spec = importlib.util.spec_from_file_location(name, path)
    mod = importlib.util.module_from_spec(spec)
    sys.modules[name] = mod
    spec.loader.exec_module(mod)
    return mod


def install(extra_stubs: Iterable[str] = ()) -> None:
    """Make `import slam_llm...` resolve to the reference's src with the stand-ins in place."""
    if not reference_available():
        raise RuntimeError("SLAM_LLM_REFERENCE does not name a checkout of the original SLAM-LLM project: the reference-run fixtures are "
                           "committed under tests/golden/")
    loaded = sys.modules.get("slam_llm")
    if loaded is not None and not getattr(loaded, "__file__", "").startswith(REFERENCE_SRC):
        raise RuntimeError("the repo's slam_llm mirror is already imported in this process; use a dedicated process")
    # transformers probes optional packages (soundfile, ...) with importlib.util.find_spec when its sub-modules are first imported:
    # import what the reference needs BEFORE the stand-ins exist so that transformers sees the truth (absent)
    import transformers.models.llama.modeling_llama  # noqa: F401
    import transformers.audio_utils  # noqa: F401
    from transformers import AutoModelForCausalLM, AutoTokenizer, AutoConfig, AutoModel, AutoModelForSeq2SeqLM, T5ForConditionalGeneration  # noqa: F401
    from transformers import LlamaTokenizer, default_data_collator  # noqa: F401
    from transformers.data import DataCollatorForSeq2Seq  # noqa: F401
    from transformers.utils import import_utils as _iu
    assert not _iu.is_peft_available() and not _iu.is_soundfile_available()           # lru_cached: stays False once the stand-ins exist
    sys.path[:] = [p for p in sys.path if os.path.abspath(p) != os.path.join(ROOT, "src")]
    sys.path.insert(0, REFERENCE_SRC)
    for mk in (_peft_module, _whisper_module, _kaldiio_module):
        m = mk()
        m.__spec__ = importlib.machinery.ModuleSpec(m.__name__, None)
        sys.modules.setdefault(m.__name__, m)
    if "omegaconf" not in sys.modules:
        try:
            importlib.import_module("omegaconf")
        except ImportError:
            _load_by_path("omegaconf", os.path.join(ROOT, "src", "slam_llm", "_compat", "omegaconf_shim.py"))
    for name in ("soundfile", "deepspeed", "deepspeed.utils", "deepspeed.utils.zero_to_fp32") + tuple(extra_stubs):
        if name not in sys.modules:
            try:
                importlib.import_module(name)
            except ImportError:
                stub = types.ModuleType(name)
                stub.__spec__ = importlib.machinery.ModuleSpec(name, None)
                sys.modules[name] = stub
    z = sys.modules["deepspeed.utils.zero_to_fp32"]
    for fn in ("get_fp32_state_dict_from_zero_checkpoint", "convert_zero_checkpoint_to_fp32_state_dict", "load_state_dict_from_zero_checkpoint"):
        if not hasattr(z, fn):
            setattr(z, fn, lambda *a, **kw: (_ for _ in ()).throw(NotImplementedError("deepspeed is absent")))


def reference_modules():
    install()
    mods = {}
    for name in ("slam_llm.models.projector", "slam_llm.utils.metric", "slam_llm.models.encoder", "slam_llm.utils.config_utils",
                 "slam_llm.models.slam_model", "slam_llm.datasets.speech_dataset", "slam_llm.datasets.speech_dataset_large"):
        mods[name.rsplit(".", 1)[-1]] = importlib.import_module(name)
    for m in mods.values():
        assert m.__file__.startswith(REFERENCE_SRC), m.__file__
    return mods


# =====================================================================================================================
# small helpers shared by the fixture generators
# =====================================================================================================================
class CharTokenizer:
    """Deterministic byte-level stand-in for the HF tokenizer object the dataset calls (.encode, eos/pad/bos ids)."""

    def __init__(self, vocab: int):
        self.vocab = vocab
        self.bos_token_id, self.eos_token_id = 1, 2
        self.pad_token_id = self.eos_token_id                                          # slam_model.py:64 `tokenizer.pad_token_id = tokenizer.eos_token_id`

    def encode(self, text: str) -> List[int]:
        return [self.bos_token_id] + [3 + (b * 7 + i) % (self.vocab - 3) for i, b in enumerate(text.encode("utf-8"))]

    def __call__(self, text, **kw):
        ids = self.encode(text)
        return types.SimpleNamespace(input_ids=ids)

    def batch_decode(self, ids, **kw):
        return ["" for _ in ids]


def write_wav(path: str, pcm_int16: np.ndarray) -> None:
    from scipy.io import wavfile
    wavfile.write(path, 16000, pcm_int16.astype(np.int16))


def whisper_checkpoint(enc_w: Dict[str, torch.Tensor], n_mels: int, n_ctx: int, d: int, heads: int, layers: int) -> dict:
    """openai-whisper .pt layout (dims + model_state_dict) holding the given AudioEncoder weights."""
    dims = dict(n_mels=n_mels, n_audio_ctx=n_ctx, n_audio_state=d, n_audio_head=heads, n_audio_layer=layers,
                n_vocab=8, n_text_ctx=8, n_text_state=d, n_text_head=heads, n_text_layer=0)
    return {"dims": dims, "model_state_dict": {"encoder." + k: v.clone() for k, v in enc_w.items()}}
