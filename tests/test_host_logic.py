"""Host-side logic that needs no GPU: config shims, plugin loaders, the dataset/collator batch contract, label-row
selection, LR schedule, the train-loop control flow (with a mock model), trainable-only checkpoints, and the
world_size-2 data-parallel arithmetic over gloo."""
import json
import math
import os
import sys
import types
import wave

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

import slam_llm  # noqa: E402,F401  (installs the offline shims for hydra / omegaconf / whisper)
from omegaconf import DictConfig, ListConfig, OmegaConf  # noqa: E402


# ------------------------------------------------------------------------------------------------- config surface
def test_omegaconf_merge_and_access_like_the_recipes():
    from dataclasses import dataclass, field
    from typing import List, Optional

    @dataclass
    class Peft:
        r: int = 8
        target_modules: List = field(default_factory=lambda: ["q_proj", "v_proj"])

    @dataclass
    class Train:
        lr: float = 1e-4
        use_peft: bool = False
        peft_config: Peft = field(default_factory=Peft)

    @dataclass
    class Run:
        train_config: Train = field(default_factory=Train)
        ckpt_path: Optional[str] = None

    cli = OmegaConf.from_dotlist(["++train_config.use_peft=true", "++train_config.peft_config.r=16", "++train_config.lr=5e-5",
                                  "++train_config.peft_config.target_modules=[q_proj,k_proj]", "++metric=acc"])
    cfg = OmegaConf.merge(Run(), cli)
    assert isinstance(cfg, DictConfig) and cfg.train_config.use_peft is True and cfg.train_config.peft_config.r == 16
    assert cfg.train_config.lr == pytest.approx(5e-5) and cfg.get("metric") == "acc" and cfg.get("nope", 3) == 3
    assert isinstance(cfg.train_config.peft_config.target_modules, ListConfig)
    assert OmegaConf.to_container(cfg.train_config.peft_config) == {"r": 16, "target_modules": ["q_proj", "k_proj"]}
    OmegaConf.set_struct(cfg, False)
    del cfg["train_config"]
    assert "train_config" not in cfg and dict(**cfg)["ckpt_path"] is None
    with pytest.raises(AttributeError):
        _ = cfg.missing_key


def test_hydra_main_parses_recipe_style_argv(tmp_path, monkeypatch):
    import hydra
    conf = tmp_path / "conf"
    conf.mkdir()
    (conf / "prompt.yaml").write_text("dataset_config:\n  prompt: 'Transcribe speech to text. '\n")
    script = tmp_path / "entry.py"
    script.write_text("import hydra\n@hydra.main(config_name=None, version_base=None)\ndef main(cfg):\n    return cfg\n")
    from slam_llm.utils.dataset_utils import load_module_from_py_file
    mod = load_module_from_py_file(str(script))
    monkeypatch.setattr(sys, "argv", ["entry.py", "--config-path", "conf", "--config-name", "prompt.yaml", f"hydra.run.dir={tmp_path}/out",
                                      "++model_config.llm_dim=2048", "++train_config.enable_ddp=true", "++dataset_config.input_type=mel"])
    cfg = mod.main()
    assert cfg.dataset_config.prompt == "Transcribe speech to text. " and cfg.dataset_config.input_type == "mel"
    assert cfg.model_config.llm_dim == 2048 and cfg.train_config.enable_ddp is True and os.path.isdir(tmp_path / "out")


def test_plugin_loaders_follow_reference_error_behaviour(tmp_path):
    from slam_llm.utils.model_utils import get_custom_model_factory
    import logging
    f = tmp_path / "m.py"
    f.write_text("def model_factory(train_config, model_config, **kw):\n    return 'model', 'tok'\n")
    fac = get_custom_model_factory(DictConfig({"file": f"{f}:model_factory"}), logging.getLogger())
    assert fac(None, None) == ("model", "tok")
    with pytest.raises(ValueError):
        get_custom_model_factory(DictConfig({"file": "notpy.txt:model_factory"}), logging.getLogger())
    with pytest.raises(FileNotFoundError):
        get_custom_model_factory(DictConfig({"file": str(tmp_path / "nope.py") + ":model_factory"}), logging.getLogger())
    with pytest.raises(AttributeError):
        get_custom_model_factory(DictConfig({"file": f"{f}:missing"}), logging.getLogger())


def test_dataset_files_load_as_path_plugins():
    """Recipes address the datasets by FILE PATH (`dataset_config.file=.../speech_dataset.py:get_speech_dataset`, reference
    utils/dataset_utils.py:14-57): the files must import cleanly when executed outside their package."""
    from slam_llm.utils.dataset_utils import load_module_from_py_file, _plugin_factory
    base = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "src", "slam_llm", "datasets")
    for name in ("speech_dataset.py", "speech_dataset_large.py"):
        mod = load_module_from_py_file(os.path.join(base, name))
        assert callable(mod.get_speech_dataset)
        assert callable(_plugin_factory(os.path.join(base, name) + ":get_speech_dataset"))


def test_zero_pool_hands_out_zeroed_disjoint_slices():
    """Scratch for the split-K thin products (engine._ZeroPool): one memset per pass, slices in call order, grows to the largest pass."""
    from slam_llm_b200.engine import _ZeroPool
    pool = _ZeroPool()
    pool.begin("cpu")
    first = pool.take(4, 8, "cpu")                      # nothing reserved yet: falls back to a fresh zero tensor and records the need
    assert first.shape == (4, 8) and float(first.abs().sum()) == 0.0
    first.fill_(1.0)
    for _ in range(2):
        pool.begin("cpu")
        a, b = pool.take(4, 8, "cpu"), pool.take(2, 8, "cpu")
        assert float(a.abs().sum()) == 0.0 and float(b.abs().sum()) == 0.0 and a.data_ptr() != b.data_ptr()
        a.fill_(2.0); b.fill_(3.0)                      # dirty them: the next begin() must clear the pool again
    assert pool.buf.numel() >= 48 and a.data_ptr() == pool.buf.data_ptr()


def test_generate_peft_config():
    from slam_llm.utils.config_utils import generate_peft_config
    tc = DictConfig({"peft_config": {"peft_method": "lora", "r": 16, "lora_alpha": 32, "target_modules": ["q_proj", "v_proj"], "bias": "none",
                                     "task_type": "CAUSAL_LM", "lora_dropout": 0.05, "inference_mode": False}})
    c = generate_peft_config(tc)
    assert (c.r, c.alpha, c.targets, c.scaling) == (16, 32, ("q_proj", "v_proj"), 2.0)
    tc.peft_config.peft_method = "prefix"
    with pytest.raises(NotImplementedError):
        generate_peft_config(tc)


# ------------------------------------------------------------------------------------------------- batch contract
class FakeTokenizer:
    pad_token_id = 0
    eos_token_id = 2

    def encode(self, text):
        return [1] + [3 + (ord(c) % 50) for c in text]


def _write_wav(path, seconds, seed):
    rng = np.random.default_rng(seed)
    pcm = (rng.standard_normal(int(16000 * seconds)) * 3000).astype(np.int16)
    with wave.open(str(path), "wb") as w:
        w.setnchannels(1); w.setsampwidth(2); w.setframerate(16000); w.writeframes(pcm.tobytes())


@pytest.mark.parametrize("gpu_frontend", [True, False])
def test_dataset_and_collator_contract(tmp_path, gpu_frontend):
    from slam_llm.datasets.speech_dataset import get_speech_dataset
    rows = []
    for i, (sec, text) in enumerate([(1.0, "hello world"), (2.5, "a"), (0.7, "the quick brown fox")]):
        _write_wav(tmp_path / f"{i}.wav", sec, i)
        rows.append({"key": f"utt{i}", "source": str(tmp_path / f"{i}.wav"), "target": text})
    (tmp_path / "train.jsonl").write_text("\n".join(json.dumps(r) for r in rows))
    cfg = DictConfig({"train_data_path": str(tmp_path / "train.jsonl"), "val_data_path": str(tmp_path / "train.jsonl"), "input_type": "mel",
                      "mel_size": 80, "prompt": "Transcribe speech to text. ", "b200_gpu_frontend": gpu_frontend})
    ds = get_speech_dataset(cfg, FakeTokenizer(), "train")
    items = [ds[i] for i in range(3)]
    assert all(it["audio_length"] == 300 for it in items)            # pad_or_trim to 30 s -> 3000 frames -> 1500 -> 300
    b = ds.collator(items)
    B, S = b["input_ids"].shape
    assert B == 3 and b["labels"].shape == (3, S) and b["attention_mask"].dtype == torch.bool
    if gpu_frontend:
        assert b["audio_mel"] is None and b["audio_pcm"].shape == (3, 480000) and b["audio_pcm"].dtype == torch.float32
    else:
        assert b["audio_pcm"] is None and b["audio_mel"].shape == (3, 3000, 80)
    for i, it in enumerate(items):
        n = len(it["input_ids"])
        p = it["audio_length"] + it["prompt_length"]
        left = max(x["audio_length"] + x["prompt_length"] for x in items) - p
        assert b["attention_mask"][i].sum().item() == n and not b["attention_mask"][i, :left].any()       # left pad on the prompt side
        assert b["modality_mask"][i, left:left + 300].all() and b["modality_mask"][i].sum().item() == 300
        assert (b["input_ids"][i, left:left + 300] == -1).all()
        lab = b["labels"][i]
        assert (lab[: left + p] == -100).all() and (lab[left + p: left + n] >= 0).all() and (lab[left + n:] == -100).all()
        assert lab[left + n - 1].item() == FakeTokenizer.eos_token_id
    # label rows (HF shift): row r predicts labels[r+1]
    from slam_llm_b200.engine import SlamStepB200
    rows_idx, tgts = SlamStepB200.label_rows(b["labels"])
    shifted = torch.full_like(b["labels"], -100)
    shifted[:, :-1] = b["labels"][:, 1:]
    assert rows_idx.dtype == torch.int32 and torch.equal(tgts, shifted.reshape(-1)[rows_idx.long()]) and (tgts != -100).all()
    assert rows_idx.numel() == (shifted != -100).sum().item()
    all_rows, all_t = SlamStepB200.label_rows(b["labels"], full=True)
    assert all_rows.numel() == B * S and (all_t == -100).sum().item() == B * S - rows_idx.numel()


def test_whisper_shim_logmel_matches_hf_feature_extractor(tmp_path):
    import whisper
    from transformers import WhisperFeatureExtractor
    _write_wav(tmp_path / "a.wav", 1.3, 5)
    audio = whisper.load_audio(str(tmp_path / "a.wav"))
    assert audio.dtype == np.float32 and audio.shape[0] == int(16000 * 1.3)
    mel = whisper.log_mel_spectrogram(whisper.pad_or_trim(audio), n_mels=80)
    ref = WhisperFeatureExtractor(feature_size=80)(audio, sampling_rate=16000, return_tensors="pt").input_features[0]
    assert mel.shape == (80, 3000) and (mel - ref).abs().max().item() < 5e-5


# ------------------------------------------------------------------------------------------------- train loop control flow
class _MockModel(torch.nn.Module):
    def __init__(self):
        super().__init__()
        self.w = torch.nn.Parameter(torch.zeros(4))
        self.calls = 0

    def forward(self, x=None, **kw):
        self.calls += 1
        loss = ((self.w - x.float().mean(0)) ** 2).sum()
        return types.SimpleNamespace(loss=loss, logits=None), torch.tensor(0.5)


class _CountingSGD(torch.optim.SGD):
    steps = 0

    def step(self, closure=None):
        type(self).steps += 1
        return super().step(closure)


def _train_cfg(**over):
    base = dict(enable_fsdp=False, enable_ddp=False, use_fp16=False, num_epochs=1, batching_strategy="custom", validation_interval=1000,
                run_validation=False, save_model=False, use_peft=True, model_name="m", output_dir="/tmp/x", run_test_during_validation=False)
    base.update(over)
    return DictConfig(base)


def test_train_loop_grad_accumulation_and_lr_break(monkeypatch):
    from slam_llm.utils import train_utils
    monkeypatch.setattr(train_utils, "_device", lambda tc, lr: torch.device("cpu"))
    data = [{"x": torch.randn(2, 4)} for _ in range(7)]
    model = _MockModel()
    _CountingSGD.steps = 0
    opt = _CountingSGD(model.parameters(), lr=0.1)
    sched = torch.optim.lr_scheduler.LambdaLR(opt, lr_lambda=lambda s: 1.0)
    res = train_utils.train(model, data, None, None, opt, sched, 3, _train_cfg(), DictConfig({"use_wandb": False, "log_interval": 5}))
    assert model.calls == 7 and _CountingSGD.steps == 3           # steps 3, 6 and the last (7th) batch of a non-dynamic loader
    assert set(res) >= {"avg_train_prep", "avg_train_loss", "avg_train_acc", "avg_epoch_time", "avg_checkpoint_time"}
    assert float(res["avg_train_acc"]) == pytest.approx(0.5 / 3)   # acc is divided by gradient_accumulation_steps (D3)
    assert float(res["avg_train_prep"]) == pytest.approx(math.exp(float(res["avg_train_loss"])), rel=1e-5)
    # the loop stops as soon as the schedule reaches lr == 0 (finetune.py:253-260 + train_utils.py:140-141)
    model2 = _MockModel()
    _CountingSGD.steps = 0
    opt2 = _CountingSGD(model2.parameters(), lr=0.1)
    warm, total = 1, 3
    sched2 = torch.optim.lr_scheduler.LambdaLR(opt2, lr_lambda=lambda s: min(s / warm, 1) if s < warm else max(0.0, 1 - (s - warm) / (total - warm)))
    train_utils.train(model2, data, None, None, opt2, sched2, 1, _train_cfg(), DictConfig({"use_wandb": False, "log_interval": 5}))
    assert _CountingSGD.steps == 3 and model2.calls == 3


def test_validation_and_checkpoint_in_reference_format(monkeypatch, tmp_path):
    from slam_llm.utils import train_utils
    monkeypatch.setattr(train_utils, "_device", lambda tc, lr: torch.device("cpu"))
    data = [{"x": torch.randn(2, 4)} for _ in range(4)]
    model = _MockModel()
    model.frozen = torch.nn.Parameter(torch.ones(3), requires_grad=False)
    opt = torch.optim.SGD([model.w], lr=0.1)
    cfg = _train_cfg(run_validation=True, validation_interval=2, save_model=True, output_dir=str(tmp_path), model_name="asr")
    res = train_utils.train(model, data, data[:2], types.SimpleNamespace(batch_decode=lambda *a, **k: []), opt, None, 1, cfg,
                            DictConfig({"use_wandb": False, "log_interval": 5}))
    assert "avg_eval_loss" in res
    saved = sorted(os.listdir(tmp_path))
    assert saved and saved[0].startswith("asr_epoch_1_step_2")
    sd = torch.load(tmp_path / saved[0] / "model.pt")
    assert set(sd) == {"w"}                                        # trainable-only (checkpoint_handler.py:185-201)


# ------------------------------------------------------------------------------------------------- multi-process (gloo)
def _ddp_worker(rank, world, port, q):
    import torch.distributed as dist
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world), LOCAL_RANK=str(rank))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    from torch.utils.data import DistributedSampler
    # (1) units shard with no overlap; (2) the one collective = all-reduce of the flat grad buffer, mean taken by grad_div
    ids = list(DistributedSampler(list(range(10)), num_replicas=world, rank=rank, shuffle=False))
    flat_grad = torch.full((5,), float(rank + 1))
    dist.all_reduce(flat_grad)
    param = torch.tensor([float(rank)] * 3)
    dist.broadcast(param, src=0)
    q.put((rank, ids, (flat_grad / world).tolist(), param.tolist()))
    dist.destroy_process_group()


def test_world_size_2_gloo_data_parallel_arithmetic():
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 29500 + os.getpid() % 500
    procs = [ctx.Process(target=_ddp_worker, args=(r, 2, port, q)) for r in range(2)]
    [p.start() for p in procs]
    out = sorted(q.get(timeout=120) for _ in range(2))
    [p.join(60) for p in procs]
    assert not (set(out[0][1]) & set(out[1][1])) and len(out[0][1]) == len(out[1][1]) == 5
    assert out[0][2] == out[1][2] == [1.5] * 5                      # mean of per-rank gradients
    assert out[0][3] == out[1][3] == [0.0] * 3                      # trainables broadcast from rank 0


class _JoinMock(_MockModel):
    """Stand-in with the DDP surface of slam_model: grads all-reduced in backward on sync micro-steps, shadow_backward for Join."""
    ddp_world_size, ddp_sync = 2, True

    def __init__(self):
        super().__init__()
        self.w.register_hook(self._hook)
        self.shadows = 0

    def _hook(self, g):
        import torch.distributed as dist
        if self.ddp_sync:
            g = g.clone()
            if self.w.grad is not None:            # accumulated micro-steps ride along with the last one (flat-buffer all-reduce)
                g += self.w.grad
                self.w.grad.zero_()
            dist.all_reduce(g)
        return g

    def shadow_backward(self):
        import torch.distributed as dist
        self.shadows += 1
        if self.w.grad is None:
            self.w.grad = torch.zeros_like(self.w)
        if self.ddp_sync:
            dist.all_reduce(self.w.grad)


def _join_worker(rank, world, port, q):
    import torch.distributed as dist
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world), LOCAL_RANK=str(rank))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    from slam_llm.utils import train_utils
    train_utils._device = lambda tc, lr: torch.device("cpu")
    torch.manual_seed(rank)
    data = [{"x": torch.randn(2, 4)} for _ in range(5 if rank == 0 else 2)]      # dynamic-frame batching: unequal step counts
    model = _JoinMock()
    _CountingSGD.steps = 0
    opt = _CountingSGD(model.parameters(), lr=0.1)
    res = train_utils.train(model, iter(data), None, None, opt, None, 1, _train_cfg(enable_ddp=True, batching_strategy="dynamic"),
                            DictConfig({"use_wandb": False, "log_interval": 5}), rank=rank, local_rank=rank)
    q.put((rank, model.calls, model.shadows, _CountingSGD.steps, model.w.detach().tolist(), float(res["avg_train_loss"])))
    dist.destroy_process_group()


def test_world_size_2_gloo_join_on_uneven_dynamic_batches():
    """Reference: the epoch runs under torch's Join (utils/train_utils.py:91) because dynamic-frame batching gives ranks different
    numbers of batches.  Here: the rank that runs dry keeps stepping with zero gradients until every rank is exhausted."""
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 30100 + os.getpid() % 500
    procs = [ctx.Process(target=_join_worker, args=(r, 2, port, q)) for r in range(2)]
    [p.start() for p in procs]
    out = sorted(q.get(timeout=180) for _ in range(2))
    [p.join(60) for p in procs]
    (r0, calls0, sh0, steps0, w0, _), (r1, calls1, sh1, steps1, w1, _) = out
    assert (calls0, sh0, calls1, sh1) == (5, 0, 2, 3)               # rank 1 shadows the 3 steps it has no data for
    assert steps0 == steps1 == 5                                    # same number of optimizer steps everywhere
    assert w0 == w1                                                 # replicas stay identical


def test_reference_arm_only_rank0_works(monkeypatch, capsys):
    sys.path.insert(0, ROOT)
    import bench
    monkeypatch.setenv("RANK", "1"); monkeypatch.setenv("WORLD_SIZE", "2"); monkeypatch.setenv("LOCAL_RANK", "1")
    bench.run_reference(types.SimpleNamespace(workload="c3", steps=1, warmup=0, gpus=2))
    assert capsys.readouterr().out == ""                            # non-zero ranks exit without work or output


def test_bench_gemm_traffic_parser_and_fallback(tmp_path, monkeypatch):
    """roofline.traffic comes from an ncu child process of bench.py: the CSV parser keeps this library's GEMM launches only and sums read +
    write bytes per launch id; without ncu (or when the child fails) the measurement reports why instead of raising."""
    sys.path.insert(0, ROOT)
    import bench
    log = tmp_path / "m.csv"
    log.write_text(
        '==PROF== Connected to process 1\n'
        '"ID","Process ID","Process Name","Host Name","Kernel Name","Context","Stream","Block Size","Grid Size","Device","CC","Section Name","Metric Name","Metric Unit","Metric Value"\n'
        '"0","1","python","h","slam::logmel_kernel(float *)","1","7","(128, 1, 1)","(1, 1, 1)","0","10.0","s","dram__bytes_read.sum","Mbyte","5.0"\n'
        '"1","1","python","h","void slam::gemm_tcgen05_pair_kernel<(int)192, (int)2>(CUtensorMap_st)","1","7","(384, 1, 1)","(148, 1, 1)","0","10.0","s","dram__bytes_read.sum","Mbyte","100.5"\n'
        '"1","1","python","h","void slam::gemm_tcgen05_pair_kernel<(int)192, (int)2>(CUtensorMap_st)","1","7","(384, 1, 1)","(148, 1, 1)","0","10.0","s","dram__bytes_write.sum","Kbyte","500"\n'
        '"2","1","python","h","slam::gemm_thin_cluster_kernel(CUtensorMap_st)","1","7","(192, 1, 1)","(104, 1, 1)","0","10.0","s","dram__bytes_read.sum","byte","1,000"\n'
        '"2","1","python","h","slam::gemm_thin_cluster_kernel(CUtensorMap_st)","1","7","(192, 1, 1)","(104, 1, 1)","0","10.0","s","dram__bytes_write.sum","byte","24"\n')
    per = bench.parse_gemm_traffic(str(log))
    assert per == {"1": 100.5e6 + 500e3, "2": 1024.0}
    monkeypatch.setattr("shutil.which", lambda name: None)
    monkeypatch.setattr(os.path, "exists", lambda p, _orig=os.path.exists: False if str(p).endswith("/ncu") else _orig(p))
    assert bench.measure_gemm_traffic("c3") == (None, "ncu not found")


# ------------------------------------------------------------------------------------------------- dynamic-frame batching (config 3)
def test_dynamic_frame_dataset_window_rule_and_right_padding(tmp_path):
    from slam_llm.datasets.speech_dataset_large import get_speech_dataset, window_class
    data_dir = tmp_path / "scp"
    data_dir.mkdir()
    secs = [1.0, 3.2, 0.5, 2.0, 31.0, 1.5, 0.9]                       # the 31 s item exceeds max_audio_length and is skipped
    rows = []
    for i, sec in enumerate(secs):
        _write_wav(data_dir / f"{i}.wav", sec, 100 + i)
        rows.append({"key": f"k{i}", "task": "ASR", "target": "word " * (1 + i % 3), "path": str(data_dir / f"{i}.wav")})
    (data_dir / "multitask.jsonl").write_text("\n".join(json.dumps(r) for r in rows))
    (tmp_path / "prompt.jsonl").write_text(json.dumps({"task": "ASR", "prompt": "Transcribe speech to text."}))
    cfg = DictConfig({"append_info_tasks": [], "multitask_prompt_path": str(tmp_path / "prompt.jsonl"), "train_scp_file_path": str(data_dir),
                      "dev_scp_file_path": str(data_dir), "test_scp_file_path": str(data_dir), "input_type": "mel", "mel_size": 80,
                      "prompt_style": "USER: {}\n ASSISTANT:", "train_max_frame_length": 260, "eval_max_frame_length": 10000, "max_audio_length": 30})
    ds = get_speech_dataset(cfg, FakeTokenizer(), "train")
    batches = list(ds)
    n_items = sum(len(b) for b in batches)
    assert n_items == len(secs) - 1
    for b in batches:                                                  # the reference rule: B * longest <= budget (single items always pass)
        assert len(b) == 1 or len(b) * max(len(x["input_ids"]) for x in b) <= 260
    assert window_class({"input_ids": [0] * 100}, [], 10) is True      # empty buffer always "flushes" (then starts a new one)
    assert window_class({"input_ids": [0] * 100}, [{"input_ids": [0] * 120}], 240) is False
    assert window_class({"input_ids": [0] * 100}, [{"input_ids": [0] * 121}], 240) is True
    big = max(batches, key=len)
    out = ds.collator(big)
    B, S = out["input_ids"].shape
    assert out["audio_mel"] is None and out["audio_pcm"].shape[0] == B and out["audio_pcm"].shape[1] % 320 == 0
    assert out["audio_pcm_lengths"].dtype == torch.int32 and out["audio_pcm_lengths"].tolist() == [x["audio_pcm"].shape[0] for x in big]
    for i, x in enumerate(big):                                        # RIGHT padding only; audio tokens first
        n = len(x["input_ids"])
        assert out["attention_mask"][i, :n].all() and not out["attention_mask"][i, n:].any()
        assert out["modality_mask"][i, : x["audio_length"]].all() and out["modality_mask"][i].sum().item() == x["audio_length"]
        assert x["audio_length"] == ((x["audio_pcm"].shape[0] // 160 + 1) // 2) // 5
        assert (out["labels"][i, n:] == -100).all()
    eval_batches = list(get_speech_dataset(cfg, FakeTokenizer(), "val"))
    assert len(eval_batches) == 1 and len(eval_batches[0]) == len(secs) - 1
