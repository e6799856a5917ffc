"""Inference-side mirror of `VanillaEncoderDecoderTransformerLightning`
(src/model/lightning_model.py:22-277): same constructor arguments for the model / generation
options, `predict_step(batch, batch_idx)`, `on_predict_start` / `on_predict_end` timing report.
Training hooks are out of scope (DESIGN.md §0); the class derives from LightningModule when
Lightning is installed so that `main.py predict` can instantiate it, and from `object` otherwise."""
from __future__ import annotations

import datetime
import json
from pathlib import Path
from timeit import default_timer as timer
from typing import Any

from .decoding.sampling import TranslationInferenceSampling
from .decoding.speculative_decoding import TranslationInferenceBeamSearchSpeculative, TranslationInferenceGreedySpeculative
from .decoding.standard_decoding import TranslationInferenceBeamSearch, TranslationInferenceGreedy
from .model import B200Transformer
from .weights import ModelConfig, random_init_state_dict

try:
    from pytorch_lightning import LightningModule as _Base
except Exception:  # pragma: no cover
    _Base = object


class VanillaEncoderDecoderTransformerLightning(_Base):
    def __init__(self, src_tokenizer=None, tgt_tokenizer=None, embedding_dim: int = 128, feedforward_dim: int = 256,
                 num_encoder_layers: int = 3, num_decoder_layers: int = 3, num_heads: int = 4, dropout_rate: float = 0.0,
                 activation: str = "relu", share_embeddings: bool = False, generation: str = "greedy_speculative",
                 beam_size: int = 0, max_len: int = 0, n_drafts: int = 0, draft_len: int = 0, smart_drafts_mode: bool = True,
                 report_prediction_time: bool = True, report_prediction_file: str | None = None,
                 state_dict: dict | None = None, precision: str = "bf16", device: int = 0, seed: int = 0,
                 batches_in_flight: int = 1, tgt_test_path: str | None = None, n_samples: int = 1, temperature: float = 1.0,
                 top_k: int = 0, sampling_seed: int = 0, **_unused):
        if _Base is not object:
            super().__init__()
        assert src_tokenizer is not None, "source tokenizer not provided"
        assert tgt_tokenizer is not None, "target tokenizer not provided"
        assert activation == "relu", "only the relu activation of the shipped configs is implemented"
        self.src_tokenizer, self.tgt_tokenizer = src_tokenizer, tgt_tokenizer
        self.generation, self.beam_size, self.max_len = generation, beam_size, max_len
        self.n_drafts, self.draft_len, self.smart_drafts_mode = n_drafts, draft_len, smart_drafts_mode
        # generation="sampling" only (DESIGN.md section 15)
        self.n_samples, self.temperature, self.top_k, self.sampling_seed = n_samples, temperature, top_k, sampling_seed
        self.report_prediction_time, self.report_prediction_file = report_prediction_time, report_prediction_file
        self.src_pad_token_i, self.tgt_pad_token_i = src_tokenizer.pad_token_idx, tgt_tokenizer.pad_token_idx
        self.tgt_bos_token_i, self.tgt_eos_token_i = tgt_tokenizer.bos_token_idx, tgt_tokenizer.eos_token_idx
        cfg = ModelConfig(src_vocab_size=src_tokenizer.n_tokens, tgt_vocab_size=tgt_tokenizer.n_tokens,
                          embedding_dim=embedding_dim, feedforward_dim=feedforward_dim,
                          num_encoder_layers=num_encoder_layers, num_decoder_layers=num_decoder_layers,
                          num_heads=num_heads, share_embeddings=share_embeddings,
                          src_pad_token_idx=self.src_pad_token_i, tgt_pad_token_idx=self.tgt_pad_token_i)
        weights = state_dict if state_dict is not None else random_init_state_dict(cfg, seed)
        # `batches_in_flight` > 1: one engine (weights, workspace, stream, CUDA graphs) per batch decoded concurrently by
        # `predict_batches` (pipeline.py); `model` / `generator` stay the first pair, which `predict_step` uses
        self.models = [B200Transformer(cfg, weights, precision=precision, device=device) for _ in range(max(1, batches_in_flight))]
        self.model = self.models[0]
        self.generators = [self._create_generator(m) for m in self.models]
        self.generator = self.generators[0]
        self._in_flight = None
        self.device_index = device
        self.prediction_start_time = None
        self.batch_size = None
        # the reference reads both from `self.trainer.datamodule` (lightning_model.py:223-224); without a Lightning trainer
        # they come from the constructor / the first batch
        self.tgt_test_path = tgt_test_path

    def load_checkpoint_state_dict(self, state_dict: dict) -> None:
        """Accepts the `state_dict` of a reference Lightning checkpoint (keys prefixed `model.`)."""
        for m in self.models:
            m.load_state_dict({k: v for k, v in state_dict.items() if "positional_encoding" not in k})

    def _create_generator(self, model=None):
        model = self.model if model is None else model
        if self.generation == "greedy":
            return TranslationInferenceGreedy(model, max_len=self.max_len, pad_token=self.tgt_pad_token_i,
                                              bos_token=self.tgt_bos_token_i, eos_token=self.tgt_eos_token_i)
        if self.generation == "beam_search":
            return TranslationInferenceBeamSearch(model, beam_size=self.beam_size, max_len=self.max_len,
                                                  pad_token=self.tgt_pad_token_i, bos_token=self.tgt_bos_token_i,
                                                  eos_token=self.tgt_eos_token_i)
        if self.generation == "greedy_speculative":
            assert self.draft_len > 0, "Number of speculative tokens must be a positive integer."
            return TranslationInferenceGreedySpeculative(
                model, max_len=self.max_len, draft_len=self.draft_len, n_drafts=self.n_drafts,
                pad_token=self.tgt_pad_token_i, bos_token=self.tgt_bos_token_i, eos_token=self.tgt_eos_token_i,
                replace_token=self.tgt_tokenizer.encoder_dict["c"])
        if self.generation == "beam_search_speculative":
            return TranslationInferenceBeamSearchSpeculative(
                model, vocab_size=self.tgt_tokenizer.n_tokens, max_len=self.max_len, n_best=self.beam_size,
                draft_len=self.draft_len, n_drafts=self.n_drafts, pad_token=self.tgt_pad_token_i,
                bos_token=self.tgt_bos_token_i, eos_token=self.tgt_eos_token_i,
                C_token=self.tgt_tokenizer.encoder_dict["c"], smart_drafts_mode=self.smart_drafts_mode)
        if self.generation == "sampling":
            return TranslationInferenceSampling(model, max_len=self.max_len, n_samples=self.n_samples, pad_token=self.tgt_pad_token_i,
                                                bos_token=self.tgt_bos_token_i, eos_token=self.tgt_eos_token_i,
                                                temperature=self.temperature, top_k=self.top_k, seed=self.sampling_seed)
        options = ", ".join(["beam_search", "greedy", "greedy_speculative", "beam_search_speculative", "sampling"])
        raise ValueError(f"Unknown generation option {self.generation}. Options are {options}.")

    def predict_step(self, batch: Any, batch_idx: int, dataloader_idx: int = 0) -> Any:
        self.batch_size = batch["src_tokens"].shape[0] if self.batch_size is None else self.batch_size
        return self.generator.generate(batch["src_tokens"])

    def predict_batches(self, batches, on_error=None):
        """Predictions of `batches` (dicts with "src_tokens", like `predict_step` gets) in order, with up to
        `batches_in_flight` batches decoded concurrently (pipeline.py).  Same results as calling `predict_step` on each."""
        from .pipeline import InFlightDecoder
        if self._in_flight is None:
            self._in_flight = InFlightDecoder(self.generators, device=self.device_index)
        batches = list(batches)
        if batches and self.batch_size is None:
            self.batch_size = batches[0]["src_tokens"].shape[0]
        dev = self.model.device
        return self._in_flight.map((b["src_tokens"] for b in batches), pre=lambda s: s.to(dev, non_blocking=True), on_error=on_error)

    def predict_queue(self, batches, queue=None, on_error=None):
        """Dynamic sharding of a prediction job over ranks and in-flight engines: every worker of every rank draws the next
        batch index from `queue` (distributed.BatchQueue over all ranks; a local one when None) until it is empty.
        Returns this rank's `(batch index, prediction)` pairs; `distributed.gather_indexed_predictions` puts the job back
        in order.  Same predictions as `predict_step` on each batch: batches are independent."""
        from .distributed import BatchQueue
        from .pipeline import InFlightDecoder
        if self._in_flight is None:
            self._in_flight = InFlightDecoder(self.generators, device=self.device_index)
        batches = list(batches)
        if batches and self.batch_size is None:
            self.batch_size = batches[0]["src_tokens"].shape[0]
        queue = queue if queue is not None else BatchQueue(len(batches), local=True)
        dev = self.model.device

        def next_item():
            i = queue.next()
            return None if i is None else (i, batches[i]["src_tokens"])

        return self._in_flight.drain(next_item, pre=lambda s: s.to(dev, non_blocking=True), on_error=on_error)

    def _counter(self, name: str):
        return sum(getattr(g, name) for g in self.generators)

    def on_predict_start(self) -> None:
        if self.report_prediction_time:
            self.prediction_start_time = timer()

    def on_predict_end(self) -> None:
        if not self.report_prediction_time:
            return
        elapsed = datetime.timedelta(seconds=timer() - self.prediction_start_time)
        n_calls = self._counter("model_calls_num")
        calls = max(n_calls, 1)
        batch_size, tgt_test_path = self.batch_size, self.tgt_test_path
        dm = getattr(getattr(self, "_trainer", None), "datamodule", None)   # under a Lightning trainer: same sources as the reference
        if dm is not None:
            batch_size = getattr(dm, "batch_size", batch_size)
            tgt_test_path = getattr(dm, "tgt_test_path", tgt_test_path)
        # keys and their order as in lightning_model.py:221-235
        report = {"algorithm": self.generation, "batch_size": batch_size, "tgt_test_path": str(tgt_test_path), "max_len": self.max_len,
                  "total_seconds": round(elapsed.total_seconds(), 4), "model_calls": n_calls,
                  "seconds_per_model_call": round(elapsed.total_seconds() / calls, 4)}
        if self.generation in ("greedy_speculative", "beam_search_speculative"):
            report["n_drafts"], report["draft_len"] = self.n_drafts, self.draft_len
            if self.generation == "beam_search_speculative":
                accepted = self._counter("accepted_tokens_num")
                report["accepted_tokens"] = accepted
                report["acceptance_rate"] = round(accepted / max(self._counter("produced_non_pad_tokens"), 1), 4)
        if self.generation == "sampling":
            report["n_samples"], report["temperature"], report["top_k"], report["seed"] = (self.n_samples, self.temperature, self.top_k,
                                                                                          self.sampling_seed)
        report = json.dumps(report)
        print(report)
        if self.report_prediction_file is not None:
            Path(self.report_prediction_file).parent.mkdir(exist_ok=True)
            with open(self.report_prediction_file, "a") as f:
                print(report, file=f)
