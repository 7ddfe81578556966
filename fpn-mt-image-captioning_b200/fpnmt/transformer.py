"""Host-side mirror of /root/reference/models/transformer.py (inference branch, training=False).

Same constructor signatures and call conventions as the reference's `Transformer` / `Encoder` / `Decoder`
(transformer.py:246-374); the arithmetic runs in libfpnmt.so.  The objects hold the variable tree
(`weights`, keys of SURVEY.md Appendix B) and build one `Engine` per (batch, beam, max_len) shape on demand.

Deviations from the reference, by design:
* `training=True` raises (this build is inference-only).
* attention-weight dicts (transformer.py:337-338) are computed on request: `return_attention=True` (keyword-only) runs one
  more teacher-forced pass that also writes them; by default `None` is returned in their place.
"""
from __future__ import annotations

import math
from typing import Dict, Optional, Tuple

import numpy as np
import torch

from . import config as C
from .engine import Engine
from .retinanet import FeatureExtractor
from .weights import init_weights


def get_angles(pos, i, d_model):
    """transformer.py:22-24."""
    angle_rates = 1 / np.power(10000, (2 * (i // 2)) / np.float32(d_model))
    return pos * angle_rates


def raw_positional_encoding(position: int, d_model: int) -> np.ndarray:
    """transformer.py:27-39 (float32 numpy instead of a tf tensor)."""
    angle_rads = get_angles(np.arange(position)[:, np.newaxis], np.arange(d_model)[np.newaxis, :], d_model)
    angle_rads[:, 0::2] = np.sin(angle_rads[:, 0::2])
    angle_rads[:, 1::2] = np.cos(angle_rads[:, 1::2])
    return angle_rads.astype(np.float32)


def positional_encoding(position: int, d_model: int) -> np.ndarray:
    return raw_positional_encoding(position, d_model)[np.newaxis, ...]


def create_look_ahead_mask(size: int) -> np.ndarray:
    """transformer.py:54-56: 1 above the diagonal.  The KV-cached decoder applies it implicitly."""
    return 1.0 - np.tril(np.ones((size, size), np.float32))


class _EngineCache:
    """Engines keyed by shape; all share one weight dict."""

    def __init__(self, weights: Dict[str, np.ndarray], backbone: str, num_layers: int, d_model: int, num_heads: int,
                 dff: int, vocab: int, max_seq_len: int, precision: str, score_mode: str, device: int,
                 start_id: int, end_id: int, use_graphs: bool):
        self.weights, self.backbone = weights, backbone
        self.kw = dict(num_layers=num_layers, d_model=d_model, num_heads=num_heads, dff=dff, vocab=vocab,
                       precision=precision, score_mode=score_mode, device=device, start_id=start_id, end_id=end_id,
                       use_graphs=use_graphs)
        self.max_seq_len = max_seq_len
        self._engines: Dict[Tuple[int, int, int, int], Engine] = {}

    def get(self, batch: int, beam: int, max_len: Optional[int] = None, lanes: int = 1) -> Engine:
        key = (batch, beam, max_len or self.max_seq_len, max(1, lanes))
        if key not in self._engines:
            self._engines[key] = Engine(self.weights, backbone=self.backbone, batch=batch, beam=beam, max_len=key[2],
                                        image_size=C.IMAGE_INPUT_SIZE, lanes=key[3], **self.kw)
        return self._engines[key]


class Encoder:
    """transformer.py:246-303.  `encoder(x, training, mask)` -> (B, 16, d_model)."""

    def __init__(self, num_layers, d_model, num_heads, dff, input_vocab_size, rate=0.1, *, _cache: _EngineCache = None):
        self.d_model, self.num_layers = d_model, num_layers
        self.x_order = [i for i in range(C.NUM_OF_PYRAMIDS) if i != C.BASELINE_INDEX] + [C.BASELINE_INDEX]
        self.pos_encoding = positional_encoding(input_vocab_size, d_model)
        self._cache = _cache
        self.feature_extractor = FeatureExtractor(None, backbone=_cache.backbone, _cache=_cache)

    def __call__(self, x, training, mask):
        if training:
            raise NotImplementedError("inference-only build: training=True is out of scope")
        x = torch.as_tensor(x) if not isinstance(x, torch.Tensor) else x
        return self._cache.get(int(x.shape[0]), 1).encode(x)

    call = __call__


class Decoder:
    """transformer.py:306-341.  `decoder(x, enc_output, training, look_ahead_mask, padding_mask)`.

    Returns (hidden states (B,t,d_model) of the last decoder layer, attention weights): computed position by position with the
    KV-cached step program (the causal mask is implicit), read out through fpnmt_decode_hidden.  The attention-weights dict
    (transformer.py:337-338) is None unless `return_attention=True`, which adds a pass through fpnmt_decode_attention."""

    def __init__(self, num_layers, d_model, num_heads, dff, target_vocab_size, rate=0.1, max_position=0, max_seq_len=12,
                 _cache=None):
        self.d_model, self.num_layers, self.max_seq_len = d_model, num_layers, max_seq_len
        self.pos_encoding = raw_positional_encoding(max_seq_len + max_position, d_model)
        self._cache = _cache

    def __call__(self, x, enc_output, training=False, look_ahead_mask=None, padding_mask=None, *, return_attention=False):
        if training:
            raise NotImplementedError("inference-only build: training=True is out of scope")
        if self._cache is None:
            raise RuntimeError("Decoder needs the engine of its Transformer (construct it through Transformer(...))")
        x = torch.as_tensor(x)
        eng = self._cache.get(int(x.shape[0]), 1, max(self.max_seq_len, int(x.shape[1])))
        hidden = eng.decode_hidden(enc_output, x)
        return hidden, (eng.decode_attention(enc_output, x) if return_attention else None)

    call = __call__


class Transformer:
    """transformer.py:344-374 with the reference's constructor signature; extra options are keyword-only."""

    def __init__(self, num_layers, d_model, num_heads, dff, input_vocab_size, target_vocab_size, rate=0.1,
                 max_position=0, max_seq_len=12, *, backbone: str = "mobilenet224_1.0",
                 weights: Optional[Dict[str, np.ndarray]] = None, seed: int = 0, precision: str = "bf16",
                 score_mode: str = "log", device: int = 0, start_id: int = C.START_ID, end_id: int = C.END_ID,
                 use_graphs: bool = True):
        if weights is None:
            weights = init_weights(backbone, vocab=target_vocab_size, seed=seed, num_layers=num_layers, d=d_model, dff=dff)
        self.weights = weights
        self.max_seq_len = max_seq_len
        self.target_vocab_size = target_vocab_size
        self._cache = _EngineCache(weights, backbone, num_layers, d_model, num_heads, dff, target_vocab_size, max_seq_len,
                                   precision, score_mode, device, start_id, end_id, use_graphs)
        self.encoder = Encoder(num_layers, d_model, num_heads, dff, input_vocab_size, rate, _cache=self._cache)
        self.decoder = Decoder(num_layers, d_model, num_heads, dff, target_vocab_size, rate, max_position, max_seq_len,
                               _cache=self._cache)
        self.final_layer = ("transformer/final_layer/kernel", "transformer/final_layer/bias")

    def __call__(self, inp, tar, training, look_ahead_mask, *, return_attention=False):
        """Inference branch (transformer.py:362-374): `inp` is the pre-computed encoder output (B,16,d);
        `tar` (B,t) token ids.  Returns (logits (B,t,V), attention-weights dict or None, see `Decoder`)."""
        if training:
            raise NotImplementedError("inference-only build: training=True is out of scope")
        tar = torch.as_tensor(tar)
        eng = self._cache.get(int(tar.shape[0]), 1, max(self.max_seq_len, int(tar.shape[1])))
        logits = eng.decode_logits(inp, tar)
        return logits, (eng.decode_attention(inp, tar) if return_attention else None)

    call = __call__

    def engine(self, batch: int, beam: int, max_len: Optional[int] = None, lanes: int = 1) -> Engine:
        """The engine for a batch shape; lanes >= 2 = that many batches in flight in `Engine.generate_stream` (throughput)."""
        return self._cache.get(batch, beam, max_len, lanes)

    @property
    def trainable_variables(self):
        return list(self.weights.values())

    def save_weights(self, path: str) -> None:
        from .weights import save_weights
        save_weights(path, self.weights)


def input_vocab_size_for(image_size: int = C.IMAGE_INPUT_SIZE) -> int:
    """utils/pipeline.py:20."""
    return math.ceil(image_size / 16) ** 2
