"""Host-side mirror of /root/reference/utils/pipeline.py (inference half).

`Pipeline(tokenizer_filename, checkpoint_path, max_seq_len)` keeps the reference constructor (pipeline.py:12) and
the attributes its callers use (`tokenizer`, `transformer`, `max_seq_len`, `target_vocab_size`; test.py:14-21,
train.py:24,68,100,104).  `predict` / `evaluate` / `evaluate_img` return exactly what the reference returns;
`predict_batch` is the additive batched entry point.  Training members (`train_step`, `loss`, optimizer,
checkpoint manager) are out of scope and absent.

Checkpoints: the reference restores a TensorFlow object-graph checkpoint through a CheckpointManager
(pipeline.py:38-48).  `checkpoint_path` may name such a directory (`checkpoint` state file + `ckpt-N.index/.data-*`, read by
`fpnmt.checkpoint` without TensorFlow), a checkpoint prefix, or an `.npz` (or a directory holding `weights.npz`) keyed by
the same variable paths.  Without any of them the model is randomly initialised with the reference's distributions.
"""
from __future__ import annotations

import math
import os
from typing import Dict, Iterable, List, Optional, Tuple

import numpy as np
import torch

from . import config as C
from .dataset import Tokenizer, load_tokenizer_from_path
from .transformer import Transformer
from .weights import init_weights, load_weights


class Pipeline:
    def __init__(self, tokenizer_filename, checkpoint_path, max_seq_len, *, backbone: str = "mobilenet224_1.0",
                 beam: int = C.BEAM_SEARCH_N, precision: str = "bf16", score_mode: str = "log", device: int = 0,
                 weights: Optional[Dict[str, np.ndarray]] = None, tokenizer: Optional[Tokenizer] = None,
                 seed: int = 0, use_graphs: bool = True):
        # load tokenizer (pipeline.py:14)
        self.tokenizer = tokenizer if tokenizer is not None else load_tokenizer_from_path(tokenizer_filename)
        self.metric_eval = None      # pycocoevalcap hand-off (pipeline.py:15) is outside the hot path
        self.max_seq_len = max_seq_len
        self.beam = beam
        self.target_vocab_size = len(self.tokenizer.index_word)                 # pipeline.py:19
        input_vocab_size = math.ceil(C.IMAGE_INPUT_SIZE / 16) ** 2             # pipeline.py:20
        if weights is None and checkpoint_path:
            cand = checkpoint_path if str(checkpoint_path).endswith(".npz") else os.path.join(str(checkpoint_path), "weights.npz")
            if os.path.exists(cand):
                weights = load_weights(cand)
                print("Latest checkpoint restored!!")                           # pipeline.py:48
            else:
                from .checkpoint import latest_checkpoint, load_checkpoint
                prefix = latest_checkpoint(str(checkpoint_path)) if os.path.isdir(str(checkpoint_path)) else \
                    (str(checkpoint_path) if os.path.exists(str(checkpoint_path) + ".index") else None)
                if prefix:                                                      # pipeline.py:46-48 (latest_checkpoint)
                    weights = load_checkpoint(prefix, backbone)
                    print("Latest checkpoint restored!!")
        vocab_padded = (self.target_vocab_size + 7) // 8 * 8                   # engine wants vocab % 8 == 0
        self._vocab_padded = vocab_padded
        if weights is None:
            weights = init_weights(backbone, vocab=self.target_vocab_size, seed=seed)
        if weights["transformer/final_layer/kernel"].shape[1] != vocab_padded:
            weights = _pad_vocab(weights, vocab_padded)
        self.transformer = Transformer(C.num_layers, C.d_model, C.num_heads, C.dff, input_vocab_size, vocab_padded,
                                       C.DROPOUT_RATE, max_seq_len=self.max_seq_len, backbone=backbone, weights=weights,
                                       seed=seed, precision=precision, score_mode=score_mode, device=device,
                                       start_id=self.tokenizer.word_index["<start>"],
                                       end_id=self.tokenizer.word_index["<end>"], use_graphs=use_graphs)

    # ----------------------------------------------------------------------------------------------
    def predict_batch(self, imgs, max_seq_len: Optional[int] = None, beam: Optional[int] = None,
                      early_stop: bool = True, return_attention: bool = False):
        """Batched `predict`: imgs (B,S,S,3) float32 in [-1,1] -> (ids (B,T) int32 zero padded, lengths (B,)).
        return_attention: also the captions' attention-weights dict (Engine.caption_attention) as numpy arrays
        (B,heads,T,T) / (B,heads,T,n_memory), zero at and beyond position min(len + 1, T) -> (ids, lens, attn)."""
        imgs = torch.as_tensor(imgs) if not isinstance(imgs, torch.Tensor) else imgs
        eng = self.transformer.engine(int(imgs.shape[0]), beam or self.beam, max_seq_len or self.max_seq_len)
        ids, lens = eng.generate(imgs, early_stop=early_stop, to_host=True)
        if not return_attention:
            return ids.numpy(), lens.numpy()
        attn = {k: v.cpu().numpy() for k, v in eng.caption_attention(ids, lens).items()}
        return ids.numpy(), lens.numpy(), attn

    def _prefix_ids(self, prefix, B: int, T: int):
        """B prefix strings -> (ids (B, p) int32, lens (B,)) tokenized as score_batch does (a leading <start> dropped), or
        (None, None) for prefix None.  ValueError for a prefix holding <end> or max_seq_len or more tokens."""
        if prefix is None:
            return None, None
        if len(prefix) != B:
            raise ValueError("prefix: one string per image (%d), got %d" % (B, len(prefix)))
        start, end = self.tokenizer.word_index["<start>"], self.tokenizer.word_index["<end>"]
        seqs = []
        for seq in self.tokenizer.texts_to_sequences(list(prefix)):
            if seq and seq[0] == start:
                seq = seq[1:]
            if end in seq:
                raise ValueError("prefix: a prefix may not contain <end>")
            if len(seq) >= T:
                raise ValueError("prefix: a prefix of %d tokens needs max_seq_len > %d (max_seq_len = %d)" % (len(seq), len(seq), T))
            seqs.append(seq)
        ids = np.zeros((B, max(1, max(len(q) for q in seqs))), np.int32)
        for i, q in enumerate(seqs):
            ids[i, :len(q)] = q
        return ids, np.array([len(q) for q in seqs], np.int32)

    def _banned_ids(self, words):
        """banned_words -> token ids through tokenizer.word_index; ValueError for an unknown word or <end> (min_len is how
        <end> is held back)."""
        if not words:
            return None
        if isinstance(words, str):
            raise ValueError("banned_words: a list of words, got a string")
        ids = []
        for w in words:
            if w not in self.tokenizer.word_index:
                raise ValueError("banned_words: %r is not in the vocabulary" % (w,))
            if w == "<end>":
                raise ValueError("banned_words: <end> cannot be banned; use min_len")
            ids.append(int(self.tokenizer.word_index[w]))
        return ids

    def sample_batch(self, imgs, max_seq_len: Optional[int] = None, num_samples: Optional[int] = None, *,
                     temperature: float = 1.0, top_k: int = 0, top_p: float = 1.0, seed: int = 0, return_logprobs: bool = False,
                     prefix=None, no_repeat_ngram: int = 0, min_len: int = 0, banned_words=None):
        """`num_samples` (default: the beam width) independent sampled captions per image (Engine.sample): imgs (B,S,S,3)
        float32 in [-1,1] -> (ids (B,num_samples,T) int32 zero padded, lengths (B,num_samples)), plus the captions'
        log-likelihoods (B,num_samples) with return_logprobs.  temperature 0 is greedy.  prefix: B strings, each image's
        samples continue its string (tokenized as score_batch does; the returned captions include it).  no_repeat_ngram,
        min_len and banned_words (words of the tokenizer, e.g. "<start>", "<unk>") constrain the draw as Engine.sample does."""
        imgs = torch.as_tensor(imgs) if not isinstance(imgs, torch.Tensor) else imgs
        T = max_seq_len or self.max_seq_len
        pids, plens = self._prefix_ids(prefix, int(imgs.shape[0]), T)
        banned = self._banned_ids(banned_words)
        eng = self.transformer.engine(int(imgs.shape[0]), num_samples or self.beam, T)
        out = eng.sample(imgs, temperature=temperature, top_k=top_k, top_p=top_p, seed=seed, early_stop=True, to_host=True,
                         return_logprobs=return_logprobs, prefix=pids, prefix_lens=plens, no_repeat_ngram=no_repeat_ngram,
                         min_len=min_len, banned=banned)
        return tuple(o.numpy() for o in out)

    def beam_search_batch(self, imgs, max_seq_len: Optional[int] = None, num_beams: Optional[int] = None, *,
                          length_penalty: float = 0.0, return_logprobs: bool = False, beam_groups: int = 1,
                          diversity: float = 0.0, prefix=None, no_repeat_ngram: int = 0, min_len: int = 0, banned_words=None):
        """The `num_beams` (default: the beam width) most likely captions per image (Engine.beam_search): imgs (B,S,S,3)
        float32 in [-1,1] -> (ids (B,num_beams,T) int32 zero padded, in rank order, lengths (B,num_beams)), plus the captions'
        log-likelihoods (B,num_beams) with return_logprobs.  Ranking by log-likelihood / ((5 + n) / 6) ** length_penalty.
        beam_groups > 1: diverse beam search in that many groups with the given diversity penalty (group-major output).
        prefix: B strings, each image's beams continue its string (tokenized as score_batch does; the returned captions
        include it).  no_repeat_ngram: no n-gram twice in a caption; min_len: no <end> before that many tokens; banned_words:
        words of the tokenizer never emitted (e.g. "<start>" or the OOV token).  They remove candidates and never change a score."""
        imgs = torch.as_tensor(imgs) if not isinstance(imgs, torch.Tensor) else imgs
        T = max_seq_len or self.max_seq_len
        pids, plens = self._prefix_ids(prefix, int(imgs.shape[0]), T)
        banned = self._banned_ids(banned_words)
        eng = self.transformer.engine(int(imgs.shape[0]), num_beams or self.beam, T)
        out = eng.beam_search(imgs, length_penalty=length_penalty, early_stop=True, to_host=True, return_logprobs=return_logprobs,
                              beam_groups=beam_groups, diversity=diversity, prefix=pids, prefix_lens=plens,
                              no_repeat_ngram=no_repeat_ngram, min_len=min_len, banned=banned)
        return tuple(o.numpy() for o in out)

    def score_batch(self, imgs, captions, max_seq_len: Optional[int] = None, *, return_token_logprobs: bool = False):
        """Log-likelihoods of given captions (Engine.score): imgs (B,S,S,3) float32 in [-1,1], captions B lists of N strings
        (N the same for every image).  Each caption is tokenized with `tokenizer`; a leading <start> and a trailing <end>
        are dropped.  The pass runs over t = min(longest caption + 1, max_seq_len) positions; a caption longer than
        max_seq_len tokens raises ValueError.  Returns (B,N) float32 numpy, plus the per-position terms (B,N,t) with
        return_token_logprobs."""
        T = max_seq_len or self.max_seq_len
        if len({len(c) for c in captions}) != 1:
            raise ValueError("score_batch: every image needs the same number of captions")
        start, end = self.tokenizer.word_index["<start>"], self.tokenizer.word_index["<end>"]
        seqs = []
        for caps in captions:
            for seq in self.tokenizer.texts_to_sequences(caps):
                if seq and seq[0] == start:
                    seq = seq[1:]
                if seq and seq[-1] == end:
                    seq = seq[:-1]
                if len(seq) > T:
                    raise ValueError("score_batch: a caption of %d tokens exceeds max_seq_len = %d" % (len(seq), T))
                seqs.append(seq)
        B, N = len(captions), len(captions[0])
        t = min(max(len(q) for q in seqs) + 1, T)
        ids = np.zeros((B * N, t), np.int32)
        for i, q in enumerate(seqs):
            ids[i, :len(q)] = q
        lens = np.array([len(q) for q in seqs], np.int32).reshape(B, N)
        imgs = torch.as_tensor(imgs) if not isinstance(imgs, torch.Tensor) else imgs
        eng = self.transformer.engine(B, N, T)
        out = eng.score(ids.reshape(B, N, t), lens, imgs, return_token_logprobs=return_token_logprobs)
        return tuple(o.numpy() for o in out) if return_token_logprobs else out.numpy()

    def predict(self, img, max_seq_len, plot_layer=False):
        """pipeline.py:82-154: img (H,W,3) -> (1-D int32 ids without <start>/<end>, attention_weights).
        attention_weights is None unless `plot_layer` is truthy; then it is the dict of the reference's last forward pass for
        the returned caption, n = len + 1 positions when <end> fired and max_seq_len otherwise: "decoder_layer{i}_block1"
        (1,heads,n,n), "decoder_layer{i}_block2" (1,heads,n,n_memory), numpy float32.  Nothing is plotted."""
        img = torch.as_tensor(img) if not isinstance(img, torch.Tensor) else img
        if not plot_layer:
            ids, lens = self.predict_batch(img[None], max_seq_len)
            return ids[0, :lens[0]], None
        ids, lens, attn = self.predict_batch(img[None], max_seq_len, return_attention=True)
        n = min(int(lens[0]) + 1, ids.shape[1])
        attn = {k: np.ascontiguousarray(v[:, :, :n, :n] if k.endswith("_block1") else v[:, :, :n, :]) for k, v in attn.items()}
        return ids[0, :lens[0]], attn

    def evaluate(self, generator: Iterable, max_seq_len, batch_size: int = 1, lanes: int = 1) -> List[dict]:
        """pipeline.py:156-175: [(img, imgId)] -> [{"image_id", "caption"}] (optionally batched; lanes >= 2 keeps that many
        batches in flight on the GPU: encoder of batch i+1 under the decode of batch i)."""
        # Batches are packed into alternating pinned buffers and streamed through Engine.generate_stream, so the
        # host->device copy of batch i+1 overlaps the compute of batch i (dataset.py:90-92's prefetch).
        eng = self.transformer.engine(int(batch_size), self.beam, max_seq_len or self.max_seq_len, lanes)
        s = eng.image_size
        nbuf = max(2, lanes + 1)                                 # a buffer is reused only after its batch was submitted AND copied
        pinned = [None] * nbuf
        metas: List[list] = []

        def pack(buf, k):
            if pinned[k % nbuf] is None:
                pinned[k % nbuf] = torch.empty((batch_size, s, s, 3), dtype=torch.float32).pin_memory()
            dst = pinned[k % nbuf]
            for j, (img, _) in enumerate(buf):
                dst[j].copy_(torch.as_tensor(img))
            for j in range(len(buf), batch_size):                # pad the last batch
                dst[j].copy_(dst[len(buf) - 1])
            metas.append([m for _, m in buf])
            return dst

        def batches():
            buf, k = [], 0
            for item in generator:
                buf.append(item)
                if len(buf) == batch_size:
                    yield pack(buf, k)
                    buf, k = [], k + 1
            if buf:
                yield pack(buf, k)

        results = []
        for i, (ids, lens) in enumerate(eng.generate_stream(batches(), early_stop=True)):
            ids, lens = ids.numpy(), lens.numpy()
            for j, image_id in enumerate(metas[i]):
                text = self.tokenizer.sequences_to_texts([ids[j, :lens[j]]])[0]          # pipeline.py:169
                results.append({"image_id": image_id, "caption": text})
        return results

    def evaluate_img(self, img, max_seq_len) -> List[dict]:
        """pipeline.py:177-194."""
        result = self.predict(img, max_seq_len)[0]
        text = self.tokenizer.sequences_to_texts([np.asarray(result)])[0]
        return [{"image_id": 0, "caption": text}]


def _pad_vocab(weights: Dict[str, np.ndarray], vocab: int) -> Dict[str, np.ndarray]:
    """Pad the vocabulary axis to `vocab` with entries that can never win the beam (bias -1e9)."""
    w = dict(weights)
    k, b, e = w["transformer/final_layer/kernel"], w["transformer/final_layer/bias"], w["transformer/decoder/embedding/embeddings"]
    extra = vocab - k.shape[1]
    if extra > 0:
        w["transformer/final_layer/kernel"] = np.concatenate([k, np.zeros((k.shape[0], extra), np.float32)], 1)
        w["transformer/final_layer/bias"] = np.concatenate([b, np.full((extra,), -1e9, np.float32)])
        w["transformer/decoder/embedding/embeddings"] = np.concatenate([e, np.zeros((extra, e.shape[1]), np.float32)], 0)
    return w
