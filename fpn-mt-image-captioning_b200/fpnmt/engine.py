"""Python owner of one `fpnmt_handle` (one per GPU).  PyTorch is used for device memory and streams only.

Tensors cross the C ABI as raw device pointers: torch CUDA tensors directly, anything else that speaks
DLPack (`__dlpack__`) through `torch.from_dlpack`.
"""
from __future__ import annotations

import ctypes as C
import json
from typing import Dict, List, Optional, Sequence, Tuple

import numpy as np
import torch

from . import _lib
from . import config as cfg


def _as_cuda(x, dtype, device) -> torch.Tensor:
    if not isinstance(x, torch.Tensor):
        if hasattr(x, "__dlpack__"):
            x = torch.from_dlpack(x)
        else:
            x = torch.as_tensor(np.asarray(x))
    if x.device.type != "cuda":
        x = x.to(device, non_blocking=True)
    if x.dtype != dtype:
        x = x.to(dtype)
    return x.contiguous()


def _stream_ptr(device) -> int:
    return torch.cuda.current_stream(device).cuda_stream


class Engine:
    """B200 caption-inference engine for a fixed (backbone, batch, beam, vocab, max_len)."""

    def __init__(self, weights: Dict[str, np.ndarray], backbone: str = "mobilenet224_1.0", batch: int = 1,
                 beam: int = cfg.BEAM_SEARCH_N, vocab: Optional[int] = None, max_len: int = cfg.SYNTH_MAX_SEQ_LEN,
                 num_layers: int = cfg.num_layers, d_model: int = cfg.d_model, num_heads: int = cfg.num_heads,
                 dff: int = cfg.dff, image_size: int = cfg.IMAGE_INPUT_SIZE, precision: str = "bf16",
                 score_mode: str = "log", start_id: int = cfg.START_ID, end_id: int = cfg.END_ID,
                 true_beam: bool = False, use_graphs: bool = True, device: int = 0, opts: Sequence[str] = (),
                 cache_mode: str = "ancestry", decode_path: str = "auto", length_penalty: float = 0.0,
                 finished_beams: bool = False, lanes: int = 1):
        """opts: names from _lib.OPT_BITS (e.g. "no_xattn") - each turns one fused kernel back into its unfused equivalent;
        cache_mode "ancestry" | "physical"; decode_path "auto" (today: the per-operator chain) | "chain" | "fused" (one
        dstep_kernel launch runs every layer, the vocabulary projection and the beam tail of all steps); length_penalty / finished_beams: flagged extensions, 0 = reference;
        lanes: batches in flight for `generate_stream` (each lane is a complete engine on the same GPU; 2 overlaps the encoder
        of batch i+1 with the decode of batch i)."""
        if not torch.cuda.is_available():
            raise RuntimeError("fpnmt.Engine needs a CUDA device (sm_100a); there is no CPU fallback")
        self.lib = _lib.load()
        if vocab is None:
            vocab = int(weights["transformer/final_layer/kernel"].shape[1])
        self.device = torch.device("cuda", device)
        self.backbone, self.batch, self.beam, self.vocab, self.max_len = backbone, batch, beam, vocab, max_len
        self.image_size, self.d_model, self.num_layers, self.num_heads = image_size, d_model, num_layers, num_heads
        self.start_id = start_id
        self.precision = precision
        c = _lib.FpnmtConfig()
        c.backbone = _lib.BACKBONE_IDS[backbone]
        c.image_size, c.batch, c.beam, c.vocab, c.max_len = image_size, batch, beam, vocab, max_len
        c.num_layers, c.d_model, c.num_heads, c.dff = num_layers, d_model, num_heads, dff
        c.precision = _lib.PREC_IDS[precision]
        c.score_mode = _lib.SCORE_IDS[score_mode]
        c.start_id, c.end_id = start_id, end_id
        c.true_beam, c.use_graphs = int(true_beam), int(use_graphs)
        c.kernel_opts = 0
        for o in opts:
            c.kernel_opts |= _lib.OPT_BITS[o]
        c.cache_mode, c.decode_path = _lib.CACHE_IDS[cache_mode], _lib.DECODE_IDS[decode_path]
        c.length_penalty, c.finished_beams = float(length_penalty), int(finished_beams)
        c.lanes = int(lanes)
        self.lanes = max(1, int(lanes))
        self._h = C.c_void_p()
        torch.cuda.init()
        with torch.cuda.device(self.device):
            _lib.check(self.lib.fpnmt_create(C.byref(c), device, C.byref(self._h)))
            for key, arr in weights.items():
                a = np.ascontiguousarray(arr, dtype=np.float32)
                shape = (C.c_int64 * a.ndim)(*a.shape)
                _lib.check(self.lib.fpnmt_set_weight(self._h, key.encode(), a.ctypes.data_as(C.c_void_p), shape, a.ndim))
            _lib.check(self.lib.fpnmt_finalize_weights(self._h))
        side = image_size // 16
        self.feature_shapes = [(batch, side >> i, side >> i, d_model) for i in range(5)]
        self.n_memory = (side >> 3) ** 2

    # ------------------------------------------------------------------------------------------
    def close(self) -> None:
        if getattr(self, "_h", None) and self._h.value:
            self.lib.fpnmt_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _images(self, images) -> Tuple[int, int, object]:
        """Returns (pointer, on_host, keepalive)."""
        s = self.image_size
        if isinstance(images, torch.Tensor) and images.device.type == "cpu" or isinstance(images, np.ndarray):
            t = torch.as_tensor(images)
            if t.dtype != torch.float32 or not t.is_contiguous():
                t = t.to(torch.float32).contiguous()
            if tuple(t.shape) != (self.batch, s, s, 3):
                raise ValueError("images must be NHWC (%d,%d,%d,3), got %s" % (self.batch, s, s, tuple(t.shape)))
            return t.data_ptr(), 1, t
        t = _as_cuda(images, torch.float32, self.device)
        if tuple(t.shape) != (self.batch, s, s, 3):
            raise ValueError("images must be NHWC (%d,%d,%d,3), got %s" % (self.batch, s, s, tuple(t.shape)))
        return t.data_ptr(), 0, t

    def _images_opt(self, images) -> Tuple[Optional[int], int, object]:
        """`_images`, or (None, 0, None) for images None: the memory of the last encode."""
        return (None, 0, None) if images is None else self._images(images)

    def _memory(self, memory) -> Tuple[Optional[int], object]:
        """(pointer, keepalive) of a memory argument (B, n_memory, d_model); (None, None) for None: the last encode's."""
        if memory is None:
            return None, None
        mem = _as_cuda(memory, torch.float32, self.device)
        return mem.data_ptr(), mem

    def _result(self, shape, dtype, to_host: bool) -> torch.Tensor:
        """Output buffer of a call: pinned host memory for to_host (the call synchronises), else device memory."""
        if to_host:
            return torch.empty(shape, dtype=dtype).pin_memory()
        return torch.empty(shape, dtype=dtype, device=self.device)

    def encode(self, images) -> torch.Tensor:
        """Encoder.call (transformer.py:266-303): (B,S,S,3) -> (B, n_memory, d_model) float32 on device."""
        ptr, on_host, keep = self._images(images)
        out = torch.empty((self.batch, self.n_memory, self.d_model), dtype=torch.float32, device=self.device)
        _lib.check(self.lib.fpnmt_encode(self._h, ptr, on_host, out.data_ptr(), _stream_ptr(self.device)))
        return out

    def features(self, images) -> List[torch.Tensor]:
        """FeatureExtractor.call (retinanet.py:306-307): five NHWC float32 maps."""
        ptr, on_host, keep = self._images(images)
        outs = [torch.empty(sh, dtype=torch.float32, device=self.device) for sh in self.feature_shapes]
        arr = (C.c_void_p * 5)(*[o.data_ptr() for o in outs])
        _lib.check(self.lib.fpnmt_features(self._h, ptr, on_host, arr, _stream_ptr(self.device)))
        return outs

    def tap(self, name: str) -> torch.Tensor:
        n = C.c_size_t(0)
        _lib.check(self.lib.fpnmt_get_tap(self._h, name.encode(), None, 0, C.byref(n), _stream_ptr(self.device)))
        out = torch.empty((n.value,), dtype=torch.float32, device=self.device)
        _lib.check(self.lib.fpnmt_get_tap(self._h, name.encode(), out.data_ptr(), n.value, C.byref(n),
                                          _stream_ptr(self.device)))
        return out

    def decode_logits(self, memory, tokens) -> torch.Tensor:
        """Transformer.call(enc_output, tar, False, mask) (transformer.py:359-374) -> logits (B,t,V)."""
        tok = _as_cuda(tokens, torch.int32, self.device)
        t = int(tok.shape[1])
        mem_ptr, keep = self._memory(memory)
        out = torch.empty((self.batch, t, self.vocab), dtype=torch.float32, device=self.device)
        _lib.check(self.lib.fpnmt_decode_logits(self._h, mem_ptr, tok.data_ptr(), t, out.data_ptr(),
                                                _stream_ptr(self.device)))
        return out

    def decode_hidden(self, memory, tokens) -> torch.Tensor:
        """Decoder.call(x, enc_output, False, mask, None) (transformer.py:321-341) -> last decoder layer's output (B,t,d)."""
        tok = _as_cuda(tokens, torch.int32, self.device)
        t = int(tok.shape[1])
        mem_ptr, keep = self._memory(memory)
        out = torch.empty((self.batch, t, self.d_model), dtype=torch.float32, device=self.device)
        _lib.check(self.lib.fpnmt_decode_hidden(self._h, mem_ptr, tok.data_ptr(), t, out.data_ptr(), _stream_ptr(self.device)))
        return out

    def decode_attention(self, memory, tokens, self_attention: bool = True, cross_attention: bool = True
                         ) -> Dict[str, torch.Tensor]:
        """The attention-weights dict of Decoder.call (transformer.py:337-338) for teacher-forced tokens (B,t):
        "decoder_layer{i}_block1" (B,heads,t,t) causal self-attention and "decoder_layer{i}_block2" (B,heads,t,n_memory)
        cross-attention over the memory tokens, i counted from 1; float32 on the device.  memory None = the last encode."""
        if not (self_attention or cross_attention):
            raise ValueError("decode_attention: nothing requested")
        tok = _as_cuda(tokens, torch.int32, self.device)
        t = int(tok.shape[1])
        mem_ptr, keep = self._memory(memory)
        L, H = self.num_layers, self.num_heads
        so = torch.empty((L, self.batch, H, t, t), dtype=torch.float32, device=self.device) if self_attention else None
        co = torch.empty((L, self.batch, H, t, self.n_memory), dtype=torch.float32, device=self.device) if cross_attention else None
        _lib.check(self.lib.fpnmt_decode_attention(self._h, mem_ptr, tok.data_ptr(), t, so.data_ptr() if so is not None else None,
                                                   co.data_ptr() if co is not None else None, _stream_ptr(self.device)))
        out = {}
        for l in range(L):
            if so is not None:
                out["decoder_layer%d_block1" % (l + 1)] = so[l]
            if co is not None:
                out["decoder_layer%d_block2" % (l + 1)] = co[l]
        return out

    def caption_attention(self, ids, lens) -> Dict[str, torch.Tensor]:
        """Attention weights of captions returned by the last `generate` on this engine (ids (B,T), lens (B,)): one
        teacher-forced pass over [<start>] + caption with the memory that generate left.  Row j of a caption is the attention
        that predicted its token j (the last row predicted <end> when it fired); rows and columns at or beyond
        n_b = min(len_b + 1, T) are zero.  What the reference's predict returns for beam row 0 (pipeline.py:82-154)."""
        tok, n = caption_prefix(_as_cuda(ids, torch.int32, self.device), _as_cuda(lens, torch.int32, self.device), self.start_id)
        return mask_caption_attention(self.decode_attention(None, tok), n)

    def beam_step(self, logits, scores) -> Tuple[torch.Tensor, torch.Tensor, torch.Tensor]:
        """One decode-tail step (pipeline.py:115-141) on caller logits (B*N,V) and scores (B*N,)."""
        lg = _as_cuda(logits, torch.float32, self.device)
        sc = _as_cuda(scores, torch.float32, self.device)
        rows = self.batch * self.beam
        parent = torch.empty((rows,), dtype=torch.int32, device=self.device)
        token = torch.empty((rows,), dtype=torch.int32, device=self.device)
        out = torch.empty((rows,), dtype=torch.float32, device=self.device)
        _lib.check(self.lib.fpnmt_beam_step(self._h, lg.data_ptr(), sc.data_ptr(), parent.data_ptr(), token.data_ptr(),
                                            out.data_ptr(), _stream_ptr(self.device)))
        return parent, token, out

    def beam_step_vstats(self, stat, val, idx, scores) -> Tuple[torch.Tensor, torch.Tensor, torch.Tensor]:
        """`beam_step` through the logits-free tail: the vocabulary projection's per-tile softmax partials stat (B*N, tiles, 2),
        candidates val (B*N, tiles, 8) and their token ids idx (B*N, tiles, 8) int32 (what `vocab_stats` returns) instead of
        the logits."""
        st = _as_cuda(stat, torch.float32, self.device)
        vl = _as_cuda(val, torch.float32, self.device)
        ix = _as_cuda(idx, torch.int32, self.device)
        sc = _as_cuda(scores, torch.float32, self.device)
        rows = self.batch * self.beam
        tiles = int(st.shape[1])
        if st.shape != (rows, tiles, 2) or vl.shape != (rows, tiles, 8) or ix.shape != (rows, tiles, 8) or sc.shape != (rows,):
            raise ValueError("beam_step_vstats: stat (%d, tiles, 2), val and idx (%d, tiles, 8), scores (%d,)" % (rows, rows, rows))
        parent = torch.empty((rows,), dtype=torch.int32, device=self.device)
        token = torch.empty((rows,), dtype=torch.int32, device=self.device)
        out = torch.empty((rows,), dtype=torch.float32, device=self.device)
        _lib.check(self.lib.fpnmt_beam_step_vstats(self._h, st.data_ptr(), vl.data_ptr(), ix.data_ptr(), tiles, sc.data_ptr(),
                                                   parent.data_ptr(), token.data_ptr(), out.data_ptr(), _stream_ptr(self.device)))
        return parent, token, out

    def generate(self, images, early_stop: bool = True, to_host: bool = True, return_scores: bool = False):
        """Pipeline.predict for a batch (pipeline.py:82-154): ids (B,T) int32 zero-padded, lengths (B,)."""
        ptr, on_host, keep = self._images(images)
        ids = self._result((self.batch, self.max_len), torch.int32, to_host)
        lens = self._result((self.batch,), torch.int32, to_host)
        scores = None
        if return_scores:
            scores = torch.zeros((self.max_len, self.batch), dtype=torch.float32, device=self.device)
        _lib.check(self.lib.fpnmt_generate(self._h, ptr, on_host, ids.data_ptr(), lens.data_ptr(), int(to_host),
                                           int(early_stop), scores.data_ptr() if scores is not None else None,
                                           _stream_ptr(self.device)))
        return (ids, lens, scores) if return_scores else (ids, lens)

    def _prefix(self, prefix, prefix_lens):
        """(ids (B, p) int32, lens (B,) int32) on the device for a prompted call; ValueError for other shapes."""
        if prefix is None:
            if prefix_lens is not None:
                raise ValueError("prefix_lens without prefix")
            return None
        ids = _as_cuda(prefix, torch.int32, self.device)
        if ids.dim() != 2 or int(ids.shape[0]) != self.batch:
            raise ValueError("prefix must be (%d, p), got %s" % (self.batch, tuple(ids.shape)))
        if prefix_lens is None:
            lens = torch.full((self.batch,), int(ids.shape[1]), dtype=torch.int32, device=self.device)
        else:
            lens = _as_cuda(prefix_lens, torch.int32, self.device)
        if tuple(lens.shape) != (self.batch,):
            raise ValueError("prefix_lens must be (%d,), got %s" % (self.batch, tuple(lens.shape)))
        return ids, lens

    def sample(self, images=None, *, temperature: float = 1.0, top_k: int = 0, top_p: float = 1.0, seed: int = 0,
               early_stop: bool = True, to_host: bool = True, return_logprobs: bool = False, prefix=None, prefix_lens=None,
               no_repeat_ngram: int = 0, min_len: int = 0, banned=None):
        """`beam` independent sampled captions per image (fpnmt_sample; semantics in include/fpnmt.h): softmax(z / temperature)
        restricted to the top_k logits (0 = off, ties kept) and then to the nucleus of top_p of that mass (1 = off), drawn with
        the Philox stream of (seed, step, image, sample).  temperature 0 is greedy.  images None = the memory of the last
        encode / generate.  Returns ids (B, N, T) int32 zero padded without <start> / <end>, lengths (B, N) and, with
        return_logprobs, the captions' log-likelihoods (B, N) float32 (log_softmax at temperature 1, <end> included).
        prefix (B, p) int32 with prefix_lens (B,) (default: p for every image), on host or device: every sample of image b
        continues prefix[b, :prefix_lens[b]] (fpnmt_sample_prefix); the returned captions and log-likelihoods include it.
        no_repeat_ngram / min_len / banned (token ids): the constraints of fpnmt_sample_constrained (no n-gram twice, no <end>
        before min_len tokens, banned ids never drawn); they remove tokens from the draw and never change a log-likelihood."""
        ptr, on_host, keep = self._images_opt(images)
        pfx = self._prefix(prefix, prefix_lens)
        B, N, T = self.batch, self.beam, self.max_len
        ids = self._result((B, N, T), torch.int32, to_host)
        lens = self._result((B, N), torch.int32, to_host)
        lp = self._result((B, N), torch.float32, to_host) if return_logprobs else None
        sp = _lib.sampling(temperature, top_k, top_p, seed)
        lpp = lp.data_ptr() if lp is not None else None
        if no_repeat_ngram or min_len or banned is not None and len(banned):
            con = _lib.constraints(no_repeat_ngram, min_len, banned)
            _lib.check(self.lib.fpnmt_sample_constrained(
                self._h, ptr, on_host, pfx[0].data_ptr() if pfx else None, pfx[1].data_ptr() if pfx else None,
                int(pfx[0].shape[1]) if pfx else 0, C.byref(sp), C.byref(con), ids.data_ptr(), lens.data_ptr(), lpp,
                int(to_host), int(early_stop), _stream_ptr(self.device)))
        elif pfx is None:
            _lib.check(self.lib.fpnmt_sample(self._h, ptr, on_host, C.byref(sp), ids.data_ptr(), lens.data_ptr(), lpp,
                                             int(to_host), int(early_stop), _stream_ptr(self.device)))
        else:
            _lib.check(self.lib.fpnmt_sample_prefix(self._h, ptr, on_host, pfx[0].data_ptr(), pfx[1].data_ptr(),
                                                    int(pfx[0].shape[1]), C.byref(sp), ids.data_ptr(), lens.data_ptr(), lpp,
                                                    int(to_host), int(early_stop), _stream_ptr(self.device)))
        return (ids, lens, lp) if return_logprobs else (ids, lens)

    def beam_search(self, images=None, *, length_penalty: float = 0.0, early_stop: bool = True, to_host: bool = True,
                    return_logprobs: bool = False, beam_groups: int = 1, diversity: float = 0.0, prefix=None, prefix_lens=None,
                    no_repeat_ngram: int = 0, min_len: int = 0, banned=None):
        """The `beam` most likely captions per image by a true beam search with frozen finished beams (fpnmt_beam_search;
        definition in include/fpnmt.h), ranked by log-likelihood / ((5 + n) / 6) ** length_penalty, n the scored positions.
        images None = the memory of the last encode / generate / sample / score.  Returns ids (B, N, T) int32 zero padded
        without <start> / <end>, in rank order, lengths (B, N) (T: truncated) and, with return_logprobs, the captions'
        log-likelihoods (B, N) float32 (<end> included): what `score` gives for them with t = T.
        beam_groups G > 1 runs the diverse beam search instead (fpnmt_beam_search_diverse): G groups of N / G beams, each
        group's candidates lowered by `diversity` per earlier group's beam that chose the same token at the same step.  The
        output is group-major (beams [g * N / G, (g + 1) * N / G) are group g), rank order within a group.
        prefix (B, p) int32 with prefix_lens (B,) (default: p for every image), on host or device: every beam of image b
        continues prefix[b, :prefix_lens[b]] (fpnmt_beam_search_prefix); the returned captions and log-likelihoods include it.
        no_repeat_ngram / min_len / banned (token ids): the constraints of fpnmt_beam_search_constrained (no n-gram twice, no
        <end> before min_len tokens, banned ids never emitted); they remove candidates and never change a score."""
        ptr, on_host, keep = self._images_opt(images)
        pfx = self._prefix(prefix, prefix_lens)
        B, N, T = self.batch, self.beam, self.max_len
        ids = self._result((B, N, T), torch.int32, to_host)
        lens = self._result((B, N), torch.int32, to_host)
        lp = self._result((B, N), torch.float32, to_host) if return_logprobs else None
        if no_repeat_ngram or min_len or banned is not None and len(banned):
            con = _lib.constraints(no_repeat_ngram, min_len, banned)
            _lib.check(self.lib.fpnmt_beam_search_constrained(
                self._h, ptr, on_host, pfx[0].data_ptr() if pfx else None, pfx[1].data_ptr() if pfx else None,
                int(pfx[0].shape[1]) if pfx else 0, int(beam_groups), float(diversity), float(length_penalty), C.byref(con),
                ids.data_ptr(), lens.data_ptr(), lp.data_ptr() if lp is not None else None, int(to_host), int(early_stop),
                _stream_ptr(self.device)))
        elif pfx is not None:
            _lib.check(self.lib.fpnmt_beam_search_prefix(self._h, ptr, on_host, pfx[0].data_ptr(), pfx[1].data_ptr(),
                                                         int(pfx[0].shape[1]), int(beam_groups), float(diversity),
                                                         float(length_penalty), ids.data_ptr(), lens.data_ptr(),
                                                         lp.data_ptr() if lp is not None else None, int(to_host),
                                                         int(early_stop), _stream_ptr(self.device)))
        elif beam_groups == 1:
            _lib.check(self.lib.fpnmt_beam_search(self._h, ptr, on_host, float(length_penalty), ids.data_ptr(), lens.data_ptr(),
                                                  lp.data_ptr() if lp is not None else None, int(to_host), int(early_stop),
                                                  _stream_ptr(self.device)))
        else:
            _lib.check(self.lib.fpnmt_beam_search_diverse(self._h, ptr, on_host, int(beam_groups), float(diversity),
                                                          float(length_penalty), ids.data_ptr(), lens.data_ptr(),
                                                          lp.data_ptr() if lp is not None else None, int(to_host),
                                                          int(early_stop), _stream_ptr(self.device)))
        return (ids, lens, lp) if return_logprobs else (ids, lens)

    def score(self, ids, lens, images=None, *, to_host: bool = True, return_token_logprobs: bool = False):
        """Log-likelihoods of `beam` given captions per image in one teacher-forced pass (fpnmt_score; definition in
        include/fpnmt.h): ids (B, N, t) int32 in the layout `sample` returns (no <start>, no <end>, 1 <= t <= max_len;
        `sample`'s ids sliced to t fit), lens (B, N).  Position j predicts ids[..., j] for j < len and <end> at j = len
        when len < t.  images None = the memory of the last encode / generate / sample.  Returns the captions'
        log-likelihoods (B, N) float32 and, with return_token_logprobs, the per-position terms (B, N, t), 0 past each
        caption's scored positions; NaN for a caption with len outside [0, t] or an id outside [0, vocab)."""
        B, N = self.batch, self.beam
        tok = _as_cuda(ids, torch.int32, self.device)
        ln = _as_cuda(lens, torch.int32, self.device)
        if tok.dim() != 3 or tuple(tok.shape[:2]) != (B, N) or tuple(ln.shape) != (B, N):
            raise ValueError("score: ids must be (%d, %d, t) and lens (%d, %d), got %s and %s"
                             % (B, N, B, N, tuple(tok.shape), tuple(ln.shape)))
        t = int(tok.shape[2])
        ptr, on_host, keep = self._images_opt(images)
        lp = self._result((B, N), torch.float32, to_host)
        tl = self._result((B, N, t), torch.float32, to_host) if return_token_logprobs else None
        _lib.check(self.lib.fpnmt_score(self._h, ptr, on_host, tok.data_ptr(), ln.data_ptr(), t, lp.data_ptr(),
                                        tl.data_ptr() if tl is not None else None, int(to_host), _stream_ptr(self.device)))
        return (lp, tl) if return_token_logprobs else lp

    def stage(self, host_images, slot: int):
        """Enqueue the host->device copy of one batch into staging slot 0/1 on the engine's copy stream (returns at once).
        Returns the host tensor actually handed to the copy; keep it alive until the matching generate_staged is done."""
        t = torch.as_tensor(host_images)
        if t.device.type != "cpu":
            raise ValueError("stage() takes HOST images; device images go straight to generate()")
        s = self.image_size
        if tuple(t.shape) != (self.batch, s, s, 3):
            raise ValueError("images must be NHWC (%d,%d,%d,3), got %s" % (self.batch, s, s, tuple(t.shape)))
        if t.dtype != torch.float32 or not t.is_contiguous():
            t = t.to(torch.float32).contiguous()
        _lib.check(self.lib.fpnmt_stage_images(self._h, t.data_ptr(), int(slot)))
        return t

    def generate_staged(self, slot: int, early_stop: bool = True, to_host: bool = True):
        """`generate` on a batch previously handed to `stage(…, slot)`."""
        ids = self._result((self.batch, self.max_len), torch.int32, to_host)
        lens = self._result((self.batch,), torch.int32, to_host)
        _lib.check(self.lib.fpnmt_generate_staged(self._h, int(slot), ids.data_ptr(), lens.data_ptr(), int(to_host),
                                                  int(early_stop), None, _stream_ptr(self.device)))
        return ids, lens

    def submit(self, lane: int, images, early_stop: bool = False):
        """Enqueue one whole batch on lane `lane` (fpnmt_submit) and return at once.  Returns a keep-alive object: the images
        must stay valid until `collect(lane)`."""
        ptr, on_host, keep = self._images(images)
        _lib.check(self.lib.fpnmt_submit(self._h, int(lane), ptr, on_host, int(early_stop), _stream_ptr(self.device)))
        return keep

    def collect(self, lane: int, to_host: bool = True):
        """Result of the batch submitted on `lane` (fpnmt_collect): ids (B,T) int32 zero-padded, lengths (B,)."""
        ids = self._result((self.batch, self.max_len), torch.int32, to_host)
        lens = self._result((self.batch,), torch.int32, to_host)
        _lib.check(self.lib.fpnmt_collect(self._h, int(lane), ids.data_ptr(), lens.data_ptr(), int(to_host),
                                          _stream_ptr(self.device)))
        return ids, lens

    def generate_stream(self, batches, early_stop: bool = True, to_host: bool = True):
        """Captions for an iterable of batches (HOST tensors: pinned memory makes the copies asynchronous; or device tensors),
        yielded as (ids, lens) per batch, in order.  With `lanes` >= 2 the batches go round-robin through the lanes
        (fpnmt_submit / fpnmt_collect): host->device copy, encoder and decode of up to `lanes` batches are in flight at once, so
        the encoder of batch i+1 runs under the decode of batch i; results are identical to `generate` batch by batch.  With one
        lane: the double-buffered input copy of fpnmt_stage_images / fpnmt_generate_staged (the tf.data prefetch of
        dataset.py:92)."""
        it = iter(batches)
        if self.lanes >= 2:
            L, pending, i = self.lanes, [], 0
            for b in it:
                if len(pending) == L:
                    lane, _keep = pending.pop(0)
                    yield self.collect(lane, to_host=to_host)
                lane = i % L
                pending.append((lane, self.submit(lane, b, early_stop=early_stop)))
                i += 1
            for lane, _keep in pending:
                yield self.collect(lane, to_host=to_host)
            return
        try:
            first = next(it)
        except StopIteration:
            return
        if isinstance(first, torch.Tensor) and first.device.type == "cuda":
            b = first
            while b is not None:
                yield self.generate(b, early_stop=early_stop, to_host=to_host)
                b = next(it, None)
            return
        keep = [self.stage(first, 0), None]
        i = 0
        while True:
            nxt = next(it, None)
            if nxt is not None:
                keep[(i + 1) & 1] = self.stage(nxt, (i + 1) & 1)
            yield self.generate_staged(i & 1, early_stop=early_stop, to_host=to_host)
            if nxt is None:
                return
            i += 1

    def decode(self, early_stop: bool = True, to_host: bool = True):
        """Decode half only, from the memory left by the last `encode`."""
        ids = self._result((self.batch, self.max_len), torch.int32, to_host)
        lens = self._result((self.batch,), torch.int32, to_host)
        _lib.check(self.lib.fpnmt_decode(self._h, ids.data_ptr(), lens.data_ptr(), int(to_host), int(early_stop), None,
                                         _stream_ptr(self.device)))
        return ids, lens

    def profile(self, iters: int = 5) -> dict:
        buf = C.create_string_buffer(1 << 20)
        _lib.check(self.lib.fpnmt_profile(self._h, iters, buf, len(buf)))
        return json.loads(buf.value.decode())

    @property
    def launch_count(self) -> int:
        return int(self.lib.fpnmt_launch_count(self._h))


def caption_prefix(ids: torch.Tensor, lens: torch.Tensor, start_id: int) -> Tuple[torch.Tensor, torch.Tensor]:
    """Decoder input of the pass that gives a caption its attention weights: tokens (B,T) = [<start>] + ids[:, :T-1], and
    n_b = min(len_b + 1, T) valid positions (the tokens predicted, plus <end> when it fired before the last step)."""
    T = ids.shape[1]
    tok = torch.cat([torch.full_like(ids[:, :1], start_id), ids[:, :T - 1]], dim=1)
    return tok, torch.clamp(lens.to(torch.int64) + 1, max=T)


def mask_caption_attention(attn: Dict[str, torch.Tensor], n: torch.Tensor) -> Dict[str, torch.Tensor]:
    """Zeroes (in place) the rows of every (B,heads,T,.) block at or beyond n_b, and the columns of the self-attention
    blocks ("_block1") too."""
    for k, v in attn.items():
        ok = (torch.arange(v.shape[2], device=v.device)[None, :] < n.to(v.device)[:, None]).to(v.dtype)   # (B,T)
        v.mul_(ok[:, None, :, None])
        if k.endswith("_block1"):
            v.mul_(ok[:, None, None, :])
    return attn


def conv2d(x: torch.Tensor, kernel_hwio: np.ndarray, bias: Optional[np.ndarray] = None, act: int = 0,
           pad: Tuple[int, int] = (0, 0), residual: Optional[torch.Tensor] = None, res_mode: int = 0,
           precision: str = "bf16", force_bn: int = 0) -> torch.Tensor:
    """Stand-alone implicit-GEMM convolution (stride 1) through the C ABI — used by the kernel parity tests."""
    lib = _lib.load()
    dev = x.device
    x = x.to(torch.float32).contiguous()
    n, h, w, cin = x.shape
    k = np.ascontiguousarray(kernel_hwio, dtype=np.float32)
    kh, kw, _, cout = k.shape
    b = None if bias is None else np.ascontiguousarray(bias, dtype=np.float32)
    out = torch.empty((n, h, w, cout), dtype=torch.float32, device=dev)
    r = None if residual is None else residual.to(torch.float32).contiguous()
    _lib.check(lib.fpnmt_op_conv2d(dev.index or 0, _lib.PREC_IDS[precision], x.data_ptr(), n, h, w, cin,
                                   k.ctypes.data_as(C.c_void_p), kh, kw, cout, pad[0], pad[1],
                                   None if b is None else b.ctypes.data_as(C.c_void_p), act,
                                   None if r is None else r.data_ptr(), res_mode, out.data_ptr(), force_bn,
                                   _stream_ptr(dev)))
    return out


def dense(x: torch.Tensor, kernel: np.ndarray, bias: Optional[np.ndarray] = None, act: int = 0,
          residual: Optional[torch.Tensor] = None, gamma: Optional[np.ndarray] = None, beta: Optional[np.ndarray] = None,
          eps: float = 1e-6, precision: str = "bf16", force_bn: int = 0) -> torch.Tensor:
    """Stand-alone skinny-row Dense (+ residual + LayerNorm) through the C ABI — used by the kernel parity tests."""
    lib = _lib.load()
    dev = x.device
    x = x.to(torch.float32).contiguous()
    r, k = x.shape
    kn = np.ascontiguousarray(kernel, dtype=np.float32)
    f = kn.shape[1]
    host = lambda a: None if a is None else np.ascontiguousarray(a, dtype=np.float32)
    b, g, be = host(bias), host(gamma), host(beta)
    ptr = lambda a: None if a is None else a.ctypes.data_as(C.c_void_p)
    res = None if residual is None else residual.to(torch.float32).contiguous()
    out = torch.empty((r, f), dtype=torch.float32, device=dev)
    _lib.check(lib.fpnmt_op_dense(dev.index or 0, _lib.PREC_IDS[precision], x.data_ptr(), r, k, ptr(kn), f, ptr(b), act,
                                  None if res is None else res.data_ptr(), ptr(g), ptr(be), eps, out.data_ptr(), force_bn,
                                  _stream_ptr(dev)))
    return out


def vocab_stats(x: torch.Tensor, kernel: np.ndarray, bias: Optional[np.ndarray] = None, stat: Optional[torch.Tensor] = None,
                val: Optional[torch.Tensor] = None, idx: Optional[torch.Tensor] = None, precision: str = "bf16"
                ) -> Tuple[torch.Tensor, torch.Tensor, torch.Tensor]:
    """Vocabulary projection of the logits-free decode tail (fpnmt_op_vocab_stats): x (R, K), kernel (K, F) -> per
    (row, 128-feature tile) stat (R, ftiles, 2) = (max, sum exp(z - max)), val / idx (R, ftiles, 8) = the tile's 8 largest
    logits and their feature ids.  stat / val / idx, when given, are updated in place and may have more than R rows: rows
    from R on are not written."""
    x = _dev32(x)
    r, k = x.shape
    kn = _host32(kernel)
    f = kn.shape[1]
    ft = (f + 127) // 128
    dev = x.device
    stat = torch.full((r, ft, 2), float("nan"), device=dev) if stat is None else stat
    val = torch.full((r, ft, 8), float("nan"), device=dev) if val is None else val
    idx = torch.full((r, ft, 8), -1, dtype=torch.int32, device=dev) if idx is None else idx
    for t, n, dt, w in ((stat, "stat", torch.float32, 2), (val, "val", torch.float32, 8), (idx, "idx", torch.int32, 8)):
        if t.dtype != dt or not t.is_contiguous() or t.device != dev or t.dim() != 3 or t.shape[0] < r or tuple(t.shape[1:]) != (ft, w):
            raise ValueError("%s must be a contiguous %s tensor of shape (>= %d, %d, %d) on %s" % (n, dt, r, ft, w, dev))
    b = _host32(bias)
    _lib.check(_lib.load().fpnmt_op_vocab_stats(dev.index or 0, _lib.PREC_IDS[precision], x.data_ptr(), r, k, _hptr(kn), f,
                                                _hptr(b), stat.data_ptr(), val.data_ptr(), idx.data_ptr(), _stream_ptr(dev)))
    return stat, val, idx


def vocab_stats_target(x: torch.Tensor, kernel: np.ndarray, target, bias: Optional[np.ndarray] = None,
                       target_logit: Optional[torch.Tensor] = None, precision: str = "bf16"
                       ) -> Tuple[torch.Tensor, torch.Tensor, torch.Tensor, torch.Tensor]:
    """`vocab_stats` with the target epilogue of a prompted beam search (fpnmt_op_vocab_stats_target): also
    target_logit[r] = z[r, target[r]] (fp32, the value the tile's statistics come from) for every row whose target (R,) int32
    lies in [0, F); the other entries of target_logit (R,) float32 (default: NaN) keep their contents.
    Returns (stat, val, idx, target_logit)."""
    x = _dev32(x)
    r, k = x.shape
    kn = _host32(kernel)
    f = kn.shape[1]
    ft = (f + 127) // 128
    dev = x.device
    stat = torch.full((r, ft, 2), float("nan"), device=dev)
    val = torch.full((r, ft, 8), float("nan"), device=dev)
    idx = torch.full((r, ft, 8), -1, dtype=torch.int32, device=dev)
    tg = _as_cuda(target, torch.int32, dev)
    if tuple(tg.shape) != (r,):
        raise ValueError("target must be (%d,), got %s" % (r, tuple(tg.shape)))
    tl = torch.full((r,), float("nan"), device=dev) if target_logit is None else target_logit
    if tl.dtype != torch.float32 or not tl.is_contiguous() or tl.device != dev or tuple(tl.shape) != (r,):
        raise ValueError("target_logit must be a contiguous float32 tensor of shape (%d,) on %s" % (r, dev))
    b = _host32(bias)
    _lib.check(_lib.load().fpnmt_op_vocab_stats_target(dev.index or 0, _lib.PREC_IDS[precision], x.data_ptr(), r, k, _hptr(kn), f,
                                                       _hptr(b), tg.data_ptr(), stat.data_ptr(), val.data_ptr(), idx.data_ptr(),
                                                       tl.data_ptr(), _stream_ptr(dev)))
    return stat, val, idx, tl


def vocab_stats_mask(x: torch.Tensor, kernel: np.ndarray, mask: torch.Tensor, bias: Optional[np.ndarray] = None, target=None,
                     precision: str = "bf16") -> Tuple[torch.Tensor, torch.Tensor, torch.Tensor, Optional[torch.Tensor]]:
    """`vocab_stats` with the ban-mask epilogue of a constrained beam search (fpnmt_op_vocab_stats_mask): stat as
    `vocab_stats` (unmasked), val / idx the 8 largest logits per tile among the features whose bit in mask (R, ceil(F / 32))
    int32 (bit f % 32 of word f / 32) is clear.  With target (R,) also the target logits as `vocab_stats_target` (else None).
    Returns (stat, val, idx, target_logit)."""
    x = _dev32(x)
    r, k = x.shape
    kn = _host32(kernel)
    f = kn.shape[1]
    ft = (f + 127) // 128
    dev = x.device
    stat = torch.full((r, ft, 2), float("nan"), device=dev)
    val = torch.full((r, ft, 8), float("nan"), device=dev)
    idx = torch.full((r, ft, 8), -1, dtype=torch.int32, device=dev)
    mk = _as_cuda(mask, torch.int32, dev)
    if tuple(mk.shape) != (r, (f + 31) // 32):
        raise ValueError("mask must be (%d, %d), got %s" % (r, (f + 31) // 32, tuple(mk.shape)))
    tg = tl = None
    if target is not None:
        tg = _as_cuda(target, torch.int32, dev)
        if tuple(tg.shape) != (r,):
            raise ValueError("target must be (%d,), got %s" % (r, tuple(tg.shape)))
        tl = torch.full((r,), float("nan"), device=dev)
    b = _host32(bias)
    _lib.check(_lib.load().fpnmt_op_vocab_stats_mask(dev.index or 0, _lib.PREC_IDS[precision], x.data_ptr(), r, k, _hptr(kn), f,
                                                     _hptr(b), mk.data_ptr(), tg.data_ptr() if tg is not None else None,
                                                     stat.data_ptr(), val.data_ptr(), idx.data_ptr(),
                                                     tl.data_ptr() if tl is not None else None, _stream_ptr(dev)))
    return stat, val, idx, tl


def ban_mask(hist, lens, vocab: int, end_id: int, no_repeat_ngram: int = 0, min_len: int = 0, banned=None,
             device: int = 0) -> torch.Tensor:
    """The ban sets of fpnmt_constraints for given captions (fpnmt_op_ban_mask): hist (rows, ld) int32 caption tokens, lens
    (rows,) -> mask (rows, ceil(vocab / 32)) int32, bit v % 32 of word v / 32 set when token v is banned at step lens[r]."""
    dev = torch.device("cuda", device)
    h = _as_cuda(hist, torch.int32, dev)
    ln = _as_cuda(lens, torch.int32, dev)
    rows, ld = h.shape
    out = torch.full((rows, (vocab + 31) // 32), -1, dtype=torch.int32, device=dev)
    ids = [int(v) for v in (banned if banned is not None else [])]
    arr = (C.c_int32 * max(1, len(ids)))(*ids)
    _lib.check(_lib.load().fpnmt_op_ban_mask(device, h.data_ptr(), ld, ln.data_ptr(), rows, int(vocab), int(end_id),
                                             int(no_repeat_ngram), int(min_len), arr if ids else None, len(ids), out.data_ptr(),
                                             _stream_ptr(dev)))
    return out


# ---- stand-alone encoder bandwidth operators (kernel parity tests) --------------------------------------------------------
# Channel views: `x` / `out` may carry more channels per pixel (the last dim, a multiple of 8) than the `channels` the
# kernel reads and writes, like DenseNet's stage buffers.  `out` is read as well as written (updated in place and
# returned): what the kernel must not write comes back unchanged.  Without `out` a zero tensor is used.
def _host32(a):
    return None if a is None else np.ascontiguousarray(a, dtype=np.float32)


def _hptr(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def _dev32(t: torch.Tensor) -> torch.Tensor:
    if t.device.type != "cuda":
        raise RuntimeError("the stand-alone operators need CUDA tensors; there is no CPU fallback")
    return t.to(torch.float32).contiguous()


def _out32(out: Optional[torch.Tensor], shape, dev) -> torch.Tensor:
    if out is None:
        return torch.zeros(shape, dtype=torch.float32, device=dev)
    if out.dtype != torch.float32 or not out.is_contiguous() or out.device != dev or tuple(out.shape[:-1]) != tuple(shape[:-1]):
        raise ValueError("out must be a contiguous float32 tensor of shape %s (+ any channel count) on %s" % (tuple(shape[:-1]), dev))
    return out


def depthwise3x3(x: torch.Tensor, kernel: np.ndarray, bias: Optional[np.ndarray] = None, stride: int = 1,
                 pad: Tuple[int, int] = (1, 1), out_hw: Optional[Tuple[int, int]] = None, act: int = 0,
                 channels: Optional[int] = None, out: Optional[torch.Tensor] = None, precision: str = "bf16") -> torch.Tensor:
    """MobileNetV2 depthwise 3x3 (BN folded): x (N,H,W,ld), kernel (3,3,C,1), bias (C,) -> out (N,Ho,Wo,ld_out)."""
    x = _dev32(x)
    n, h, w, ld = x.shape
    c = channels or ld
    ho, wo = out_hw or ((h + 2 * pad[0] - 3) // stride + 1, (w + 2 * pad[1] - 3) // stride + 1)
    out = _out32(out, (n, ho, wo, c), x.device)
    k, b = _host32(kernel), _host32(bias)
    _lib.check(_lib.load().fpnmt_op_depthwise3x3(x.device.index or 0, _lib.PREC_IDS[precision], x.data_ptr(), n, h, w, c, ld,
                                                 _hptr(k), _hptr(b), stride, pad[0], pad[1], ho, wo, act, out.data_ptr(),
                                                 out.shape[-1], _stream_ptr(x.device)))
    return out


POOL_MAX, POOL_AVG2, POOL_SUBSAMPLE2 = 0, 1, 2


def pool(x: torch.Tensor, kind: int, k: int = 2, stride: int = 2, pad: Tuple[int, int] = (0, 0),
         out_hw: Optional[Tuple[int, int]] = None, zero_pad: bool = False, channels: Optional[int] = None,
         out: Optional[torch.Tensor] = None, precision: str = "bf16") -> torch.Tensor:
    """Max pool k x k / stride (POOL_MAX), 2x2 average pool (POOL_AVG2) or x[:, ::2, ::2] (POOL_SUBSAMPLE2) in NHWC."""
    x = _dev32(x)
    n, h, w, ld = x.shape
    c = channels or ld
    if out_hw is None:
        out_hw = {POOL_MAX: ((h + 2 * pad[0] - k) // stride + 1, (w + 2 * pad[1] - k) // stride + 1),
                  POOL_AVG2: (h // 2, w // 2), POOL_SUBSAMPLE2: ((h + 1) // 2, (w + 1) // 2)}[kind]
    ho, wo = out_hw
    out = _out32(out, (n, ho, wo, c), x.device)
    _lib.check(_lib.load().fpnmt_op_pool(x.device.index or 0, _lib.PREC_IDS[precision], kind, x.data_ptr(), n, h, w, c, ld, k,
                                         stride, pad[0], pad[1], ho, wo, int(zero_pad), out.data_ptr(), out.shape[-1],
                                         _stream_ptr(x.device)))
    return out


def scale_shift_relu(x: torch.Tensor, scale: np.ndarray, shift: np.ndarray, channels: Optional[int] = None,
                     out: Optional[torch.Tensor] = None, precision: str = "bf16") -> torch.Tensor:
    """DenseNet pre-activation BN + ReLU over the pixels of x (..., ld): relu(x[..., c] * scale[c] + shift[c])."""
    x = _dev32(x)
    ld = x.shape[-1]
    c = channels or ld
    pixels = x.numel() // ld
    out = _out32(out, tuple(x.shape[:-1]) + (c,), x.device)
    sc, sh = _host32(scale), _host32(shift)
    _lib.check(_lib.load().fpnmt_op_scale_shift_relu(x.device.index or 0, _lib.PREC_IDS[precision], x.data_ptr(), pixels, c, ld,
                                                     _hptr(sc), _hptr(sh), out.data_ptr(), out.shape[-1], _stream_ptr(x.device)))
    return out


def score_conv(x: torch.Tensor, kernel: np.ndarray, bias: np.ndarray, out: Optional[torch.Tensor] = None,
               precision: str = "bf16") -> torch.Tensor:
    """Co-attention score map: 3x3 'same' convolution of x (N,H,W,256) to one channel -> (N,H,W).  bf16 only."""
    x = _dev32(x)
    n, h, w, _ = x.shape
    if out is None:
        out = torch.zeros((n, h, w), dtype=torch.float32, device=x.device)
    elif out.dtype != torch.float32 or not out.is_contiguous() or tuple(out.shape) != (n, h, w):
        raise ValueError("out must be a contiguous float32 tensor of shape %s" % ((n, h, w),))
    k, b = _host32(kernel), _host32(np.reshape(bias, (1,)))
    _lib.check(_lib.load().fpnmt_op_score_conv(x.device.index or 0, _lib.PREC_IDS[precision], x.data_ptr(), n, h, w, _hptr(k),
                                               _hptr(b), out.data_ptr(), _stream_ptr(x.device)))
    return out


def coattention(score: torch.Tensor, cls: torch.Tensor, out: Optional[torch.Tensor] = None,
                precision: str = "bf16") -> torch.Tensor:
    """CoAttention_CNN: softmax over the HW positions of score (N,HW) times cls (N,HW,C) -> (N,HW,C)."""
    score, cls = _dev32(score), _dev32(cls)
    n, hw, c = cls.shape
    if tuple(score.shape) != (n, hw):
        raise ValueError("score must be (N, HW) to match cls (N, HW, C)")
    out = _out32(out, (n, hw, c), cls.device)
    if out.shape[-1] != c:
        raise ValueError("out must have the C channels of cls")
    _lib.check(_lib.load().fpnmt_op_coattention(cls.device.index or 0, _lib.PREC_IDS[precision], score.data_ptr(), cls.data_ptr(),
                                                n, hw, c, out.data_ptr(), _stream_ptr(cls.device)))
    return out


def tokens_ln_pos(x: torch.Tensor, hw: int, gamma: np.ndarray, beta: np.ndarray, pos: np.ndarray, eps: float = 1e-6,
                  out: Optional[torch.Tensor] = None, precision: str = "bf16") -> torch.Tensor:
    """Encoder token pre-amble: LayerNorm(x[n*hw+p]) + pos[p] over rows of x (N*hw, 512)."""
    x = _dev32(x)
    rows = x.shape[0]
    if x.shape[-1] != 512 or rows % hw:
        raise ValueError("x must be (N*hw, 512)")
    out = _out32(out, (rows, 512), x.device)
    if out.shape[-1] != 512:
        raise ValueError("out must be (N*hw, 512)")
    g, b, p = _host32(gamma), _host32(beta), _host32(pos)
    if p.size != hw * 512:
        raise ValueError("pos must be (hw, 512)")
    _lib.check(_lib.load().fpnmt_op_tokens_ln_pos(x.device.index or 0, _lib.PREC_IDS[precision], x.data_ptr(), rows // hw, hw,
                                                  _hptr(g), _hptr(b), eps, _hptr(p), out.data_ptr(), _stream_ptr(x.device)))
    return out


def enc_attention(q: torch.Tensor, kvs: Sequence[torch.Tensor], batch: int, heads: int, k_col: int, v_col: int,
                  force_simt: bool = False, out: Optional[torch.Tensor] = None, precision: str = "bf16") -> torch.Tensor:
    """Cross-level attention of the encoder: q (B*Tq, len(kvs)*heads*64) against the K/V columns [k_col, k_col+heads*64) /
    [v_col, ...) of each view's kvs[v] (B*Tk_v, kv_ld) -> (B*Tq, len(kvs)*heads*64).  All views share kv_ld."""
    q = _dev32(q)
    kvs = [_dev32(t) for t in kvs]
    nv = len(kvs)
    if q.shape[0] % batch or any(t.shape[0] % batch or t.shape[1] != kvs[0].shape[1] for t in kvs):
        raise ValueError("q and every K/V tensor must hold `batch` images, the K/V tensors one width")
    tq = q.shape[0] // batch
    out = _out32(out, (q.shape[0], q.shape[1]), q.device)
    if q.shape[1] != nv * heads * 64 or out.shape[1] != q.shape[1]:
        raise ValueError("q and out must be (B*Tq, len(kvs)*heads*64)")
    ptrs = (C.c_void_p * nv)(*[t.data_ptr() for t in kvs])
    tks = (C.c_int * nv)(*[t.shape[0] // batch for t in kvs])
    _lib.check(_lib.load().fpnmt_op_enc_attention(q.device.index or 0, _lib.PREC_IDS[precision], q.data_ptr(), ptrs, tks, nv,
                                                  kvs[0].shape[1], k_col, v_col, batch, tq, heads, int(force_simt),
                                                  out.data_ptr(), _stream_ptr(q.device)))
    return out


# ---- stand-alone decoder operators (kernel parity tests) ------------------------------------------------------------------
# Tensors the kernel writes (`out`, the caches, `dst`) are updated in place and must already be contiguous float32 CUDA
# tensors; integer tables are host arrays, checked by the library before upload.
def _inout32(t: torch.Tensor, shape, name: str) -> torch.Tensor:
    if t.dtype != torch.float32 or not t.is_contiguous() or t.device.type != "cuda" or tuple(t.shape) != tuple(shape):
        raise ValueError("%s must be a contiguous float32 CUDA tensor of shape %s" % (name, tuple(shape)))
    return t


def _host_i32(a):
    return None if a is None else np.ascontiguousarray(a, dtype=np.int32)


DEC_ATT_KERNELS = {"auto": 0, "simt": 1, "mma": 2}


def dec_self_attention(qkv: torch.Tensor, kc: torch.Tensor, vc: torch.Tensor, anc, t: int, heads: int, beam: int = 1, rep=None,
                       kc2: Optional[torch.Tensor] = None, vc2: Optional[torch.Tensor] = None, kernel: str = "auto",
                       out: Optional[torch.Tensor] = None, precision: str = "bf16") -> torch.Tensor:
    """Decode self-attention of step t: qkv (rows, 3*heads*64) against the caches kc / vc (rows*T, heads*64) through the
    ancestry table anc (2, rows, T); appends the new K/V to kc / vc (kc2 / vc2 on odd steps in the physical mode, which
    passing them selects).  rep (2, rows): token-history class representatives, or None.  Returns out (rows, heads*64)."""
    qkv = _dev32(qkv)
    rows, d = qkv.shape[0], heads * 64
    a = _host_i32(anc)
    T = a.shape[-1]
    if a.shape != (2, rows, T) or qkv.shape[1] != 3 * d:
        raise ValueError("qkv must be (rows, 3*heads*64) and anc (2, rows, T)")
    r = _host_i32(rep)
    if r is not None and r.shape != (2, rows):
        raise ValueError("rep must be (2, rows)")
    if (kc2 is None) != (vc2 is None):
        raise ValueError("kc2 and vc2 go together (the physical cache mode)")
    caches = [_inout32(c, (rows * T, d), n) for c, n in ((kc, "kc"), (vc, "vc"), (kc2, "kc2"), (vc2, "vc2")) if c is not None]
    out = _out32(out, (rows, d), qkv.device)
    _lib.check(_lib.load().fpnmt_op_dec_self_attention(
        qkv.device.index or 0, _lib.PREC_IDS[precision], qkv.data_ptr(), caches[0].data_ptr(), caches[1].data_ptr(),
        kc2.data_ptr() if kc2 is not None else None, vc2.data_ptr() if vc2 is not None else None, _hptr(a), _hptr(r), rows, T,
        t, heads, beam, DEC_ATT_KERNELS[kernel], out.data_ptr(), _stream_ptr(qkv.device)))
    return out


def dec_cross_attention(q: torch.Tensor, kv: torch.Tensor, beam: int, heads: int, k_col: int, v_col: int,
                        out: Optional[torch.Tensor] = None, precision: str = "bf16") -> torch.Tensor:
    """Decode cross-attention: q (rows, heads*64) against the memory tokens of its image, K/V at columns [k_col, +heads*64)
    / [v_col, ...) of kv (rows/beam*Tk, kv_ld) -> (rows, heads*64)."""
    q, kv = _dev32(q), _dev32(kv)
    rows = q.shape[0]
    if rows % beam or kv.shape[0] % (rows // beam) or q.shape[1] != heads * 64:
        raise ValueError("q must be (rows, heads*64), rows a multiple of beam, kv (rows/beam*Tk, kv_ld)")
    tk = kv.shape[0] // (rows // beam)
    out = _out32(out, (rows, heads * 64), q.device)
    _lib.check(_lib.load().fpnmt_op_dec_cross_attention(q.device.index or 0, _lib.PREC_IDS[precision], q.data_ptr(), kv.data_ptr(),
                                                        kv.shape[1], k_col, v_col, rows, beam, tk, heads, out.data_ptr(),
                                                        _stream_ptr(q.device)))
    return out


def xattn(ckv: torch.Tensor, wq: np.ndarray, bq: np.ndarray, wo: np.ndarray, bo: np.ndarray, gamma: np.ndarray,
          beta: np.ndarray, out1: torch.Tensor, beam: int, layer: int, b0: int = 0, images: Optional[int] = None,
          out2: Optional[torch.Tensor] = None, fold_outputs: bool = False, precision: str = "bf16"):
    """Fused decoder cross-attention block of `layer` on images [b0, b0 + images) of the batch: ckv (Btot*n_mem, L*1024)
    memory K/V of all layers; wq / wo (L, 512, 512) Dense kernels as stored; bq (L, 512); bo, gamma, beta (512,) of the
    layer; out1 (Btot*beam, 512).  Returns out2 (Btot*beam, 512), and with fold_outputs also the fold's (Mt, Nt, sbias)."""
    ckv, out1 = _dev32(ckv), _dev32(out1)
    wq, bq, wo = _host32(wq), _host32(bq), _host32(wo)
    L = wq.shape[0]
    Btot = out1.shape[0] // beam
    if out1.shape != (Btot * beam, 512) or ckv.shape[1] != L * 1024 or ckv.shape[0] % Btot or wq.shape != (L, 512, 512) or \
            wo.shape != (L, 512, 512) or bq.shape != (L, 512):
        raise ValueError("ckv (Btot*n_mem, L*1024), wq / wo (L, 512, 512), bq (L, 512), out1 (Btot*beam, 512)")
    n_mem = ckv.shape[0] // Btot
    images = Btot - b0 if images is None else images
    out2 = _out32(out2, (Btot * beam, 512), out1.device)
    dev = out1.device
    mt = torch.full((L * Btot * 128, 512), float("nan"), device=dev) if fold_outputs else None
    nt = torch.full((L * Btot * 512, 128), float("nan"), device=dev) if fold_outputs else None
    sb = torch.full((L * Btot * 128,), float("nan"), device=dev) if fold_outputs else None
    bo, gamma, beta = _host32(bo), _host32(gamma), _host32(beta)
    ptr = lambda t: None if t is None else t.data_ptr()
    _lib.check(_lib.load().fpnmt_op_xattn(dev.index or 0, _lib.PREC_IDS[precision], ckv.data_ptr(), _hptr(wq), _hptr(bq),
                                          _hptr(wo), _hptr(bo), _hptr(gamma), _hptr(beta), Btot, n_mem, L, layer, b0, images,
                                          beam, out1.data_ptr(), out2.data_ptr(), ptr(mt), ptr(nt), ptr(sb), _stream_ptr(dev)))
    return (out2, mt, nt, sb) if fold_outputs else out2


def kv_reorder(src: torch.Tensor, dst: torch.Tensor, parent, beam: int, t: int, precision: str = "bf16") -> torch.Tensor:
    """Physical KV-cache reorder after step t-1: src and dst (ncaches, rows, T, D); dst[c, r, :t] = src[c, (r // beam) * beam
    + parent[t-1][r], :t] in place; parent (T, rows) beam indices."""
    src = _dev32(src)
    nc, rows, T, D = src.shape
    _inout32(dst, src.shape, "dst")
    par = _host_i32(parent)
    if par.shape != (T, rows):
        raise ValueError("parent must be (T, rows)")
    _lib.check(_lib.load().fpnmt_op_kv_reorder(src.device.index or 0, _lib.PREC_IDS[precision], src.data_ptr(), dst.data_ptr(), nc,
                                               _hptr(par), rows, beam, T, D, t, _stream_ptr(src.device)))
    return dst


def embed_pos(tokens, emb: np.ndarray, pos: np.ndarray, t: int, out: Optional[torch.Tensor] = None, precision: str = "bf16",
              device: int = 0) -> torch.Tensor:
    """Decoder input of step t: emb[tokens[r]] + pos[t] -> (rows, C); emb (V, C), pos (T, C)."""
    tok = _host_i32(tokens).reshape(-1)
    emb, pos = _host32(emb), _host32(pos)
    (V, Cc), T = emb.shape, pos.shape[0]
    if pos.shape[1] != Cc:
        raise ValueError("emb and pos must have the same width")
    out = _out32(out, (tok.size, Cc), torch.device("cuda", device))
    _lib.check(_lib.load().fpnmt_op_embed_pos(device, _lib.PREC_IDS[precision], _hptr(tok), tok.size, _hptr(emb), V, _hptr(pos), T,
                                              Cc, t, out.data_ptr(), _stream_ptr(out.device)))
    return out


def layernorm_rows(x: torch.Tensor, gamma: np.ndarray, beta: np.ndarray, eps: float = 1e-6, out: Optional[torch.Tensor] = None,
                   precision: str = "bf16") -> torch.Tensor:
    """LayerNorm of fp32 rows x (rows, 512) into a bf16 / bf16x3 activation, read back as (rows, 512)."""
    x = _dev32(x)
    if x.dim() != 2 or x.shape[1] != 512:
        raise ValueError("x must be (rows, 512)")
    out = _out32(out, x.shape, x.device)
    g, b = _host32(gamma), _host32(beta)
    _lib.check(_lib.load().fpnmt_op_layernorm_rows(x.device.index or 0, _lib.PREC_IDS[precision], x.data_ptr(), x.shape[0],
                                                   _hptr(g), _hptr(b), eps, out.data_ptr(), _stream_ptr(x.device)))
    return out


def sample_step(logits: torch.Tensor, samples_per_image: int, t: int, temperature: float = 1.0, top_k: int = 0,
                top_p: float = 1.0, seed: int = 0) -> Tuple[torch.Tensor, torch.Tensor, torch.Tensor]:
    """One step of the sampling kernel (fpnmt_op_sample_step) on logits (rows, V): row r is sample r % samples_per_image of
    image r // samples_per_image at step t.  Returns (token (rows,) int32, log_softmax(logits)[token] at temperature 1
    (rows,) float32, the rows' Philox uniforms (rows,) float32), on the logits' device."""
    lg = logits if isinstance(logits, torch.Tensor) and logits.is_cuda else _as_cuda(logits, torch.float32, torch.device("cuda", 0))
    lg = lg.to(torch.float32).contiguous()
    rows, V = lg.shape
    device = lg.device.index or 0
    tok = torch.empty((rows,), dtype=torch.int32, device=lg.device)
    lp = torch.empty((rows,), dtype=torch.float32, device=lg.device)
    u = torch.empty((rows,), dtype=torch.float32, device=lg.device)
    sp = _lib.sampling(temperature, top_k, top_p, seed)
    _lib.check(_lib.load().fpnmt_op_sample_step(device, lg.data_ptr(), rows, V, int(samples_per_image), int(t), C.byref(sp),
                                                tok.data_ptr(), lp.data_ptr(), u.data_ptr(), _stream_ptr(lg.device)))
    return tok, lp, u


def preprocess(images_u8: torch.Tensor, size: int = cfg.IMAGE_INPUT_SIZE) -> torch.Tensor:
    """GPU `load_image` after the JPEG decode (dataset.py:21-24): uint8 (N,H,W,3) -> float32 (N,size,size,3) in [-1,1]."""
    lib = _lib.load()
    if images_u8.dtype != torch.uint8 or images_u8.dim() != 4 or images_u8.shape[-1] != 3:
        raise ValueError("images must be uint8 (N,H,W,3)")
    if images_u8.device.type != "cuda":
        raise RuntimeError("fpnmt.preprocess needs CUDA tensors; there is no CPU fallback")
    x = images_u8.contiguous()
    n, h, w, _ = x.shape
    out = torch.empty((n, size, size, 3), dtype=torch.float32, device=x.device)
    _lib.check(lib.fpnmt_op_preprocess(x.device.index or 0, x.data_ptr(), n, h, w, size, out.data_ptr(), _stream_ptr(x.device)))
    return out


def decode_jpeg(jpegs: Sequence[bytes], size: int = cfg.IMAGE_INPUT_SIZE, device: int = 0, return_sizes: bool = False):
    """GPU `load_image` for a batch of encoded JPEG files (dataset.py:19-26): nvJPEG decode (channels=3) -> bilinear resize
    (TF2 half-pixel, no antialias) -> x / 127.5 - 1.  Returns float32 (n, size, size, 3) on the device, ready for
    `Engine.encode` / `generate`; the decoded RGB images never visit the host."""
    lib = _lib.load()
    if not torch.cuda.is_available():
        raise RuntimeError("fpnmt.decode_jpeg needs a CUDA device; there is no CPU fallback")
    n = len(jpegs)
    bufs = [np.frombuffer(b, dtype=np.uint8) for b in jpegs]
    ptrs = (C.c_void_p * n)(*[b.ctypes.data for b in bufs])
    lens = (C.c_size_t * n)(*[b.size for b in bufs])
    dev = torch.device("cuda", device)
    out = torch.empty((n, size, size, 3), dtype=torch.float32, device=dev)
    sizes = np.zeros((n, 2), np.int32)
    with torch.cuda.device(dev):
        _lib.check(lib.fpnmt_op_decode_jpeg(device, ptrs, lens, n, size, out.data_ptr(), sizes.ctypes.data_as(C.c_void_p),
                                            _stream_ptr(dev)))
        torch.cuda.current_stream(dev).synchronize()       # the encoded bytes (host) may be released after this
    return (out, sizes) if return_sizes else out
