"""Drop-in for ppasr/infer_utils/inference_predictor.py::InferencePredictor on a B200.

Same constructor signature, method names, NumPy array contracts and error behaviour as the reference
class (infer_utils/inference_predictor.py:11-220); the Paddle static graph behind `predictor.run()` is
replaced by the sm_100a kernels of libppasr_b200.so. Differences, all additive:
  * `model_dir` holds `model.npz` (or `model.pdparams`) with the reference's own parameter names, not an
    exported `.pdmodel/.pdiparams` pair;
  * `predict` accepts any batch size for every model type (the reference's streaming export is B=1);
  * `predict_decode` runs the fused CTC-head + greedy decode and returns ids / texts without ever
    materialising the [B, T', V] posterior (the reference copies it to the host, :143-145);
  * `weights=` lets tests/bench pass an in-memory parameter dict.
There is no CPU mode: `use_gpu=False` raises (the reference's CPU path is what bench.py times as the
baseline through the oracle).
"""
import os

import numpy as np

from .. import _lib as L
from ..engine import ConformerEngine
from ..parallel import detokenize
from ..weights import ConformerConfig, DeepSpeech2Config, EfficientConformerConfig, SqueezeformerConfig, load_npz, load_pdiparams, load_pdparams, read_mean_istd


def _get(obj, key, default=None):
    if obj is None:
        return default
    if isinstance(obj, dict):
        return obj.get(key, default)
    return getattr(obj, key, default)


def model_config_from(use_model, enc, n_mels, vocab_size, streaming):
    """yaml `encoder_conf` (a dict) -> the engine's config object, keeping the keys that shape the inference graph and
    dropping the training-only ones (dropout rates, activation_type 'swish', input_layer 'conv2d', ...), the way the
    reference model classes pass `**encoder_conf` to their encoders (conformer/model.py:43-47 etc.)."""
    if use_model == 'efficient_conformer':
        allowed = ('output_size', 'attention_heads', 'linear_units', 'num_blocks', 'cnn_module_kernel',
                   'cnn_module_norm', 'max_len', 'stride_layer_idx', 'stride', 'group_layer_idx', 'group_size',
                   'stride_kernel')
        kw = {k: enc[k] for k in allowed if k in enc}
        return EfficientConformerConfig(input_dim=n_mels, vocab_size=vocab_size, streaming=streaming, **kw)
    if use_model == 'deepspeech2':
        # configs/deepspeech2.yml encoder_conf (deepspeech2/encoder.py:8-16); streaming => forward-only RNN (model.py:40)
        kw = {k: enc[k] for k in ('num_rnn_layers', 'rnn_size', 'use_gru') if k in enc}
        return DeepSpeech2Config(input_dim=n_mels, vocab_size=vocab_size, streaming=streaming, **kw)
    if use_model == 'squeezeformer':
        # keys of configs/squeezeformer.yml encoder_conf (squeezeformer/encoder.py:24-53)
        allowed = ('encoder_dim', 'output_size', 'attention_heads', 'num_blocks', 'reduce_idx', 'recover_idx',
                   'feed_forward_expansion_factor', 'cnn_module_kernel', 'cnn_norm_type', 'adaptive_scale', 'max_len')
        kw = {k: enc[k] for k in allowed if k in enc}
        return SqueezeformerConfig(input_dim=n_mels, vocab_size=vocab_size, streaming=streaming, **kw)
    allowed = ('output_size', 'attention_heads', 'linear_units', 'num_blocks', 'cnn_module_kernel',
               'cnn_module_norm', 'max_len')
    kw = {k: enc[k] for k in allowed if k in enc}
    return ConformerConfig(input_dim=n_mels, vocab_size=vocab_size, streaming=streaming, **kw)


class InferencePredictor:
    def __init__(self,
                 configs,
                 use_model,
                 streaming=True,
                 model_dir='models/conformer_streaming_fbank/infer/',
                 use_gpu=True,
                 use_tensorrt=False,
                 gpu_mem=1000,
                 num_threads=10,
                 weights=None,
                 vocab_size=None,
                 device=0):
        if not use_gpu:
            raise Exception("ppasr_b200 only runs on a B200 GPU (use_gpu=False is not supported)")
        if use_model not in ('conformer', 'squeezeformer', 'deepspeech2', 'efficient_conformer'):
            raise Exception(f'当前模型不支持该方法，当前模型为：{use_model} (ppasr_b200 implements conformer, squeezeformer, efficient_conformer and deepspeech2)')
        self.configs = configs
        self.use_model = use_model
        self.streaming = streaming
        # streaming state, mirrors inference_predictor.py:35-39
        self.output_state_h = None
        self.output_state_c = None
        self._stream_active = False
        self._stream_batch = 0
        self._caches_stale = False
        self.cnn_cache = np.zeros([0, 0, 0, 0], dtype=np.float32)
        self.att_cache = np.zeros([0, 0, 0, 0], dtype=np.float32)
        self.offset = np.array([0], dtype=np.int32)

        enc = _get(configs, 'encoder_conf', {}) or {}
        enc = dict(enc) if isinstance(enc, dict) else {k: getattr(enc, k) for k in vars(enc)}
        pre = _get(configs, 'preprocess_conf', {}) or {}
        n_mels = _get(pre, 'n_mels', 80)
        if weights is None:
            npz = os.path.join(model_dir, 'model.npz')
            pdp = os.path.join(model_dir, 'model.pdparams')
            if os.path.exists(npz):
                weights, _ = load_npz(npz)
            elif os.path.exists(pdp):
                weights = load_pdparams(pdp)
            elif os.path.exists(os.path.join(model_dir, 'model.pdiparams')):
                # the reference's own exported inference model (inference_predictor.py:41-45)
                weights = load_pdiparams(os.path.join(model_dir, 'model.pdiparams'))
            else:
                # same failure mode as inference_predictor.py:43-44
                raise Exception("模型文件不存在，请检查%s和%s是否存在！" % (npz, pdp))
            mi = os.path.join(model_dir, 'mean_istd.json')
            if 'encoder.global_cmvn.mean' not in weights and os.path.exists(mi):
                mean, istd = read_mean_istd(mi)
                weights['encoder.global_cmvn.mean'] = mean
                weights['encoder.global_cmvn.istd'] = istd
        if vocab_size is None:
            key = 'decoder.ctc_lo.weight' if use_model == 'deepspeech2' else 'ctc.ctc_lo.weight'
            vocab_size = int(weights[key].shape[1])
        self.model_config = model_config_from(use_model, enc, n_mels, vocab_size, streaming)
        self._weights_ref = weights  # kept for DecodePipeline (extra engines pack their own copy)
        self.engine = ConformerEngine(self.model_config, weights, device=device)

    # ---------------------------------------------------------------------------------------------
    def predict(self, speech, speech_lengths):
        """inference_predictor.py:103-145: speech f32 [B,T,n_mels], speech_lengths i64 [B] -> probs f32 [B,T',V]
        (host NumPy). For streaming *former models the reference resets the caches and runs the whole
        utterance with full attention (:127-137); the batched engine path is that computation."""
        speech = np.ascontiguousarray(speech, dtype=np.float32)
        if 'former' in self.use_model and self.streaming:
            self.reset_stream()
        self.engine.encode(speech, speech_lengths)
        return self.engine.ctc_probs(to_host=True)

    def predict_decode(self, speech, speech_lengths=None, vocabulary=None, trim_to_lens=None, blank_id=0):
        """Extension: fused encoder + CTC head + greedy decode. speech may be host NumPy (copied H2D inside) or
        a CUDA tensor. Returns (ids [B,T'] int32, out_lens [B], scores [B] in the reference's 0..100 scale)
        or, when `vocabulary` is given, a list of (score, text) like greedy_decoder.
        trim_to_lens (default: True whenever speech_lengths is given) collapses each utterance over its own valid encoder
        frames only -- the frames the reference's subsampled mask keeps (4 j < len, utils/mask.py:22-68 after
        subsampling.py:113-115) -- so the padding frames of shorter utterances never add tokens or skew the score. Pass
        trim_to_lens=False to decode all T' frames of every row, which is what the reference's batched evaluation does
        (trainer.py:347-349 hands outs[i, :, :] to greedy_decoder_batch without slicing). PPASRPredictor.predict_batch trims
        further, to the frame count of a stand-alone run of each utterance."""
        if trim_to_lens is None:
            trim_to_lens = speech_lengths is not None
        self.engine.encode(speech, speech_lengths)
        ids, ol, sc = self.engine.ctc_greedy(to_host=True, trim_to_lens=trim_to_lens, blank_id=blank_id)
        scores = [float(s) * 100.0 if n > 0 else 0 for s, n in zip(sc, ol)]
        if vocabulary is None:
            return ids, ol, scores
        texts = detokenize(ids, ol, vocabulary)
        return list(zip(scores, texts))

    def pipeline(self, depth=2):
        """Double-buffered throughput mode: `depth` engines on private CUDA streams so the host->device copy of
        request i+1 overlaps the kernels of request i. See DecodePipeline."""
        return DecodePipeline(self, depth)

    def predict_chunk_deepspeech(self, x_chunk):
        """inference_predictor.py:147-182: x_chunk f32 [B, t, n_mels] -> (probs f32 [B, t', V], lens i64 [B]). The LSTM /
        GRU states (zero at the start of a stream, :157-164) stay on the device; `output_state_h` / `output_state_c`
        mirror them as NumPy [num_rnn_layers, B, rnn_size] after every call like the reference attributes."""
        if not (self.use_model == 'deepspeech2' and self.streaming):
            raise Exception(f'当前模型不支持该方法，当前模型为：{self.use_model}')
        x_chunk = np.ascontiguousarray(x_chunk, dtype=np.float32)
        if self.output_state_h is None or self._stream_batch != x_chunk.shape[0]:
            self.engine.stream_reset(x_chunk.shape[0])
            self._stream_active, self._stream_batch = True, x_chunk.shape[0]
        self.engine.encode_chunk(x_chunk)
        output_chunk_probs = self.engine.ctc_probs(to_host=True)
        self.output_state_h, self.output_state_c = self.engine.ds2_states()
        output_lens = np.full([x_chunk.shape[0]], output_chunk_probs.shape[1], dtype=np.int64)
        return output_chunk_probs, output_lens

    def predict_chunk_conformer(self, x_chunk, required_cache_size):
        """inference_predictor.py:184-212: x_chunk f32 [1, <=67, n_mels] -> probs f32 [1, chunk, V]; advances
        self.offset. The attention / conv caches stay on the device between calls; `self.att_cache` and
        `self.cnn_cache` are exported lazily in the reference layouts when read. Batched lock-step streams
        ([B, t, n_mels]) are accepted as an extension."""
        if not ('former' in self.use_model and self.streaming):
            raise Exception(f'当前模型不支持该方法，当前模型为：{self.use_model}')
        x_chunk = np.ascontiguousarray(x_chunk, dtype=np.float32)
        if not self._stream_active or self._stream_batch != x_chunk.shape[0]:
            self.engine.stream_reset(x_chunk.shape[0])
            self._stream_active, self._stream_batch = True, x_chunk.shape[0]
        self.engine.encode_chunk(x_chunk, int(required_cache_size))
        output_chunk_probs = self.engine.ctc_probs(to_host=True)
        self.offset += output_chunk_probs.shape[1]
        self._caches_stale = True
        return output_chunk_probs

    def _refresh_caches(self):
        if self._stream_active and self._caches_stale:
            self._att_cache, self._cnn_cache = self.engine.stream_export()
            self._caches_stale = False

    @property
    def att_cache(self):
        self._refresh_caches()
        return self._att_cache

    @att_cache.setter
    def att_cache(self, v):
        self._att_cache = v

    @property
    def cnn_cache(self):
        self._refresh_caches()
        return self._cnn_cache

    @cnn_cache.setter
    def cnn_cache(self, v):
        self._cnn_cache = v

    def reset_stream(self):
        """inference_predictor.py:215-220."""
        self.output_state_h = None
        self.output_state_c = None
        self._stream_active = False
        self._caches_stale = False
        self.att_cache = np.zeros([0, 0, 0, 0], dtype=np.float32)
        self.cnn_cache = np.zeros([0, 0, 0, 0], dtype=np.float32)
        self.offset = np.array([0], dtype=np.int32)


class DecodePipeline:
    """submit(speech[, lens]) -> ticket ; result(ticket) -> (ids, out_lens, scores).

    Each slot owns an engine (its own packed weights / workspace), a non-blocking CUDA stream and pinned host result
    buffers. submit() only enqueues work (pinned host features are copied asynchronously inside ppasr_b200_encode);
    result() synchronises that slot's stream. With depth 2 the PCIe copy of one batch hides behind the compute of the
    previous one."""

    def __init__(self, predictor, depth=2):
        import torch
        self.torch = torch
        self.pred = predictor
        self.slots = []
        for k in range(depth):
            eng = predictor.engine if k == 0 else ConformerEngine(predictor.model_config, predictor._weights_ref,
                                                                  device=predictor.engine.device.index)
            eng.set_option("host_sync", 0)
            self.slots.append({"eng": eng, "stream": torch.cuda.Stream(device=predictor.engine.device), "bufs": None,
                               "key": None})
        self.next = 0
        if depth > 1:
            predictor.engine.lib.ppasr_b200_set_pdl(0)  # early-started dependent CTAs would only hold SMs
            # several batches in flight fill the GPU by themselves: use the FFN variant with the least SM time per launch
            L.check(predictor.engine.lib.ppasr_b200_set_ffn_split(int(os.environ.get("PPASR_B200_FFN_PIPE", "2"))))

    def submit(self, speech, speech_lengths=None, trim_to_lens=False, blank_id=0, to_host=True):
        torch = self.torch
        k = self.next
        self.next = (self.next + 1) % len(self.slots)
        slot = self.slots[k]
        eng = slot["eng"]
        with torch.cuda.stream(slot["stream"]):
            eng.encode(speech, speech_lengths, stream=slot["stream"])
            B, Tp = eng.B, eng.Tp
            key = (B, Tp, bool(to_host))
            if slot["bufs"] is None or slot["key"] != key:
                if to_host:
                    slot["bufs"] = (torch.empty((B, Tp), dtype=torch.int32).pin_memory(),
                                    torch.empty((B,), dtype=torch.int32).pin_memory(),
                                    torch.empty((B,), dtype=torch.float32).pin_memory())
                else:
                    dev = eng.device
                    slot["bufs"] = (torch.empty((B, Tp), dtype=torch.int32, device=dev),
                                    torch.empty((B,), dtype=torch.int32, device=dev),
                                    torch.empty((B,), dtype=torch.float32, device=dev))
                slot["key"] = key
            ids, ol, sc = slot["bufs"]
            L.check(eng.lib.ppasr_b200_ctc_greedy(eng._ctx, L.ptr(ids), L.ptr(ol), L.ptr(sc), None, None,
                                                   0 if to_host else 1, int(trim_to_lens), blank_id,
                                                   L.stream_ptr(slot["stream"])))
        return k

    def stream(self, ticket):
        return self.slots[ticket]["stream"]

    def device_result(self, ticket):
        """Device tensors (ids, out_lens, scores) of a to_host=False request; valid on that slot's stream."""
        return self.slots[ticket]["bufs"]

    def result(self, ticket):
        slot = self.slots[ticket]
        slot["stream"].synchronize()
        ids, ol, sc = slot["bufs"]
        ids, ol, sc = ids.cpu().numpy().copy(), ol.cpu().numpy().copy(), sc.cpu().numpy().copy()
        scores = [float(s) * 100.0 if n > 0 else 0 for s, n in zip(sc, ol)]
        return ids, ol, scores

    def close(self):
        for slot in self.slots[1:]:
            slot["eng"].close()
        self.slots[0]["eng"].set_option("host_sync", 1)
        self.pred.engine.lib.ppasr_b200_set_pdl(1)
        L.check(self.pred.engine.lib.ppasr_b200_set_ffn_split(int(os.environ.get("PPASR_B200_FFN_SPLIT", "1"))))
