"""The model-level inference surface of `ppasr.model_utils` over the B200 engine (SURVEY §8b, "Model-level ops").

Mirrors the inference half of the reference model classes -- same class names, constructor arguments and method names:
    ConformerModel            ppasr/model_utils/conformer/model.py:16-66,148-184
    SqueezeformerModel        ppasr/model_utils/squeezeformer/model.py:16-66,150-186
    EfficientConformerModel   ppasr/model_utils/efficient_conformer/model.py:16-63,147-183
    DeepSpeech2Model          ppasr/model_utils/deepspeech2/model.py:24-72
so that callers such as PPASRTrainer.evaluate (`eval_model.get_encoder_out(inputs, input_lens).numpy()`, trainer.py:626) or
PPASRTrainer.export consumers can be pointed at the CUDA path. What they compute is the reference's
`get_encoder_out` (encoder -> CTC projection -> softmax: probabilities [B, T', V]) and `get_encoder_out_chunk`.

Differences, all stated:
  * parameters come from `set_state_dict(dict name -> array)` (what `paddle.load('model.pdparams')` yields, reference names
    and layouts) or from `weights=` / `model_dir=` at construction; the engine is built on first use;
  * `get_encoder_out_chunk` is functional in the reference (caches in, caches out). Here the K/V and conv caches live on the
    device: an EMPTY `att_cache` starts a new stream, anything else must be the continuation of the previous call (same
    `offset`) -- feeding caches from elsewhere raises. The returned caches are host copies in the reference layout for the
    Conformer and opaque continuation tokens for the Squeezeformer;
  * training (`forward`, losses, the attention decoder) and `export` are outside the hot path and raise;
  * results are host NumPy arrays wrapped so that `.numpy()` works like on a Paddle tensor.
"""
import numpy as np

from ..infer_utils.inference_predictor import InferencePredictor
from ..weights import read_mean_istd

__all__ = ["ConformerModel", "SqueezeformerModel", "EfficientConformerModel", "DeepSpeech2Model"]


class HostArray(np.ndarray):
    """A NumPy array that also answers `.numpy()` (what the reference callers do with the returned Paddle tensor)."""

    def numpy(self):
        return np.asarray(self)


def _wrap(a):
    return np.asarray(a).view(HostArray)


class _HotPathModel:
    use_model = None
    ctc_prefix = "ctc."

    def __init__(self, input_dim, vocab_size, mean_istd_path=None, streaming=True, encoder_conf=None, decoder_conf=None,
                 weights=None, model_dir=None, device=0, **training_only):
        self.input_dim = input_dim
        self.vocab_size = vocab_size
        self.streaming = streaming
        self.sos = self.eos = vocab_size - 1
        self._encoder_conf = dict(encoder_conf) if encoder_conf is not None else {}
        self._mean_istd_path = mean_istd_path
        self._weights = dict(weights) if weights is not None else None
        self._model_dir = model_dir
        self._device = device
        self._predictor = None

    # -- parameters -------------------------------------------------------------------------------------------------
    def set_state_dict(self, state_dict):
        """trainer.py:607-608 `model.set_state_dict(paddle.load(...))`: name -> array with the reference's names."""
        self._weights = {k: np.asarray(v) for k, v in state_dict.items()}
        self.close()

    def eval(self):
        return self

    def train(self):
        return self

    @property
    def predictor(self):
        if self._predictor is None:
            w = self._weights
            if w is not None and "encoder.global_cmvn.mean" not in w:
                if self._mean_istd_path is None:
                    raise Exception("GlobalCMVN statistics missing: pass mean_istd_path (normalizer.py:27-41)")
                w = dict(w)
                w["encoder.global_cmvn.mean"], w["encoder.global_cmvn.istd"] = read_mean_istd(self._mean_istd_path)
            if w is None and self._model_dir is None:
                raise Exception("no parameters: call set_state_dict(), or pass weights= / model_dir=")
            configs = {"encoder_conf": self._encoder_conf, "preprocess_conf": {"n_mels": self.input_dim}}
            kw = {} if self._model_dir is None else {"model_dir": self._model_dir}
            self._predictor = InferencePredictor(configs, self.use_model, streaming=self.streaming, weights=w,
                                                 vocab_size=self.vocab_size, device=self._device, **kw)
        return self._predictor

    def close(self):
        if self._predictor is not None:
            self._predictor.engine.close()
            self._predictor = None

    # -- inference ---------------------------------------------------------------------------------------------------
    def get_encoder_out(self, speech, speech_lengths):
        """model.py:148-162: speech [B, T, n_mels] fp32, speech_lengths [B] -> CTC probabilities [B, T', V]."""
        speech = np.ascontiguousarray(np.asarray(speech), dtype=np.float32)
        lens = np.asarray(speech_lengths).astype(np.int64)
        return _wrap(self.predictor.predict(speech, lens))

    def get_encoder_out_chunk(self, speech, offset, required_cache_size, att_cache=None, cnn_cache=None):
        """model.py:164-184: one streaming chunk [1, t, n_mels] -> (probabilities [1, t', V], att_cache, cnn_cache)."""
        if self.use_model == "deepspeech2":
            raise Exception("DeepSpeech2Model.get_encoder_out_chunk takes (speech, speech_lengths, init_state_h_box, init_state_c_box)")
        p = self.predictor
        fresh = att_cache is None or np.asarray(att_cache).size == 0
        offset = int(np.asarray(offset).reshape(-1)[0])
        if fresh:
            p.reset_stream()
            if offset != 0:
                raise Exception("a stream that starts with empty caches must start at offset 0")
        elif offset != int(p.offset[0]):
            raise Exception(f"device-resident caches: the chunk must continue the previous call (offset {int(p.offset[0])}), "
                            f"got offset {offset}")
        probs = p.predict_chunk_conformer(np.asarray(speech, dtype=np.float32), int(np.asarray(required_cache_size).reshape(-1)[0]))
        if self.use_model == "conformer":
            return _wrap(probs), _wrap(p.att_cache), _wrap(p.cnn_cache)
        # Squeezeformer keeps the caches of its half-rate blocks at half rate on the device; the reference layout (every key
        # repeated, squeezeformer/encoder.py:355-358) is not exported: the caller gets opaque non-empty continuation tokens
        token = np.full([1, 1, 1, 1], float(int(p.offset[0])), dtype=np.float32)
        return _wrap(probs), _wrap(token), _wrap(token.copy())

    # -- outside the hot path ----------------------------------------------------------------------------------------
    def forward(self, *a, **k):
        raise Exception("training (losses, attention decoder) is outside the ppasr_b200 hot path")

    __call__ = forward

    def export(self):
        raise Exception("paddle.jit export is outside the ppasr_b200 hot path: the engine is built from the config + weights")


class ConformerModel(_HotPathModel):
    use_model = "conformer"


class SqueezeformerModel(_HotPathModel):
    use_model = "squeezeformer"


class EfficientConformerModel(_HotPathModel):
    """efficient_conformer/model.py:16-63,147-183. get_encoder_out_chunk (forward_chunk, encoder.py:266-394) keeps its
    append-only grouped / half-rate caches on the device (run_encoder in csrc/runtime.cu); like the Squeezeformer the caller gets
    opaque continuation tokens instead of the reference's cache tensors. Streams run up to max_len encoder frames between
    reset_stream() calls and need required_cache_size < 0 (what PPASRPredictor passes, predict.py:304-306)."""
    use_model = "efficient_conformer"


class DeepSpeech2Model(_HotPathModel):
    """deepspeech2/model.py:24-72: `encoder_conf` keys num_rnn_layers / rnn_size / use_gru; the CTC head is called `decoder`."""
    use_model = "deepspeech2"
    ctc_prefix = "decoder."

    def __init__(self, input_dim, vocab_size, mean_istd_path=None, streaming=True, encoder_conf=None, decoder_conf=None, **kw):
        super().__init__(input_dim, vocab_size, mean_istd_path, streaming, encoder_conf, decoder_conf, **kw)

    def get_encoder_out_chunk(self, speech, speech_lengths, init_state_h_box=None, init_state_c_box=None):
        """model.py:67-72 -> (probabilities, lens, final_state_h_box, final_state_c_box). `init_state_h_box=None` starts a
        stream; otherwise the call must continue the previous one (states stay on the device)."""
        p = self.predictor
        if init_state_h_box is None:
            p.reset_stream()
        elif p.output_state_h is None:
            raise Exception("device-resident states: the first chunk of a stream passes init_state_h_box=None")
        probs, lens = p.predict_chunk_deepspeech(np.asarray(speech, dtype=np.float32))
        c = None if p.output_state_c is None else _wrap(p.output_state_c)
        return _wrap(probs), _wrap(lens), _wrap(p.output_state_h), c
