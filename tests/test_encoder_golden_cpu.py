"""The encoder oracles against the reference's OWN model code.

tests/golden/encoder_golden_*.npz were produced by tests/golden/make_encoder_golden.py, which imports the unmodified classes of
/root/reference/ppasr/model_utils/** (ConformerEncoder, SqueezeformerEncoder, EfficientConformerEncoder, CRNNEncoder, CTCLoss,
GlobalCMVN) on top of tests/golden/paddle_shim (a torch-CPU stand-in for the `paddle` package) and records their outputs for
seeded weights. Here the restatements in oracle/ must reproduce those outputs: offline CTC logits / probabilities of a ragged
batch (valid AND padded frames), the logits of a forward_chunk chain driven like predict.py:232-337, and the final caches /
recurrent state boxes. Tolerance: 5e-5 absolute on logits of magnitude ~30 (fp32 summation-order noise; observed <= 1.4e-5).
"""
import ast
import glob
import os

import numpy as np
import pytest
import torch

from oracle.conformer_oracle import ConformerConf, ConformerOracle, stream_windows
from oracle.deepspeech2_oracle import DeepSpeech2Conf, DeepSpeech2Oracle
from oracle.efficient_conformer_oracle import EfficientConformerConf, EfficientConformerOracle
from oracle.squeezeformer_oracle import SqueezeformerConf, SqueezeformerOracle
from ppasr_b200 import weights as W

GOLDEN = os.path.join(os.path.dirname(__file__), "golden")
ATOL = 5e-5

FAMILIES = {
    "conformer": (W.ConformerConfig, W.init_conformer_weights, ConformerConf, ConformerOracle),
    "squeezeformer": (W.SqueezeformerConfig, W.init_squeezeformer_weights, SqueezeformerConf, SqueezeformerOracle),
    "efficient_conformer": (W.EfficientConformerConfig, W.init_efficient_conformer_weights, EfficientConformerConf,
                            EfficientConformerOracle),
    "deepspeech2": (W.DeepSpeech2Config, W.init_deepspeech2_weights, DeepSpeech2Conf, DeepSpeech2Oracle),
}
FILES = sorted(os.path.basename(p) for p in glob.glob(os.path.join(GOLDEN, "encoder_golden_*.npz")))


def _family(fname):
    stem = fname[len("encoder_golden_"):]
    return max((f for f in FAMILIES if stem.startswith(f)), key=len)


def _oracle(g, family):
    cfg_cls, init, conf_cls, oracle_cls = FAMILIES[family]
    cfgd = ast.literal_eval(str(g["cfg"]))
    weights = init(cfg_cls(**cfgd), seed=int(g["seed"]))
    names = conf_cls.__init__.__code__.co_varnames
    if family in ("efficient_conformer", "deepspeech2"):
        conf = conf_cls(**cfgd)
    else:
        conf = conf_cls(**{k: v for k, v in cfgd.items() if k in names})
    return oracle_cls(conf, weights)


def test_fixtures_present():
    assert len(FILES) >= 21, FILES
    assert {_family(f) for f in FILES} == set(FAMILIES)


@pytest.mark.parametrize("fname", FILES)
def test_offline_matches_reference_code(fname):
    g = np.load(os.path.join(GOLDEN, fname))
    o = _oracle(g, _family(fname))
    feats, lens = torch.from_numpy(g["feats"]), torch.from_numpy(g["lens"])
    logits = o.get_encoder_out(feats, lens, return_logits=True).numpy()
    ref = g["offline_logits"]
    assert logits.shape == ref.shape
    np.testing.assert_allclose(logits, ref, rtol=0, atol=ATOL)  # padded frames included: the reference computes them too
    probs = o.get_encoder_out(feats, lens).numpy()
    np.testing.assert_allclose(probs, g["offline_probs"], rtol=0, atol=2e-5)
    assert (probs.argmax(-1) == g["offline_probs"].argmax(-1)).mean() > 0.999


@pytest.mark.parametrize("fname", [f for f in FILES if "stream" in f])
def test_chunk_chain_matches_reference_code(fname):
    g = np.load(os.path.join(GOLDEN, fname))
    family = _family(fname)
    o = _oracle(g, family)
    cf = g["chunk_feats"]
    assert cf.shape[0] > 0
    outs = []
    if family == "deepspeech2":
        h = c = None
        cfb = cf if cf.ndim == 3 else cf[None]  # the engine-size fixture streams a batch of 2
        for (a, b) in stream_windows(cfb.shape[1], is_end=True):
            x, _, h, c = o.get_encoder_out_chunk(torch.from_numpy(cfb[:, a:b]), torch.tensor([b - a] * cfb.shape[0]), h, c,
                                                 return_logits=True)
            outs.append(x.numpy() if cf.ndim == 3 else x[0].numpy())
        np.testing.assert_allclose(h.numpy(), g["chunk_state_h"], rtol=0, atol=1e-5)
        if "chunk_state_c" in g.files:
            np.testing.assert_allclose(c.numpy(), g["chunk_state_c"], rtol=0, atol=1e-5)
    else:
        att, cnn, off = torch.zeros(0, 0, 0, 0), torch.zeros(0, 0, 0, 0), 0
        required = int(g["required_cache_size"]) if "required_cache_size" in g.files else -16  # 32 / 0: bounded / no history
        for (a, b) in stream_windows(cf.shape[0], is_end=True):
            x, att, cnn = o.get_encoder_out_chunk(torch.from_numpy(cf[None, a:b]), off, required, att, cnn, return_logits=True)
            off += x.shape[1]
            outs.append(x[0].numpy())
        # the largest fixture stores every step-th channel of the attention cache (make_encoder_golden.py, att_cache_step)
        step = int(g["chunk_att_cache_step"]) if "chunk_att_cache_step" in g.files else 1
        att_shape = tuple(g["chunk_att_cache_shape"]) if step > 1 else g["chunk_att_cache"].shape
        assert tuple(att.shape) == att_shape and tuple(cnn.shape) == g["chunk_cnn_cache"].shape
        np.testing.assert_allclose(att.numpy()[..., ::step], g["chunk_att_cache"], rtol=0, atol=1e-5)
        np.testing.assert_allclose(cnn.numpy(), g["chunk_cnn_cache"], rtol=0, atol=1e-5)
    outs = np.concatenate(outs, 1 if outs[0].ndim == 3 else 0)
    assert outs.shape == g["chunk_logits"].shape
    np.testing.assert_allclose(outs, g["chunk_logits"], rtol=0, atol=ATOL)


@pytest.mark.parametrize("fname", [f for f in FILES if "stream" in f and "deepspeech2" not in f and "efficient" not in f])
def test_streaming_predict_is_whole_utterance_forward_chunk(fname):
    """InferencePredictor.predict on a streaming *former export feeds the forward_chunk graph with offset 0, no caches and
    required_cache_size -1 (inference_predictor.py:127-137; model.py:188-198 exports get_encoder_out_chunk). The engine computes
    the batched offline forward instead; for one utterance the two are the same function (odd and even subsampled lengths)."""
    g = np.load(os.path.join(GOLDEN, fname))
    o = _oracle(g, _family(fname))
    for T in (131, 135, 71):
        x = torch.from_numpy(W.synthetic_fbank(1, T, 80, seed=T))
        a = o.get_encoder_out(x, torch.tensor([T]), return_logits=True)
        b, _, _ = o.get_encoder_out_chunk(x, 0, -1, torch.zeros(0, 0, 0, 0), torch.zeros(0, 0, 0, 0), return_logits=True)
        assert a.shape == b.shape
        assert (a - b).abs().max().item() < 1e-5
