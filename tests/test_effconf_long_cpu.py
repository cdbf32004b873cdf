"""The Efficient Conformer oracle past 768 encoder frames (more than 256 key groups in the grouped blocks) against the
reference's OWN model code.

tests/golden/effconf_long_golden.npz was recorded by `golden/make_effconf_long_golden.py` from the unmodified
EfficientConformerEncoder (shipped 12-block layout, engine widths): the offline forward of one 40 s utterance and a forward_chunk
chain over its first chunk_T feature frames (848 encoder frames). Tolerances as in test_encoder_golden_cpu.py.
"""
import ast
import os

import numpy as np
import torch

from oracle.conformer_oracle import stream_windows
from oracle.efficient_conformer_oracle import EfficientConformerConf, EfficientConformerOracle
from ppasr_b200 import weights as W

FIXTURE = os.path.join(os.path.dirname(__file__), "golden", "effconf_long_golden.npz")
ATOL = 5e-5


def _load():
    g = np.load(FIXTURE)
    cfgd = ast.literal_eval(str(g["cfg"]))
    w = W.init_efficient_conformer_weights(W.EfficientConformerConfig(**cfgd), seed=int(g["seed"]))
    return g, EfficientConformerOracle(EfficientConformerConf(**cfgd), w)


def test_long_offline_matches_reference_code():
    g, o = _load()
    feats = torch.from_numpy(g["feats"].astype(np.float32))
    assert ((feats.shape[1] - 1) // 2 - 1) // 2 > 768
    logits = o.get_encoder_out(feats, torch.from_numpy(g["lens"]), return_logits=True).numpy()
    assert logits.shape == g["offline_logits"].shape
    np.testing.assert_allclose(logits, g["offline_logits"], rtol=0, atol=ATOL)
    probs = o.get_encoder_out(feats, torch.from_numpy(g["lens"])).numpy()
    np.testing.assert_allclose(probs, g["offline_probs"], rtol=0, atol=2e-5)


def test_long_chunk_chain_matches_reference_code():
    g, o = _load()
    cf = g["feats"][0, :int(g["chunk_T"])].astype(np.float32)
    att, cnn, off, outs = torch.zeros(0, 0, 0, 0), torch.zeros(0, 0, 0, 0), 0, []
    for (a, b) in stream_windows(cf.shape[0], is_end=True):
        x, att, cnn = o.get_encoder_out_chunk(torch.from_numpy(cf[None, a:b]), off, int(g["required_cache_size"]), att, cnn,
                                              return_logits=True)
        off += x.shape[1]
        outs.append(x[0].numpy())
    assert att.shape[2] > 768  # the grouped blocks attended more than 256 key groups
    outs = np.concatenate(outs, 0)
    assert outs.shape == g["chunk_logits"].shape
    np.testing.assert_allclose(outs, g["chunk_logits"], rtol=0, atol=ATOL)
    sa, sc = int(g["chunk_att_cache_step"]), int(g["chunk_cnn_cache_step"])
    assert tuple(att.shape) == tuple(g["chunk_att_cache_shape"]) and tuple(cnn.shape) == tuple(g["chunk_cnn_cache_shape"])
    np.testing.assert_allclose(att.numpy()[..., ::sa], g["chunk_att_cache"], rtol=0, atol=1e-5)
    np.testing.assert_allclose(cnn.numpy()[:, :, ::sc], g["chunk_cnn_cache"], rtol=0, atol=1e-5)
