"""Generate tests/golden/effconf_long_golden.npz by running the reference's OWN, unmodified EfficientConformerEncoder past
768 encoder frames, where the grouped attention attends more than 256 key groups.

Same setup as make_encoder_golden.py (its helpers are reused): the reference classes are imported from the reference source
tree with `paddle` provided by tests/golden/paddle_shim, weights from the seeded initialisers of ppasr_b200/weights.py. Checked by
tests/test_effconf_long_cpu.py (oracle, 5e-5) and tests/test_gpu_effconf_long.py (CUDA path, 1e-2 of max logit).

The name stays outside the encoder_golden_*_gpu_*.npz pattern, whose count the engine-width fixture tests pin.

Run where the reference source tree is available (the tests only read the recorded file); deterministic, byte for byte:
    python tests/golden/make_effconf_long_golden.py
"""
import os
import sys

import numpy as np

sys.dont_write_bytecode = True
HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)

from make_encoder_golden import W, load_into, run_former, t  # noqa: E402  (sets up the paddle shim and the reference path)


def make_efficient_conformer_long(path, seed=1007, T=4000, chunk_T=67 + 64 * 52, vocab=24, att_cache_step=128, cnn_cache_step=4):
    """The shipped 12-block layout (configs/efficient_conformer.yml: group_layer_idx 0-3, stride_layer_idx 3) at engine widths
    past 768 encoder frames, where the grouped attention has more than 256 key groups: the offline forward of one 40 s
    utterance (T' = 999) and a forward_chunk chain (67-frame windows, required_cache_size -16) over its first chunk_T frames
    (848 encoder frames). Size: a small vocabulary, features stored as float16 (rounded BEFORE the reference consumes them, so
    the stored values are exactly its input; the chain reads the same array), and every step-th channel of the final caches
    (with their full shapes)."""
    from ppasr.model_utils.efficient_conformer.encoder import EfficientConformerEncoder
    from ppasr.model_utils.loss.ctc import CTCLoss
    from ppasr.model_utils.utils.cmvn import GlobalCMVN
    cfg = W.EfficientConformerConfig(input_dim=80, vocab_size=vocab, cnn_module_kernel=15, streaming=True,
                                     cnn_module_norm="layer_norm", group_size=3, num_blocks=12, group_layer_idx=(0, 1, 2, 3),
                                     stride_layer_idx=3)
    weights = W.init_efficient_conformer_weights(cfg, seed=seed)
    cmvn = GlobalCMVN(t(weights["encoder.global_cmvn.mean"]), t(weights["encoder.global_cmvn.istd"]))
    enc = EfficientConformerEncoder(input_size=cfg.input_dim, global_cmvn=cmvn, use_dynamic_chunk=True, causal=True,
                                    output_size=cfg.output_size, attention_heads=cfg.attention_heads,
                                    linear_units=cfg.linear_units, num_blocks=cfg.num_blocks,
                                    cnn_module_kernel=cfg.cnn_module_kernel, cnn_module_norm=cfg.cnn_module_norm,
                                    stride_layer_idx=cfg.stride_layer_idx, stride=cfg.stride,
                                    group_layer_idx=list(cfg.group_layer_idx), group_size=cfg.group_size,
                                    stride_kernel=cfg.stride_kernel)
    ctc = CTCLoss(cfg.vocab_size, enc.output_size())
    load_into(enc, weights, "encoder.", unused=("concat_linear",))
    load_into(ctc, weights, "ctc.")
    feats16 = W.synthetic_fbank(1, T, 80, seed=seed + 2).astype(np.float16)
    feats = feats16.astype(np.float32)
    lens = np.array([T], dtype=np.int64)
    out = run_former(enc, ctc, feats, lens, feats[0, :chunk_T])
    att, cnn = out.pop("chunk_att_cache"), out.pop("chunk_cnn_cache")
    out.update(chunk_att_cache=np.ascontiguousarray(att[..., ::att_cache_step]), chunk_att_cache_shape=np.array(att.shape),
               chunk_att_cache_step=np.array(att_cache_step), chunk_cnn_cache=np.ascontiguousarray(cnn[:, :, ::cnn_cache_step]),
               chunk_cnn_cache_shape=np.array(cnn.shape), chunk_cnn_cache_step=np.array(cnn_cache_step))
    np.savez_compressed(path, cfg=np.array(repr(cfg.to_dict())), seed=seed, feats=feats16, lens=lens, chunk_T=np.array(chunk_T),
                        required_cache_size=np.array(-16), **out)
    return out


if __name__ == "__main__":
    o = make_efficient_conformer_long(os.path.join(HERE, "effconf_long_golden.npz"))
    print("efficient_conformer long", {k: np.shape(v) for k, v in o.items()})
