"""Generate tests/golden/encoder_golden_<model>.npz by running the reference's OWN, unmodified model code.

PaddlePaddle is not installable here, so the reference classes are imported from /root/reference with `paddle` provided by
tests/golden/paddle_shim (a torch-CPU stand-in implementing exactly the Paddle calls those files make, see its README).
Weights: the seeded synthetic initialisers of ppasr_b200/weights.py (reference parameter names), small dimensions so the
fixtures stay a few hundred KB. Recorded per model: the offline `get_encoder_out` CTC probabilities (+ logits) for a ragged
batch, and a `get_encoder_out_chunk` chain (67-frame windows, stride 64, as predict.py:232-337 drives it) for one utterance.

Run (in the build container only; /root/reference is not on the GPU box):
    python tests/golden/make_encoder_golden.py [conformer squeezeformer efficient_conformer deepspeech2]
tests/test_oracle_cpu.py::test_encoder_oracle_vs_reference_code then checks oracle/*_oracle.py against these files.
"""
import os
import sys

import numpy as np

sys.dont_write_bytecode = True  # /root/reference is read-only
HERE = os.path.dirname(os.path.abspath(__file__))
REPO = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, os.path.join(HERE, "paddle_shim"))
sys.path.insert(0, "/root/reference")
sys.path.insert(0, REPO)

import paddle  # noqa: E402  (the shim)
import torch  # noqa: E402

from ppasr_b200 import weights as W  # noqa: E402


def load_into(layer, weights, prefix, unused=()):
    """`unused`: substrings of parameters the reference constructs but never reads at inference (left at zero)."""
    own = layer.state_dict()
    sub = {k[len(prefix):]: v for k, v in weights.items() if k.startswith(prefix)}
    for k in [k for k in own if any(u in k for u in unused)]:
        own.pop(k)
    missing = [k for k in own if k not in sub]
    extra = [k for k in sub if k not in own]
    assert not missing and not extra, ("state mismatch", prefix, missing[:6], extra[:6])
    with torch.no_grad():
        for k, v in own.items():
            assert tuple(v.shape) == tuple(sub[k].shape), (k, v.shape, sub[k].shape)
            v.copy_(torch.from_numpy(sub[k]))


def stream_windows(num_frames, window=67, stride=64):
    """predict.py:281-297 with is_end on the last call: offsets of the decoding windows over the whole feature matrix."""
    out = []
    for cur in range(0, num_frames - 7 + 1, stride):
        out.append((cur, min(cur + window, num_frames)))
    return out


def t(x, dtype=None):
    return paddle.to_tensor(np.ascontiguousarray(x), dtype=dtype)


def logits_of(ctc, hs):
    return ctc.ctc_lo(hs)


# ---------------------------------------------------------------------------------------------------------------------
def build_conformer(cfg, weights, streaming):
    from ppasr.model_utils.conformer.encoder import ConformerEncoder
    from ppasr.model_utils.loss.ctc import CTCLoss
    from ppasr.model_utils.utils.cmvn import GlobalCMVN
    cmvn = GlobalCMVN(t(weights["encoder.global_cmvn.mean"]), t(weights["encoder.global_cmvn.istd"]))
    enc = ConformerEncoder(input_size=cfg.input_dim, global_cmvn=cmvn, use_dynamic_chunk=streaming, causal=streaming,
                           output_size=cfg.output_size, attention_heads=cfg.attention_heads, linear_units=cfg.linear_units,
                           num_blocks=cfg.num_blocks, cnn_module_kernel=cfg.cnn_module_kernel,
                           cnn_module_norm=cfg.cnn_module_norm, max_len=cfg.max_len)
    ctc = CTCLoss(cfg.vocab_size, enc.output_size())
    return enc, ctc


def run_former(enc, ctc, feats, lens, chunk_feats, required=-16):
    """model.py:148-184 get_encoder_out / get_encoder_out_chunk, called on the reference encoder + CTC head."""
    enc.eval(), ctc.eval()
    out = {}
    with torch.no_grad():
        hs, _ = enc(t(feats), t(lens, "int64"), decoding_chunk_size=-1, num_decoding_left_chunks=-1)
        out["offline_logits"] = logits_of(ctc, hs).numpy()
        out["offline_probs"] = ctc.softmax(hs).numpy()
        if chunk_feats is not None:
            att = paddle.zeros([0, 0, 0, 0])
            cnn = paddle.zeros([0, 0, 0, 0])
            offset = 0
            logits = []
            for (a, b) in stream_windows(chunk_feats.shape[0]):
                xs, att, cnn = enc.forward_chunk(xs=t(chunk_feats[None, a:b]), offset=offset, required_cache_size=required,
                                                 att_cache=att, cnn_cache=cnn)
                offset += int(xs.shape[1])
                logits.append(logits_of(ctc, xs).numpy()[0])
            out["chunk_logits"] = np.concatenate(logits, 0)
            out["chunk_att_cache"] = att.numpy()
            out["chunk_cnn_cache"] = cnn.numpy()
    return out


SMALL = dict(output_size=64, attention_heads=4, linear_units=128, num_blocks=3, max_len=600)  # CPU-test fixtures
LENS = (131, 96, 57)


def inputs(lens, chunk_T, seed):
    lens = np.array(lens, dtype=np.int64)
    feats = W.synthetic_fbank(len(lens), int(lens.max()), 80, seed=seed + 2)
    for b, n in enumerate(lens):
        feats[b, n:] = 0
    chunk_feats = W.synthetic_fbank(1, chunk_T, 80, seed=seed + 3)[0] if chunk_T else None
    return feats, lens, chunk_feats


def make_conformer(path, streaming=True, norm="layer_norm", seed=1000, lens=LENS, chunk_T=211, vocab=40, required=-16, **kw):
    cfg = W.ConformerConfig(input_dim=80, vocab_size=vocab, cnn_module_kernel=15, streaming=streaming, cnn_module_norm=norm,
                            **(kw or SMALL))
    weights = W.init_conformer_weights(cfg, seed=seed)
    enc, ctc = build_conformer(cfg, weights, streaming)
    load_into(enc, weights, "encoder.")
    load_into(ctc, weights, "ctc.")
    feats, lens, chunk_feats = inputs(lens, chunk_T if streaming else 0, seed)
    out = run_former(enc, ctc, feats, lens, chunk_feats, required)
    out["required_cache_size"] = np.array(required)
    np.savez_compressed(path, cfg=np.array(repr(cfg.to_dict())), seed=seed, feats=feats.astype(np.float32), lens=lens,
                        chunk_feats=(chunk_feats if chunk_feats is not None else np.zeros((0, 80), np.float32)), **out)
    return out


def make_squeezeformer(path, streaming=True, seed=1000, lens=LENS, chunk_T=211, vocab=40, norm="layer_norm", required=-16,
                       **kw):
    from ppasr.model_utils.loss.ctc import CTCLoss
    from ppasr.model_utils.squeezeformer.encoder import SqueezeformerEncoder
    from ppasr.model_utils.utils.cmvn import GlobalCMVN
    kw = kw or dict(encoder_dim=64, output_size=64, attention_heads=4, num_blocks=4, reduce_idx=1, recover_idx=3,
                    feed_forward_expansion_factor=2, cnn_module_kernel=15, max_len=600)
    cfg = W.SqueezeformerConfig(input_dim=80, vocab_size=vocab, streaming=streaming, cnn_norm_type=norm, **kw)
    weights = W.init_squeezeformer_weights(cfg, seed=seed)
    cmvn = GlobalCMVN(t(weights["encoder.global_cmvn.mean"]), t(weights["encoder.global_cmvn.istd"]))
    # squeezeformer/model.py:35-50
    enc = SqueezeformerEncoder(input_size=cfg.input_dim, global_cmvn=cmvn,
                               time_reduction_layer_type="stream" if streaming else "conv1d", use_dynamic_chunk=streaming,
                               causal=streaming, encoder_dim=cfg.encoder_dim, output_size=cfg.output_size,
                               attention_heads=cfg.attention_heads, num_blocks=cfg.num_blocks, reduce_idx=cfg.reduce_idx,
                               recover_idx=cfg.recover_idx, feed_forward_expansion_factor=cfg.feed_forward_expansion_factor,
                               cnn_module_kernel=cfg.cnn_module_kernel, cnn_norm_type=cfg.cnn_norm_type,
                               adaptive_scale=cfg.adaptive_scale)
    ctc = CTCLoss(cfg.vocab_size, enc.output_size())
    load_into(enc, weights, "encoder.")
    load_into(ctc, weights, "ctc.")
    feats, lens, chunk_feats = inputs(lens, chunk_T if streaming else 0, seed)
    out = run_former(enc, ctc, feats, lens, chunk_feats, required)
    out["required_cache_size"] = np.array(required)
    np.savez_compressed(path, cfg=np.array(repr(cfg.to_dict())), seed=seed, feats=feats.astype(np.float32), lens=lens,
                        chunk_feats=(chunk_feats if chunk_feats is not None else np.zeros((0, 80), np.float32)), **out)
    return out


def make_efficient_conformer(path, streaming=False, seed=1000, norm="batch_norm", lens=LENS, chunk_T=211, vocab=40,
                             att_cache_step=1, **kw):
    """att_cache_step > 1 stores every att_cache_step-th channel of the final attention cache (all blocks, heads and frames)
    together with its full shape, to keep a large fixture under 1 MB."""
    from ppasr.model_utils.efficient_conformer.encoder import EfficientConformerEncoder
    from ppasr.model_utils.loss.ctc import CTCLoss
    from ppasr.model_utils.utils.cmvn import GlobalCMVN
    kw = kw or dict(output_size=64, attention_heads=4, linear_units=128, num_blocks=4, max_len=600, stride_layer_idx=1,
                    group_layer_idx=(0, 1))
    cfg = W.EfficientConformerConfig(input_dim=80, vocab_size=vocab, cnn_module_kernel=15, streaming=streaming,
                                     cnn_module_norm=norm, group_size=3, **kw)
    weights = W.init_efficient_conformer_weights(cfg, seed=seed)
    cmvn = GlobalCMVN(t(weights["encoder.global_cmvn.mean"]), t(weights["encoder.global_cmvn.istd"]))
    # efficient_conformer/model.py:34-47
    enc = EfficientConformerEncoder(input_size=cfg.input_dim, global_cmvn=cmvn, use_dynamic_chunk=streaming, causal=streaming,
                                    output_size=cfg.output_size, attention_heads=cfg.attention_heads,
                                    linear_units=cfg.linear_units, num_blocks=cfg.num_blocks,
                                    cnn_module_kernel=cfg.cnn_module_kernel, cnn_module_norm=cfg.cnn_module_norm,
                                    stride_layer_idx=cfg.stride_layer_idx, stride=cfg.stride,
                                    group_layer_idx=list(cfg.group_layer_idx), group_size=cfg.group_size,
                                    stride_kernel=cfg.stride_kernel)
    ctc = CTCLoss(cfg.vocab_size, enc.output_size())
    # StrideConformerEncoderLayer always builds concat_linear (efficient_conformer/encoder.py:453) but only reads it when
    # concat_after=True (:504-506), which no shipped config sets
    load_into(enc, weights, "encoder.", unused=("concat_linear",))
    load_into(ctc, weights, "ctc.")
    feats, lens, chunk_feats = inputs(lens, chunk_T if streaming else 0, seed)
    out = run_former(enc, ctc, feats, lens, chunk_feats)
    if att_cache_step > 1:
        att = out["chunk_att_cache"]
        out["chunk_att_cache_shape"] = np.array(att.shape)
        out["chunk_att_cache_step"] = np.array(att_cache_step)
        out["chunk_att_cache"] = np.ascontiguousarray(att[..., ::att_cache_step])
    np.savez_compressed(path, cfg=np.array(repr(cfg.to_dict())), seed=seed, feats=feats.astype(np.float32), lens=lens,
                        chunk_feats=(chunk_feats if chunk_feats is not None else np.zeros((0, 80), np.float32)), **out)
    return out


def make_deepspeech2(path, streaming, use_gru, seed=1000, lens=LENS, chunk_T=211, chunk_B=1, vocab=40, nl=3, H=64):
    """deepspeech2/model.py:24-72: CRNNEncoder + CTC head `decoder`; offline get_encoder_out for a ragged batch and, for the
    streaming (forward-RNN) model, a get_encoder_out_chunk chain carrying the state boxes. The recurrent cells themselves are
    torch.nn.LSTM/GRU inside the shim (same gate order and equations as paddle.nn.LSTM/GRU), so this pins the wiring
    (conv reshape, lengths, state-box split/concat, LayerNorm placement), not the cell arithmetic."""
    from ppasr.model_utils.deepspeech2.encoder import CRNNEncoder
    from ppasr.model_utils.loss.ctc import CTCLoss
    from ppasr.model_utils.utils.cmvn import GlobalCMVN
    cfg = W.DeepSpeech2Config(input_dim=80, vocab_size=vocab, num_rnn_layers=nl, rnn_size=H, use_gru=use_gru, streaming=streaming)
    weights = W.init_deepspeech2_weights(cfg, seed=seed)
    cmvn = GlobalCMVN(t(weights["encoder.global_cmvn.mean"]), t(weights["encoder.global_cmvn.istd"]))
    enc = CRNNEncoder(input_dim=cfg.input_dim, vocab_size=cfg.vocab_size, global_cmvn=cmvn, num_rnn_layers=cfg.num_rnn_layers,
                      rnn_size=cfg.rnn_size, rnn_direction="forward" if streaming else "bidirect", use_gru=use_gru)
    dec = CTCLoss(cfg.vocab_size, enc.output_size)
    load_into(enc, weights, "encoder.")
    load_into(dec, weights, "decoder.")
    enc.eval(), dec.eval()
    feats, lens, _ = inputs(lens, 0, seed)
    out = {}
    with torch.no_grad():
        eouts, eouts_len, _, _ = enc(t(feats), t(lens, "int64"))
        out["offline_logits"] = dec.ctc_lo(eouts).numpy()
        out["offline_probs"] = dec.softmax(eouts).numpy()
        out["offline_lens"] = eouts_len.numpy()
        chunk_feats = np.zeros((0, 80), np.float32)
        if streaming:
            chunk_feats = W.synthetic_fbank(chunk_B, chunk_T, 80, seed=seed + 3)
            h = c = None
            logits = []
            for (a, b) in stream_windows(chunk_feats.shape[1]):
                x = t(chunk_feats[:, a:b])
                eo, el, h, c = enc(x, t(np.array([b - a] * chunk_B), "int64"), h, c)
                logits.append(dec.ctc_lo(eo).numpy())
            out["chunk_logits"] = np.concatenate(logits, 1)
            if chunk_B == 1:
                chunk_feats, out["chunk_logits"] = chunk_feats[0], out["chunk_logits"][0]
            out["chunk_state_h"] = h.numpy()
            if c is not None:
                out["chunk_state_c"] = c.numpy()
    np.savez_compressed(path, cfg=np.array(repr(cfg.to_dict())), seed=seed, feats=feats.astype(np.float32), lens=lens,
                        chunk_feats=chunk_feats, **out)
    return out


if __name__ == "__main__":
    which = sys.argv[1:] or ["conformer"]
    if "conformer" in which:
        o = make_conformer(os.path.join(HERE, "encoder_golden_conformer_stream.npz"), streaming=True)
        print("conformer stream", {k: v.shape for k, v in o.items()})
        o = make_conformer(os.path.join(HERE, "encoder_golden_conformer_offline_bn.npz"), streaming=False, norm="batch_norm")
        print("conformer offline/bn", {k: v.shape for k, v in o.items()})
        for req in (32, 0):  # bounded / no attention history (encoder.py:255-260 next_cache_start)
            o = make_conformer(os.path.join(HERE, f"encoder_golden_conformer_stream_req{req}.npz"), streaming=True, seed=1002,
                               lens=(71,), required=req)
            print("conformer stream required", req, {k: np.shape(v) for k, v in o.items()})
    if "squeezeformer" in which:
        o = make_squeezeformer(os.path.join(HERE, "encoder_golden_squeezeformer_stream.npz"), streaming=True)
        print("squeezeformer stream", {k: v.shape for k, v in o.items()})
        o = make_squeezeformer(os.path.join(HERE, "encoder_golden_squeezeformer_offline.npz"), streaming=False)
        print("squeezeformer offline", {k: v.shape for k, v in o.items()})
        o = make_squeezeformer(os.path.join(HERE, "encoder_golden_squeezeformer_offline_bn.npz"), streaming=False,
                               norm="batch_norm", seed=1001)
        print("squeezeformer offline/bn", {k: v.shape for k, v in o.items()})
        o = make_squeezeformer(os.path.join(HERE, "encoder_golden_squeezeformer_stream_req32.npz"), streaming=True, seed=1003,
                               lens=(71,), chunk_T=67 + 64 * 2 + 21, required=32)
        print("squeezeformer stream required 32", {k: np.shape(v) for k, v in o.items()})
    if "efficient_conformer" in which:
        o = make_efficient_conformer(os.path.join(HERE, "encoder_golden_efficient_conformer_offline.npz"), streaming=False)
        print("efficient_conformer offline", {k: v.shape for k, v in o.items()})
        o = make_efficient_conformer(os.path.join(HERE, "encoder_golden_efficient_conformer_stream.npz"), streaming=True,
                                     norm="layer_norm")
        print("efficient_conformer stream", {k: v.shape for k, v in o.items()})
    if "deepspeech2" in which:
        for streaming, gru, tag in ((False, False, "offline_lstm"), (True, False, "stream_lstm"), (True, True, "stream_gru"),
                                    (False, True, "offline_gru")):
            o = make_deepspeech2(os.path.join(HERE, f"encoder_golden_deepspeech2_{tag}.npz"), streaming, gru)
            print("deepspeech2", tag, {k: v.shape for k, v in o.items()})
    if "gpu" in which:
        # Engine-size fixtures (d_model 256 / 4 heads / FFN 2048, the only widths the CUDA path is built for) for
        # tests/test_gpu_reference_golden.py: the CUDA path against the reference's own code, no oracle in between. Shapes
        # mirror cases of tests/test_gpu_parity.py that the engine is known to run.
        G = lambda n: os.path.join(HERE, f"encoder_golden_{n}.npz")  # noqa: E731
        make_conformer(G("conformer_gpu_stream"), streaming=True, lens=(131, 90), chunk_T=215, vocab=97, num_blocks=2)
        make_conformer(G("conformer_gpu_offline_bn"), streaming=False, norm="batch_norm", lens=(300, 200), vocab=97,
                       num_blocks=2)
        make_squeezeformer(G("squeezeformer_gpu_stream"), streaming=True, lens=(203, 150, 99), chunk_T=67 + 64 * 3, vocab=120,
                           num_blocks=4, reduce_idx=1, recover_idx=3)
        make_squeezeformer(G("squeezeformer_gpu_offline"), streaming=False, lens=(207, 150, 5), vocab=120, num_blocks=3,
                           reduce_idx=1, recover_idx=2)
        make_efficient_conformer(G("efficient_conformer_gpu_causal"), streaming=True, norm="layer_norm", lens=(203, 150, 99),
                                 chunk_T=0, vocab=120, num_blocks=2, group_layer_idx=(0, 1), stride_layer_idx=1)
        make_efficient_conformer(G("efficient_conformer_gpu_offline"), streaming=False, norm="batch_norm", lens=(207, 150, 5),
                                 vocab=120, num_blocks=2, group_layer_idx=(0, 1), stride_layer_idx=1)
        # forward_chunk of the Efficient Conformer (encoder.py:266-394): grouped attention on cache + chunk, the stride block and
        # half-rate blocks behind it; 67-frame windows incl. an odd last window. The 12-block one has the shipped layout
        # (configs/efficient_conformer.yml: group_layer_idx 0-3, stride_layer_idx 3).
        make_efficient_conformer(G("efficient_conformer_gpu_stream"), streaming=True, norm="layer_norm", lens=(203, 150, 99),
                                 chunk_T=67 + 64 * 3 + 24, vocab=120, num_blocks=4, group_layer_idx=(0, 1), stride_layer_idx=1,
                                 seed=1005)
        make_efficient_conformer(G("efficient_conformer_gpu_stream12"), streaming=True, norm="layer_norm", lens=(99,),
                                 chunk_T=67 + 64 * 5, vocab=120, num_blocks=12, group_layer_idx=(0, 1, 2, 3), stride_layer_idx=3,
                                 seed=1006, att_cache_step=4)
        make_deepspeech2(G("deepspeech2_gpu_stream_lstm"), True, False, lens=(203, 150, 99), chunk_T=67 + 64 * 2, chunk_B=2,
                         vocab=120, nl=2, H=256)
        make_deepspeech2(G("deepspeech2_gpu_offline_gru"), False, True, lens=(203, 150, 99), vocab=120, nl=2, H=256)
        print("gpu fixtures written")
