"""Efficient Conformer past 768 encoder frames (pytest -m gpu): grouped attention over more than 256 key groups.

grouped_attention_kernel keeps up to 4 blocks of 64 key groups resident in TMEM and recomputes the score blocks through the
same four slots beyond that. Checked here: the op against an fp32 restatement of attention.py:128-193 on both sides of the
4-block boundary (offline and streaming operand layouts, ragged key lengths), whole models offline and streaming against the
oracle and against the reference code's own outputs (tests/golden/effconf_long_golden.npz), a stream run to max_len and
PPASRPredictor.predict_stream on 41 s of audio. Tolerances as in test_gpu_parity.py: op 2e-2, logits 1e-2 of max |logit|.
"""
import ast
import os

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

FIXTURE = os.path.join(os.path.dirname(__file__), "golden", "effconf_long_golden.npz")
GCAP = 1672  # group capacity of the streaming caches at max_len 5000: ceil(4999 / 3) rounded up to a multiple of 8


def _grouped_ref(q2g, kk, vt, pos, T, Tgk, klens):
    """attention.py:128-193 in fp32 on the kernel's operands: S = [q+u | q+v] . [k | p]^T / sqrt(192), keys g with 3g >= len
    masked, softmax, P V, the (group, head, 192) tokens re-viewed as frames and rows >= T dropped."""
    B, H, Tg, _ = q2g.shape
    q = q2g.float()
    k = kk[:, :, :Tgk].float()
    v = vt[..., :Tgk].float().transpose(-1, -2)
    p = pos[:Tgk].float().view(Tgk, H, 192).transpose(0, 1)
    s = (q[..., :192] @ k.transpose(-1, -2) + q[..., 192:] @ p[None].transpose(-1, -2)) / 192 ** 0.5
    if klens is not None:
        mask = 3 * torch.arange(Tgk, device=q.device)[None, :] >= klens[:, None]
        s = s.masked_fill(mask[:, None, None, :], float("-inf"))
    o = torch.softmax(s, -1) @ v                                  # [B, H, Tg, 192]
    o = o.transpose(1, 2).reshape(B, Tg * 3, 256)[:, :T]
    return o.reshape(B * T, 256)


def _op(lib, q2g, kk, k_pitch, vt, vt_pitch, pos, B, T, Tgk, klens, cuda):
    from ppasr_b200 import _lib as L
    out = torch.zeros(B * T, 256, device=cuda, dtype=torch.bfloat16)
    L.check(lib.ppasr_b200_op_grouped_attention(L.ptr(q2g), L.ptr(kk), k_pitch, L.ptr(vt), vt_pitch, L.ptr(pos), L.ptr(out), B,
                                                4, T, Tgk, L.ptr(klens) if klens is not None else None, L.stream_ptr()))
    torch.cuda.synchronize()
    return out


def _rel_err(got, ref):
    return (got.float() - ref.float()).abs().max().item() / ref.float().abs().max().item()


@pytest.mark.parametrize("layout", ["offline", "streaming"])
@pytest.mark.parametrize("Tgk", [64, 256, 257, 320, 321, 512, 1667])
def test_grouped_attention_op_any_key_length(lib, cuda, Tgk, layout):
    torch.manual_seed(Tgk * 2 + (layout == "streaming"))
    H = 4
    if layout == "offline":   # queries == keys: k_pitch = Tg, V^T pitch = Tg rounded to 64 (build_plan), ragged lengths
        B, T = 2, 3 * Tgk - 1
        Tg = (T + 2) // 3
        k_pitch, vt_pitch = Tg, (Tg + 63) // 64 * 64
        klens = torch.tensor([T, max(1, T // 2 - 5)], device=cuda, dtype=torch.int32)
    else:                     # one 16-frame chunk of queries against the whole append-only cache (k_pitch = Gcap)
        B, T = 2, 16
        Tg = (T + 2) // 3
        k_pitch, vt_pitch = GCAP, GCAP
        klens = None
    q2g = (torch.randn(B, H, Tg, 384, device=cuda) * 0.5).to(torch.bfloat16)
    kk = (torch.randn(B, H, k_pitch, 192, device=cuda) * 0.5).to(torch.bfloat16)
    vt = torch.randn(B, H, 192, vt_pitch, device=cuda).to(torch.bfloat16)
    pos = (torch.randn(Tgk, 768, device=cuda) * 0.5).to(torch.bfloat16)
    out = _op(lib, q2g, kk, k_pitch, vt, vt_pitch, pos, B, T, Tgk, klens, cuda)
    ref = _grouped_ref(q2g, kk, vt, pos, T, Tgk, klens)
    err = _rel_err(out, ref)
    print(f"[grouped attention] {layout} Tgk={Tgk}: rel err {err:.3e}")
    assert err < 2e-2


def test_grouped_attention_op_ragged_blocks(lib, cuda):
    """One utterance's last valid key in block 0, one in block 5, one at the end of block 7 (recompute path)."""
    torch.manual_seed(7)
    B, H, Tgk = 3, 4, 512
    T = 3 * Tgk
    q2g = (torch.randn(B, H, Tgk, 384, device=cuda) * 0.5).to(torch.bfloat16)
    kk = (torch.randn(B, H, Tgk, 192, device=cuda) * 0.5).to(torch.bfloat16)
    vt = torch.randn(B, H, 192, Tgk, device=cuda).to(torch.bfloat16)
    pos = (torch.randn(Tgk, 768, device=cuda) * 0.5).to(torch.bfloat16)
    klens = torch.tensor([100, 3 * 330 - 2, T], device=cuda, dtype=torch.int32)   # 34, 330 and 512 valid groups
    out = _op(lib, q2g, kk, Tgk, vt, Tgk, pos, B, T, Tgk, klens, cuda)
    ref = _grouped_ref(q2g, kk, vt, pos, T, Tgk, klens)
    assert _rel_err(out, ref) < 2e-2


# ------------------------------------------------------------------------------------------------------------------------
def test_long_offline_matches_oracle_12_blocks(lib, cuda):
    """Shipped 12-block layout, ragged: T' = 1001 (334 key groups, recompute path) and T' = 699 (< 768) in one batch."""
    from test_gpu_parity import _run_model
    _run_model(cuda, 12, 2, 4007, [4007, 2800], model="efficient_conformer")


def test_offline_near_max_len_matches_oracle(lib, cuda):
    """One utterance of T' = 4991 encoder frames (1664 key groups, max_len 5000); grouped blocks 0-3 and the stride block."""
    from test_gpu_parity import _run_model
    _run_model(cuda, 4, 1, 19967, [19967], model="efficient_conformer", group_layer_idx=(0, 1, 2, 3), stride_layer_idx=3)


def _fixture():
    from ppasr_b200 import weights as W
    g = np.load(FIXTURE)
    cfg = W.EfficientConformerConfig(**ast.literal_eval(str(g["cfg"])))
    return g, cfg, W.init_efficient_conformer_weights(cfg, seed=int(g["seed"]))


def test_long_offline_matches_reference_code(lib, cuda):
    from ppasr_b200.engine import ConformerEngine
    g, cfg, w = _fixture()
    eng = ConformerEngine(cfg, w)
    eng.encode(torch.from_numpy(g["feats"].astype(np.float32)).to(cuda), [int(v) for v in g["lens"]])
    logits = eng.ctc_logits().float().cpu().numpy()
    eng.close()
    ref = g["offline_logits"]
    assert logits.shape == ref.shape and ref.shape[1] * 2 > 768
    scale = float(np.abs(ref).max())
    worst = float(np.abs(logits - ref).max()) / scale
    top2 = np.sort(ref, -1)[..., -2:]
    big = (top2[..., 1] - top2[..., 0]) > 3.0 * worst * scale
    same = logits.argmax(-1) == ref.argmax(-1)
    print(f"[effconf long offline] logits rel err {worst:.3e}; arg-max agreement {int(same.sum())}/{same.size}")
    assert worst < 1e-2
    assert bool((same | ~big).all()) and same.mean() >= 0.95


def test_long_chunk_chain_matches_reference_code(lib, cuda):
    """The reference's forward_chunk chain past 768 encoder frames, chunk by chunk."""
    from ppasr_b200.infer_utils.inference_predictor import InferencePredictor
    from oracle.conformer_oracle import stream_windows
    g, cfg, w = _fixture()
    pred = InferencePredictor({"encoder_conf": cfg.to_dict(), "preprocess_conf": {"n_mels": 80}}, "efficient_conformer",
                              streaming=True, weights=w)
    cf = g["feats"][0, :int(g["chunk_T"])].astype(np.float32)
    ref = g["chunk_logits"]
    off, worst = 0, 0.0
    for (a, b) in stream_windows(cf.shape[0], is_end=True):
        pred.predict_chunk_conformer(np.ascontiguousarray(cf[None, a:b]), int(g["required_cache_size"]))
        lg = pred.engine.ctc_logits().float().cpu().numpy()[0]
        r = ref[off:off + lg.shape[0]]
        assert lg.shape == r.shape
        worst = max(worst, float(np.abs(lg - r).max()) / float(np.abs(r).max()))
        assert worst < 1e-2, (a, worst)
        off += lg.shape[0]
    assert off == ref.shape[0] and 2 * off > 768
    print(f"[effconf long chunk chain] {off} output frames, worst chunk rel err {worst:.3e}")
    pred.reset_stream()


def test_long_lockstep_streams_across_reset_match_oracle(lib, cuda):
    """Two lock-step utterances streamed to 1104 encoder frames, reset_stream, then two new ones to 1040 frames: the second
    stream's partially filled last groups must read zeros where the first stream wrote (the reset clears what it used)."""
    from oracle.efficient_conformer_oracle import EfficientConformerConf, EfficientConformerOracle
    from ppasr_b200.infer_utils.inference_predictor import InferencePredictor
    from ppasr_b200.weights import EfficientConformerConfig, init_efficient_conformer_weights, synthetic_fbank
    cfg = EfficientConformerConfig(num_blocks=4, vocab_size=120, group_layer_idx=(0, 1, 2, 3), stride_layer_idx=3)
    w = init_efficient_conformer_weights(cfg)
    orc = EfficientConformerOracle(EfficientConformerConf(**cfg.to_dict()), w)
    pred = InferencePredictor({"encoder_conf": cfg.to_dict(), "preprocess_conf": {"n_mels": 80}}, "efficient_conformer",
                              streaming=True, weights=w)
    for n_win, seed in ((69, 11), (65, 12)):
        feats = synthetic_fbank(2, 67 + 64 * (n_win - 1), seed=seed)
        states = [(torch.zeros(0, 0, 0, 0), torch.zeros(0, 0, 0, 0), 0) for _ in range(2)]
        worst = 0.0
        for s in range(0, feats.shape[1] - 6, 64):
            ch = feats[:, s:s + 67]
            refs = []
            for b in range(2):
                att, cnn, off = states[b]
                r, att, cnn = orc.get_encoder_out_chunk(torch.from_numpy(ch[b:b + 1]), off, -16, att, cnn, return_logits=True)
                states[b] = (att, cnn, off + r.shape[1])
                refs.append(r)
            ref = torch.cat(refs, 0)
            pred.predict_chunk_conformer(ch, -16)
            lg = pred.engine.ctc_logits().float().cpu()
            worst = max(worst, ((lg - ref).abs().max() / ref.abs().max()).item())
            assert worst < 1e-2, (n_win, s, worst)
        assert states[0][0].shape[2] == 16 * n_win > 768
        print(f"[effconf lock-step stream] {16 * n_win} encoder frames: worst chunk rel err {worst:.3e}")
        pred.reset_stream()


def test_stream_to_max_len_is_refused_cleanly(lib, cuda):
    """A stream that would pass the positional table (max_len 5000) gets the positional-table error, and the context keeps
    working after reset_stream."""
    from ppasr_b200.infer_utils.inference_predictor import InferencePredictor
    from ppasr_b200.weights import EfficientConformerConfig, init_efficient_conformer_weights, synthetic_fbank
    cfg = EfficientConformerConfig(num_blocks=4, vocab_size=120, group_layer_idx=(0, 1, 2, 3), stride_layer_idx=3)
    pred = InferencePredictor({"encoder_conf": cfg.to_dict(), "preprocess_conf": {"n_mels": 80}}, "efficient_conformer",
                              streaming=True, weights=init_efficient_conformer_weights(cfg))
    big = synthetic_fbank(1, 64 * 62 + 3, seed=5)   # 992 encoder frames per call
    small = synthetic_fbank(1, 67, seed=6)           # 16
    for _ in range(5):
        probs = pred.predict_chunk_conformer(big, -16)
        assert np.isfinite(probs).all()
    for _ in range(2):                               # 4960 -> 4992 frames
        pred.predict_chunk_conformer(small, -16)
    assert int(pred.offset[0]) * 2 == 4992
    with pytest.raises(Exception, match="max_len"):
        pred.predict_chunk_conformer(small, -16)    # 5008 >= max_len
    pred.reset_stream()
    probs = pred.predict_chunk_conformer(small, -16)
    assert probs.shape[1] == 8 and np.isfinite(probs).all()
    pred.reset_stream()


def test_predict_stream_41_seconds_of_audio(lib, cuda):
    """PPASRPredictor.predict_stream (use_model efficient_conformer) over 41 s of 16 kHz audio in 0.5 s pieces."""
    from ppasr_b200.predict import PPASRPredictor
    from ppasr_b200 import weights as W
    cfg = W.EfficientConformerConfig(num_blocks=4, vocab_size=150, group_layer_idx=(0, 1, 2, 3), stride_layer_idx=3)
    p = PPASRPredictor({"use_model": "efficient_conformer", "streaming": True, "decoder": "ctc_greedy",
                        "encoder_conf": cfg.to_dict(), "preprocess_conf": {"feature_method": "fbank", "n_mels": 80}},
                       vocab_list=W.make_vocab(150), weights=W.init_efficient_conformer_weights(cfg))
    rng = np.random.RandomState(3)
    n = 41 * 16000
    t = np.arange(n) / 16000.0
    audio = (0.3 * np.sin(2 * np.pi * (200 + 150 * np.sin(0.7 * t)) * t) + 0.05 * rng.randn(n)) * 32767
    audio = audio.astype(np.int16)
    piece, res = 8000, None
    for s in range(0, n, piece):
        r = p.predict_stream(audio[s:s + piece], is_end=s + piece >= n)
        res = r if r is not None else res
    assert res is not None and isinstance(res["text"], str)
    assert int(p.predictor.offset[0]) * 2 > 768   # the grouped blocks attended more than 256 key groups
    p.reset_stream()
