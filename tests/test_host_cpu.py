"""CPU tests: the C-ABI library loads and exports every symbol of include/ppasr_b200.h, fails loudly
without a GPU, and the host-side logic (weights, sharding, gloo all-gather) behaves."""
import ctypes
import os
import re
import socket
import subprocess
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def header_symbols():
    src = open(os.path.join(ROOT, "include", "ppasr_b200.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(ppasr_b200_[a-z0-9_]+)\s*\(", src)))


def test_library_exports_every_header_symbol(lib):
    from ppasr_b200 import _lib
    syms = header_symbols()
    assert len(syms) >= 20
    for s in syms:
        assert hasattr(lib, s), f"{s} declared in include/ppasr_b200.h but not exported"
    for s in syms:
        if s in ("ppasr_b200_last_error", "ppasr_b200_abi_version"):
            continue
        assert s in _lib.PROTOTYPES, f"{s} has no ctypes prototype in ppasr_b200/_lib.py"
    assert lib.ppasr_b200_abi_version() == 3


def test_config_struct_matches_header():
    import re
    from ppasr_b200.engine import Config
    hdr = open(os.path.join(os.path.dirname(__file__), "..", "include", "ppasr_b200.h")).read()
    body = hdr[hdr.index("typedef struct ppasr_b200_config {"):hdr.index("} ppasr_b200_config;")]
    body = re.sub(r"/\*.*?\*/", "", body, flags=re.S)
    names = re.findall(r"int32_t\s+(\w+)(\[(\d+)\])?;", body)
    n_ints = sum(int(n[2]) if n[2] else 1 for n in names)
    assert ctypes.sizeof(Config) == 4 * n_ints
    assert [n[0] for n in names] == [f[0] for f in Config._fields_]


def test_create_validates_and_finalize_reports_missing(lib):
    from ppasr_b200 import _lib
    from ppasr_b200.engine import Config
    c = Config(model_type=0, feat_dim=80, d_model=256, n_heads=4, ffn_dim=2048, n_layers=1, conv_kernel=15, causal=1,
               conv_norm=0, vocab_size=100, max_len=5000)
    ctx = ctypes.c_void_p()
    assert lib.ppasr_b200_create(ctypes.byref(c), ctypes.byref(ctx)) == 0
    bad = Config(model_type=9, feat_dim=80, d_model=256, n_heads=4, ffn_dim=2048, n_layers=1, conv_kernel=15,
                 vocab_size=100, max_len=5000)
    ctx2 = ctypes.c_void_p()
    assert lib.ppasr_b200_create(ctypes.byref(bad), ctypes.byref(ctx2)) != 0
    assert b"model_type" in lib.ppasr_b200_last_error()
    if not torch.cuda.is_available():
        # no device: must fail loudly, never fall back
        rc = lib.ppasr_b200_finalize(ctx)
        assert rc != 0 and len(lib.ppasr_b200_last_error()) > 0
        with pytest.raises(_lib.PPASRB200Error):
            _lib.check(rc)
    lib.ppasr_b200_destroy(ctx)


def test_engine_refuses_without_gpu():
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    from ppasr_b200 import _lib
    from ppasr_b200.engine import ConformerEngine
    from ppasr_b200.weights import ConformerConfig
    with pytest.raises(_lib.PPASRB200Error):
        ConformerEngine(ConformerConfig(num_blocks=1, vocab_size=10), {})
    from ppasr_b200.decoders.ctc_greedy_decoder import greedy_decoder
    with pytest.raises(_lib.PPASRB200Error):
        greedy_decoder(np.ones((3, 4), dtype=np.float32) / 4, ["a", "b", "c", "d"])


def test_product_never_imports_oracle():
    for dirpath, _, files in os.walk(os.path.join(ROOT, "ppasr_b200")):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                txt = open(os.path.join(dirpath, f), encoding="utf-8").read()
                assert "import oracle" not in txt and "from oracle" not in txt, f


def test_weight_shapes_and_counts():
    from ppasr_b200.weights import ConformerConfig, conformer_param_shapes, init_conformer_weights, make_vocab
    cfg = ConformerConfig()
    shapes = conformer_param_shapes(cfg)
    enc = sum(int(np.prod(s)) for n, s in shapes.items() if n.startswith("encoder.") and "global_cmvn" not in n)
    assert enc == 33_464_576 - 0 or abs(enc - 33.46e6) < 0.02e6  # SURVEY Appendix B: 33.46 M encoder params
    w = init_conformer_weights(ConformerConfig(num_blocks=1, vocab_size=50))
    assert w["encoder.embed.out.0.weight"].shape == (256 * 19, 256)
    assert w["encoder.encoders.0.feed_forward.w_1.weight"].shape == (256, 2048)
    v = make_vocab(4233)
    assert len(v) == 4233 and v[0] == "<blank>" and v[-1] == "<eos>"


def test_out_frames_and_shard_range():
    from ppasr_b200.engine import out_frames
    from ppasr_b200.parallel import shard_range
    assert [out_frames(t) for t in (498, 998, 2998, 67, 7, 6)] == [123, 248, 748, 16, 1, 0]
    for n, w in ((256, 8), (33, 4), (5, 8)):
        cover = []
        for r in range(w):
            s, e = shard_range(n, w, r)
            cover += list(range(s, e))
        assert cover == list(range(n))
    assert shard_range(256, 8, 3) == (96, 128)


WORKER = r'''
import os, sys
sys.path.insert(0, {root!r})
import torch, torch.distributed as dist
from ppasr_b200.parallel import shard_range, all_gather_results, all_gather_records, unpack_records
dist.init_process_group("gloo", rank=int(os.environ["RANK"]), world_size=int(os.environ["WORLD_SIZE"]))
rank, world = dist.get_rank(), dist.get_world_size()
N, L = 7, 6
g = torch.Generator().manual_seed(0)
ids_all = torch.randint(1, 50, (N, L), generator=g, dtype=torch.int32)
lens_all = torch.randint(0, L + 1, (N,), generator=g, dtype=torch.int32)
sc_all = torch.rand(N, generator=g)
s, e = shard_range(N, world, rank)
ids, ol, sc = all_gather_results(ids_all[s:e].clone(), lens_all[s:e].clone(), sc_all[s:e].clone(), N, L)
assert torch.equal(ids, ids_all) and torch.equal(ol, lens_all) and torch.equal(sc, sc_all), "gather mismatch"
# the serving-loop form: preallocated record / gathered buffers reused over steps, records split on the host (NumPy)
max_local = (N + world - 1) // world
rec = torch.zeros((max_local, L + 2), dtype=torch.int32)
out = torch.empty((world * max_local, L + 2), dtype=torch.int32)
for step in range(2):
    g2 = all_gather_records(ids_all[s:e].clone(), lens_all[s:e].clone(), sc_all[s:e].clone(), N, L, rec=rec, out=out)
    assert g2.data_ptr() == out.data_ptr()
    hi, hl, hs = unpack_records(g2.numpy(), N, world, L)
    assert (hi == ids_all.numpy()).all() and (hl == lens_all.numpy()).all() and (hs == sc_all.numpy()).all(), "records mismatch"
dist.barrier(); dist.destroy_process_group()
print("RANK_OK", rank)
'''


def test_gloo_world2_all_gather(tmp_path):
    """The N>1 path: contiguous shards + ONE all-gather reproduce the single-process result (gloo, world 2)."""
    script = tmp_path / "worker.py"
    script.write_text(WORKER.format(root=ROOT))
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    procs = []
    for r in range(2):
        env = dict(os.environ, RANK=str(r), WORLD_SIZE="2", MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
        procs.append(subprocess.Popen([sys.executable, str(script)], env=env, stdout=subprocess.PIPE,
                                      stderr=subprocess.STDOUT, text=True))
    for p in procs:
        out, _ = p.communicate(timeout=120)
        assert p.returncode == 0 and "RANK_OK" in out, out


def test_header_is_plain_c_and_links_from_c(tmp_path):
    """The boundary is a C ABI: include/ppasr_b200.h compiles as C99 and a C program links against the library."""
    import subprocess
    root = os.path.join(os.path.dirname(__file__), "..")
    exe = str(tmp_path / "c_abi_demo")
    libdir = os.path.abspath(os.path.join(root, "ppasr_b200", "lib"))
    r = subprocess.run(["gcc", "-std=c99", "-Wall", "-Werror", "-I" + os.path.join(root, "include"),
                        os.path.join(root, "examples", "c_abi_demo.c"), "-L" + libdir, "-lppasr_b200",
                        "-Wl,-rpath," + libdir, "-o", exe], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    out = subprocess.run([exe], capture_output=True, text=True)
    assert out.returncode == 0 and "out_frames(998) = 248" in out.stdout and "fbank_frames(160000) = 998" in out.stdout


def test_pdiparams_roundtrip(tmp_path):
    """model.pdiparams (+ .info) reader: LoDTensor stream layout restated from the Paddle sources (unverified against a real
    file); the writer emits the same layout so at least the parser, dtype / dims decoding and name mapping are exercised."""
    from ppasr_b200.weights import (ConformerConfig, init_conformer_weights, load_pdiparams, save_pdiparams)
    cfg = ConformerConfig(num_blocks=1, vocab_size=40)
    w = init_conformer_weights(cfg)
    p = str(tmp_path / "model.pdiparams")
    save_pdiparams(p, w)
    r = load_pdiparams(p)
    assert list(r) == list(w)
    for k in w:
        assert r[k].shape == w[k].shape and np.array_equal(r[k], w[k])
    os.remove(p + ".info")
    r2 = load_pdiparams(p)
    assert list(r2)[0] == "param_0" and len(r2) == len(w)


def test_detokenize_matches_reference_join():
    """parallel.detokenize (vectorised) == ''.join(vocabulary[i] ...).replace('<space>', ' ') of ctc_greedy_decoder.py:27-31."""
    from ppasr_b200.parallel import detokenize
    rng = np.random.RandomState(0)
    vocab = ["<blank>", "<unk>", "<space>"] + [chr(0x4E00 + i) for i in range(50)] + ["ab", "<eos>"]
    ids = rng.randint(0, len(vocab), size=(7, 33)).astype(np.int32)
    lens = np.array([33, 0, 5, 17, 1, 32, 9], dtype=np.int32)
    ref = ["".join(vocab[int(i)] for i in ids[b, :lens[b]]).replace("<space>", " ") for b in range(7)]
    assert detokenize(ids, lens, vocab) == ref
    vocab2 = list(reversed(vocab))  # a different vocabulary object must not hit the cached table of the first one
    ref2 = ["".join(vocab2[int(i)] for i in ids[b, :lens[b]]).replace("<space>", " ") for b in range(7)]
    assert detokenize(ids, lens, vocab2) == ref2


def test_stream_scheduler_window_logic_cpu(monkeypatch):
    """StreamScheduler host logic with a fake engine (and the oracle's chunk decoder: the product one needs the GPU): each session is cut into exactly the reference's windows (67 frames,
    stride 64, short tail at is_end: predict.py:277-300 == oracle stream_windows), sessions are batched by window length,
    slots are unique inside a step and recycled on close."""
    from oracle.conformer_oracle import stream_windows
    from ppasr_b200.infer_utils import stream_scheduler as SS

    class FakeEngine:
        def __init__(self):
            self.calls = []

        def sessions_init(self, n):
            self.n = n

        def sessions_reset(self, slot):
            pass

        def sessions_step(self, batch, slots, required):
            assert len(set(slots)) == len(slots)
            self.calls.append((batch.copy(), list(slots)))
            self.last = batch

        def ctc_probs(self, to_host=True):
            B, t, _ = self.last.shape
            Tp = ((t - 1) // 2 - 1) // 2
            p = np.zeros((B, Tp, 5), dtype=np.float32)
            p[:, :, 0] = 1.0
            return p

    class FakePred:
        use_model, streaming = "conformer", True

        class model_config:
            input_dim = 4

        def __init__(self):
            self.engine = FakeEngine()

    from oracle import decoders_oracle as DO
    monkeypatch.setattr(SS, "greedy_decoder_chunk", DO.greedy_decoder_chunk)
    pred = FakePred()
    sch = SS.StreamScheduler(pred, ["<blank>", "a", "b", "c", "d"], max_sessions=3)
    lens = {0: 67 + 64 * 2 + 20, 1: 67 + 5, 2: 30}
    feats = {k: np.arange(n * 4, dtype=np.float32).reshape(n, 4) + 1000 * k for k, n in lens.items()}
    sids = {k: sch.open() for k in lens}
    seen = {k: [] for k in lens}
    pos = {k: 0 for k in lens}
    for rnd in range(40):
        for k in lens:
            n = min(45, lens[k] - pos[k])
            if n > 0:
                sch.feed(sids[k], feats[k][pos[k]:pos[k] + n], is_end=(pos[k] + n >= lens[k]))
                pos[k] += n
        before = len(pred.engine.calls)
        sch.step()
        for batch, slots in pred.engine.calls[before:]:
            for b, slot in enumerate(slots):
                k = [kk for kk in lens if sch._sessions[sids[kk]].slot == slot][0]
                seen[k].append(batch[b])
        if all(pos[k] >= lens[k] for k in lens) and not sch.pending():
            break
    for k, n in lens.items():
        wins = stream_windows(n, is_end=True)
        assert len(seen[k]) == len(wins), (k, len(seen[k]), wins)
        for w, (s, e) in zip(seen[k], wins):
            assert np.array_equal(w, feats[k][s:e])
    for k in lens:
        sch.close(sids[k])
    assert sorted(sch._free) == [0, 1, 2]
    with pytest.raises(Exception):
        SS.StreamScheduler(type("P", (), {"use_model": "deepspeech2", "streaming": True})(), [], 1)


def test_read_vocab_file_matches_reference_golden(tmp_path):
    """weights.read_vocab_file == TextFeaturizer.vocab_list of the reference run on the same file
    (tests/golden/make_vocab_golden.py; text_featurizer.py:52-59)."""
    import json
    from ppasr_b200.weights import read_vocab_file
    g = json.load(open(os.path.join(os.path.dirname(__file__), "golden", "vocab_golden.json"), encoding="utf-8"))
    p = tmp_path / "vocabulary.txt"
    p.write_text(g["file"], encoding="utf-8")
    assert read_vocab_file(str(p)) == g["vocab_list"] and len(g["vocab_list"]) == g["vocab_size"]


def test_model_utils_surface_cpu(monkeypatch, tmp_path):
    """ppasr_b200.model_utils: the reference's model-level names (conformer/model.py:148-184, deepspeech2/model.py:62-72) over
    InferencePredictor -- argument plumbing, lazy engine construction from set_state_dict + mean_istd.json, the
    continuation rule of the device-resident caches, and the errors. The engine itself is replaced by a recorder (GPU only)."""
    import json
    import ppasr_b200.model_utils as MU

    made = []

    class FakePredictor:
        def __init__(self, configs, use_model, streaming=True, weights=None, vocab_size=None, device=0, **kw):
            self.args = dict(configs=configs, use_model=use_model, streaming=streaming, weights=weights, vocab_size=vocab_size, kw=kw)
            self.offset = np.array([0], dtype=np.int32)
            self.att_cache = np.zeros([0, 0, 0, 0], np.float32)
            self.cnn_cache = np.zeros([0, 0, 0, 0], np.float32)
            self.output_state_h = self.output_state_c = None
            self.resets = 0
            self.engine = self
            made.append(self)

        def close(self):
            self.closed = True

        def predict(self, speech, lens):
            assert speech.dtype == np.float32 and lens.dtype == np.int64
            return np.full((speech.shape[0], 3, 5), 0.2, np.float32)

        def reset_stream(self):
            self.resets += 1
            self.offset = np.array([0], dtype=np.int32)
            self.att_cache = np.zeros([0, 0, 0, 0], np.float32)
            self.output_state_h = None

        def predict_chunk_conformer(self, x, req):
            assert x.dtype == np.float32 and isinstance(req, int)
            self.offset = self.offset + 16
            self.att_cache = np.ones([2, 4, int(self.offset[0]), 128], np.float32)
            self.cnn_cache = np.ones([2, 1, 256, 14], np.float32)
            return np.full((1, 16, 5), 0.2, np.float32)

        def predict_chunk_deepspeech(self, x):
            self.output_state_h = np.zeros((2, x.shape[0], 8), np.float32)
            self.output_state_c = np.zeros((2, x.shape[0], 8), np.float32)
            return np.full((x.shape[0], 16, 5), 0.2, np.float32), np.full([x.shape[0]], 16, np.int64)

    monkeypatch.setattr(MU, "InferencePredictor", FakePredictor)
    mi = tmp_path / "mean_istd.json"
    mi.write_text(json.dumps({"mean": [1.0] * 80, "istd": [0.5] * 80}))
    m = MU.ConformerModel(input_dim=80, vocab_size=5, mean_istd_path=str(mi), streaming=True,
                          encoder_conf={"num_blocks": 2}, decoder_conf={"x": 1}, ctc_weight=0.3)
    with pytest.raises(Exception, match="no parameters"):
        m.get_encoder_out(np.zeros((1, 67, 80), np.float32), np.array([67]))
    m.set_state_dict({"ctc.ctc_lo.weight": np.zeros((256, 5), np.float32)})
    out = m.eval().get_encoder_out(np.zeros((2, 67, 80)), [67, 60])
    assert out.numpy().shape == (2, 3, 5) and isinstance(out.numpy(), np.ndarray)
    a = made[-1].args
    assert a["use_model"] == "conformer" and a["streaming"] is True and a["vocab_size"] == 5
    assert a["configs"]["encoder_conf"] == {"num_blocks": 2} and a["configs"]["preprocess_conf"] == {"n_mels": 80}
    assert np.allclose(a["weights"]["encoder.global_cmvn.istd"], 0.5) and "ctc.ctc_lo.weight" in a["weights"]
    # chunk API: empty caches start a stream, afterwards only the continuation is accepted
    x = np.zeros((1, 67, 80), np.float32)
    p1, att, cnn = m.get_encoder_out_chunk(x, np.array([0], np.int32), np.array([-16], np.int32), np.zeros([0, 0, 0, 0]), np.zeros([0, 0, 0, 0]))
    assert p1.shape == (1, 16, 5) and att.shape == (2, 4, 16, 128) and cnn.shape == (2, 1, 256, 14) and made[-1].resets == 1
    p2, att, cnn = m.get_encoder_out_chunk(x, 16, -16, att, cnn)
    assert att.shape == (2, 4, 32, 128) and made[-1].resets == 1
    with pytest.raises(Exception, match="continue the previous call"):
        m.get_encoder_out_chunk(x, 16, -16, att, cnn)
    with pytest.raises(Exception, match="offset 0"):
        m.get_encoder_out_chunk(x, 16, -16, None, None)
    m.get_encoder_out_chunk(x, 0, -16)              # restart
    assert made[-1].resets == 3
    with pytest.raises(Exception, match="outside the ppasr_b200 hot path"):
        m(x, [67], None, None)
    with pytest.raises(Exception, match="export"):
        m.export()
    n_before = len(made)
    m.set_state_dict({"ctc.ctc_lo.weight": np.zeros((256, 5), np.float32)})   # new parameters -> new engine on next use
    assert made[-1].closed
    m.get_encoder_out(np.zeros((1, 67, 80)), [67])
    assert len(made) == n_before + 1
    # DeepSpeech2: states instead of caches; EfficientConformer: device-resident caches like the Squeezeformer
    d = MU.DeepSpeech2Model(80, 5, str(mi), streaming=True, encoder_conf={"num_rnn_layers": 2, "rnn_size": 8},
                            weights={"decoder.ctc_lo.weight": np.zeros((8, 5), np.float32)})
    pr, ln, h, c = d.get_encoder_out_chunk(np.zeros((3, 67, 80)), np.array([67] * 3))
    assert pr.shape == (3, 16, 5) and ln.tolist() == [16] * 3 and h.shape == (2, 3, 8) and c.shape == (2, 3, 8)
    d.get_encoder_out_chunk(np.zeros((3, 67, 80)), np.array([67] * 3), h, c)
    assert made[-1].args["use_model"] == "deepspeech2" and made[-1].resets == 1
    e = MU.EfficientConformerModel(80, 5, str(mi), weights={"ctc.ctc_lo.weight": np.zeros((256, 5), np.float32)})
    assert e.get_encoder_out(np.zeros((1, 67, 80)), [67]).shape == (1, 3, 5)
    pe, tok_a, tok_c = e.get_encoder_out_chunk(x, 0, -16)   # forward_chunk runs on the device; opaque continuation tokens
    assert tok_a.shape == (1, 1, 1, 1) and tok_c.shape == (1, 1, 1, 1) and made[-1].args["use_model"] == "efficient_conformer"
    assert {c.use_model for c in (MU.ConformerModel, MU.SqueezeformerModel, MU.EfficientConformerModel, MU.DeepSpeech2Model)} == \
        {"conformer", "squeezeformer", "efficient_conformer", "deepspeech2"}


def test_param_tables_match_reference_state_dict():
    """ppasr_b200/weights.py against the reference's own model classes (tests/golden/state_dict_golden.json, recorded by
    make_state_dict_golden.py from the reference <Family>Model classes built from the reference's shipped configs/*.yml, both
    `streaming` settings): the yaml encoder_conf goes through the same mapping InferencePredictor uses, and the parameter
    table the weight packer expects must be exactly the reference state_dict minus the attention decoder (never read by CTC
    inference) and minus parameters the reference constructs but never reads."""
    import json
    from ppasr_b200 import weights as W
    from ppasr_b200.infer_utils.inference_predictor import model_config_from
    g = json.load(open(os.path.join(os.path.dirname(__file__), "golden", "state_dict_golden.json"), encoding="utf-8"))
    tables = {"conformer": W.conformer_param_shapes, "squeezeformer": W.squeezeformer_param_shapes,
              "efficient_conformer": W.efficient_conformer_param_shapes, "deepspeech2": W.deepspeech2_param_shapes}
    # built by the reference but unused at inference: StrideConformerEncoderLayer.concat_linear (efficient_conformer/encoder.py:453,
    # read only when concat_after=True)
    unused = ("concat_linear",)
    assert len(g["models"]) == 8
    for m in g["models"]:
        cfg = model_config_from(m["use_model"], m["encoder_conf"], g["n_mels"], g["vocab_size"], m["streaming"])
        mine = {k: list(v) for k, v in tables[m["use_model"]](cfg).items()}
        ref = {k: v for k, v in m["state_dict"].items() if not any(u in k for u in unused)}
        assert set(mine) == set(ref), (m["use_model"], m["streaming"], sorted(set(mine) ^ set(ref))[:8])
        bad = {k: (mine[k], ref[k]) for k in mine if mine[k] != ref[k]}
        assert not bad, (m["use_model"], m["streaming"], list(bad.items())[:5])
        if m["use_model"] != "deepspeech2":
            assert m["attention_decoder_tensors"] > 0


def test_predictor_config_loading(tmp_path):
    """PPASRPredictor.load_configs (predict.py:36-60): yaml path or loaded config; no configs (model download) raises."""
    from ppasr_b200.predict import PPASRPredictor, SUPPORT_MODEL
    y = tmp_path / "c.yml"
    y.write_text("use_model: squeezeformer\nstreaming: True\ndecoder: ctc_greedy\nencoder_conf:\n  num_blocks: 12\n"
                 "preprocess_conf:\n  feature_method: fbank\n  n_mels: 80\n", encoding="utf-8")
    c = PPASRPredictor.load_configs(str(y))
    assert c["use_model"] == "squeezeformer" and c["encoder_conf"]["num_blocks"] == 12 and c["streaming"] is True
    assert PPASRPredictor.load_configs(c) is c
    with pytest.raises(Exception, match="needs the network"):
        PPASRPredictor.load_configs(None, "conformer_streaming_fbank_wenetspeech")
    assert set(SUPPORT_MODEL) == {"conformer", "squeezeformer", "efficient_conformer", "deepspeech2"}
    with pytest.raises(AssertionError, match="没有该模型"):
        PPASRPredictor({"use_model": "whisper"})


def test_inference_predictor_config_roundtrip(monkeypatch):
    """InferencePredictor builds the engine config from the yaml-style encoder_conf: a config's own to_dict() must survive the
    trip unchanged for all four families (the engine itself is replaced: it needs the GPU)."""
    from ppasr_b200 import weights as W
    from ppasr_b200.infer_utils import inference_predictor as IP
    made = []

    class FakeEngine:
        def __init__(self, cfg, w, device=0):
            made.append((cfg, w))

    monkeypatch.setattr(IP, "ConformerEngine", FakeEngine)
    cases = [("conformer", W.ConformerConfig(num_blocks=2, vocab_size=50, cnn_module_norm="batch_norm", streaming=False),
              W.init_conformer_weights),
             ("squeezeformer", W.SqueezeformerConfig(num_blocks=3, vocab_size=50, reduce_idx=1, recover_idx=2),
              W.init_squeezeformer_weights),
             ("efficient_conformer", W.EfficientConformerConfig(num_blocks=2, vocab_size=50, stride_layer_idx=1,
                                                                group_layer_idx=(0, 1)), W.init_efficient_conformer_weights),
             ("deepspeech2", W.DeepSpeech2Config(num_rnn_layers=2, rnn_size=64, vocab_size=50, use_gru=True),
              W.init_deepspeech2_weights)]
    for use_model, cfg, init in cases:
        w = init(cfg)
        p = IP.InferencePredictor({"encoder_conf": cfg.to_dict(), "preprocess_conf": {"n_mels": 80}}, use_model,
                                  streaming=cfg.streaming, weights=w)
        got, gw = made[-1]
        assert got.to_dict() == cfg.to_dict() and gw is w and p.model_config is got
        assert type(got) is type(cfg)
    with pytest.raises(Exception, match="use_gpu=False"):
        IP.InferencePredictor({}, "conformer", use_gpu=False)
    with pytest.raises(Exception, match="当前模型不支持该方法"):
        IP.InferencePredictor({}, "whisper")


def test_decoder_fallback_like_reference(tmp_path):
    """predict.py:92-105: the reference degrades to ctc_greedy with a warning when its beam-search decoder cannot be
    initialised. Here an unsupported configuration (KenLM binary LM, missing LM file, beam > 512) raises by default -- a
    stock config must not silently decode differently -- and degrades only with decoder_fallback=True."""
    from ppasr_b200.decoders.beam_search_decoder import UnsupportedDecoderConfig
    from ppasr_b200.predict import PPASRPredictor
    klm = tmp_path / "zh_giga.no_cna_cmn.prune01244.klm"
    klm.write_bytes(b"mmap lm http://kheafield.com/code format version 5\n\x00" + bytes(64))
    p = object.__new__(PPASRPredictor)
    p.configs = {"ctc_beam_search_decoder_conf": {"alpha": 2.2, "beta": 4.3, "beam_size": 300, "cutoff_prob": 0.99,
                                                  "cutoff_top_n": 40, "num_processes": 10, "language_model_path": str(klm)}}
    p.vocab_list = ["<blank>", "a"]
    p.decoder = "ctc_beam_search"
    with pytest.raises(UnsupportedDecoderConfig, match="ARPA"):
        p._init_decoder()
    with pytest.warns(UserWarning, match="ctc_greedy"):
        p._init_decoder(decoder_fallback=True)
    assert p.decoder == "ctc_greedy" and not hasattr(p, "beam_search_decoder")
    p.decoder = "ctc_beam_search"
    p.configs["ctc_beam_search_decoder_conf"]["language_model_path"] = str(tmp_path / "missing.klm")
    with pytest.raises(UnsupportedDecoderConfig, match="not found"):
        p._init_decoder()
    p.configs["ctc_beam_search_decoder_conf"].update(language_model_path=None, beam_size=600)
    with pytest.raises(UnsupportedDecoderConfig, match="beam_size 600"):
        p._init_decoder()
    p.decoder = "ctc_greedy"
    p._init_decoder()   # nothing to do


def _abi_config(**kw):
    from ppasr_b200.engine import Config
    c = Config()
    base = dict(model_type=0, feat_dim=80, d_model=256, n_heads=4, ffn_dim=2048, n_layers=2, conv_kernel=15, causal=1,
                conv_norm=0, vocab_size=50, max_len=5000, reduce_idx=-1, recover_idx=-1, time_reduce_kernel=0, use_gru=0,
                stride_layer_idx=-1, group_layer_mask=0, group_size=0, stride_kernel=0)
    base.update(kw)
    for k, v in base.items():
        setattr(c, k, v)
    return c


def test_c_abi_create_validates_configs_without_a_gpu():
    """ppasr_b200_create / out_frames / load_tensor / destroy are host-only: configuration errors come back as a status code
    plus ppasr_b200_last_error() (never a crash), valid configurations give a context whose out_frames follows the model's
    subsampling rule, and finalize (which needs the device) fails cleanly on a machine without one."""
    import ctypes
    from ppasr_b200 import _lib as L
    lib = L.load()

    def create(cfg):
        ctx = ctypes.c_void_p()
        return lib.ppasr_b200_create(ctypes.byref(cfg), ctypes.byref(ctx)), ctx

    for bad, msg in [(dict(d_model=512, n_heads=8), "d_model must be 256"), (dict(n_heads=8), "head dim"),
                     (dict(ffn_dim=1000), "ffn_dim"), (dict(conv_kernel=9), "conv_kernel"), (dict(model_type=7), "model_type"),
                     (dict(model_type=1, reduce_idx=3, recover_idx=1, time_reduce_kernel=1), "reduce_idx"),
                     (dict(model_type=2, d_model=2048), "rnn_size"),
                     (dict(model_type=3, group_size=2), "group_size"),
                     (dict(model_type=3, group_size=3, n_layers=4, stride_layer_idx=1, group_layer_mask=0b1100), "up to the stride"),
                     (dict(vocab_size=1), "bad config")]:
        rc, ctx = create(_abi_config(**bad))
        assert rc != 0 and not ctx.value, bad
        assert msg in lib.ppasr_b200_last_error().decode(), (bad, lib.ppasr_b200_last_error())
    # valid contexts: the output-frame rule (two k3/s2 convs; the Efficient Conformer's stride block halves again, ceil)
    rc, ctx = create(_abi_config())
    assert rc == 0 and ctx.value
    for T in (0, 6, 7, 10, 11, 67, 498, 998, 2998):
        want = ((T - 1) // 2 - 1) // 2 if T >= 7 else 0
        assert lib.ppasr_b200_out_frames(ctx, T) == want
    x = np.zeros((4, 4, 4, 4, 4), np.float32)
    shape = (ctypes.c_int64 * 5)(4, 4, 4, 4, 4)
    assert lib.ppasr_b200_load_tensor(ctx, b"x", x.ctypes.data_as(ctypes.c_void_p), 5, shape) != 0   # ndim > 4 rejected
    if not __import__("torch").cuda.is_available():
        assert lib.ppasr_b200_finalize(ctx) != 0 and lib.ppasr_b200_last_error()                      # needs the device
    assert lib.ppasr_b200_destroy(ctx) == 0 and lib.ppasr_b200_destroy(None) == 0
    rc, ctx = create(_abi_config(model_type=3, group_size=3, n_layers=4, stride_layer_idx=1, group_layer_mask=0b0011, stride_kernel=1))
    assert rc == 0
    assert [lib.ppasr_b200_out_frames(ctx, T) for T in (7, 67, 131, 135, 498)] == [1, 8, 16, 17, 62]
    lib.ppasr_b200_destroy(ctx)
    rc, ctx = create(_abi_config(model_type=2, d_model=1024, n_layers=5, causal=0))
    assert rc == 0 and lib.ppasr_b200_out_frames(ctx, 498) == 123
    lib.ppasr_b200_destroy(ctx)


def test_c_abi_state_errors_option_names_and_host_helpers_without_a_gpu():
    """Calls in the wrong state fail with a status + message before touching the device; set_option accepts the current
    switches and rejects removed ones; the sizing / naming helpers are pure host code."""
    import ctypes
    from ppasr_b200 import _lib as L
    lib = L.load()
    ctx = ctypes.c_void_p()
    assert lib.ppasr_b200_create(ctypes.byref(_abi_config()), ctypes.byref(ctx)) == 0
    feats = np.zeros((1, 67, 80), np.float32)
    p = feats.ctypes.data_as(ctypes.c_void_p)
    assert lib.ppasr_b200_encode(ctx, p, 0, None, 1, 67, None) != 0
    assert "finalize" in lib.ppasr_b200_last_error().decode()
    assert lib.ppasr_b200_encode(ctx, None, 0, None, 1, 67, None) != 0 and lib.ppasr_b200_encode(ctx, p, 0, None, 0, 67, None) != 0
    out = np.zeros((1, 16, 50), np.float32)
    assert lib.ppasr_b200_ctc_logits(ctx, out.ctypes.data_as(ctypes.c_void_p), 0, None) != 0
    assert "encode first" in lib.ppasr_b200_last_error().decode()
    assert lib.ppasr_b200_set_option(ctx, b"host_sync", 0) == 0 and lib.ppasr_b200_set_option(ctx, b"host_sync", 1) == 0
    assert lib.ppasr_b200_set_option(ctx, b"no_such_option", 1) != 0
    assert lib.ppasr_b200_set_option(None, b"host_sync", 1) != 0
    # removed kernel variants and unfused paths
    for gone in (b"qkv_wide", b"qkv_co", b"fused_dwconv", b"attn_out_v2", b"fused_ffn", b"fused_attn_out"):
        assert lib.ppasr_b200_set_option(ctx, gone, 1) != 0 and "unknown option" in lib.ppasr_b200_last_error().decode()
    assert lib.ppasr_b200_set_option(ctx, b"fused_conv", 0) == 0 and lib.ppasr_b200_set_option(ctx, b"fused_conv", 2) == 0
    assert lib.ppasr_b200_set_option(ctx, b"fused_conv", 1) != 0
    split = lib.ppasr_b200_get_ffn_split()
    assert lib.ppasr_b200_set_ffn_split(0) != 0 and lib.ppasr_b200_set_option(ctx, b"ffn_split", 3) != 0
    assert lib.ppasr_b200_get_ffn_split() == split
    lib.ppasr_b200_destroy(ctx)
    # sizes grow with the problem and are positive
    s1, s2, s3 = (lib.ppasr_b200_beam_state_bytes(1, 100, 10), lib.ppasr_b200_beam_state_bytes(2, 100, 10),
                  lib.ppasr_b200_beam_state_bytes(2, 200, 20))
    assert 0 < s1 < s2 < s3
    assert 0 < lib.ppasr_b200_beam_workspace_bytes(1, 50) < lib.ppasr_b200_beam_workspace_bytes(4, 500)
    names = [lib.ppasr_b200_profile_class_name(i).decode() for i in range(lib.ppasr_b200_profile_num_classes())]
    assert len(names) == len(set(names)) >= 8 and {"fused_ffn", "attention", "qkv_gemm"} <= set(names)
    assert lib.ppasr_b200_abi_version() == 3
