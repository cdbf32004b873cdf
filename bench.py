#!/usr/bin/env python
"""Benchmark of the B200-native PPASR hot path (contract: see the task statement / DESIGN.md §Measurement).

Default workload = BASELINE.json configs[1] (the config the headline metric is quoted on): conformer.yml streaming model,
batch 32 x 10 s synthetic fbank ([32, 998, 80] fp32) per GPU, fused CTC head + ctc_greedy. A "step" = one pass of the hot
path over one batch: encoder forward -> CTC projection -> decode (-> one NCCL all-gather of the decoded ids when N > 1).
Weak scaling: every GPU processes its own batch.

  python bench.py [--gpus N] [--steps K] [--warmup W]               # our arm (torchrun for N > 1)
  python bench.py --impl reference [--steps K] [--warmup W]         # CPU reference arm (oracle port, host threads)
  python bench.py --config {c1,c2,c3,c4,c5} ...                     # the other BASELINE configs, same JSON schema
  python bench.py --dump-outputs DIR ...                            # also write the last timed step's results to DIR

--config: c2 (default) conformer streaming b32x10s greedy; c1 deepspeech2 non-streaming 1x5s greedy (CPU arm: one core);
c3 conformer non-streaming b64x30s ctc_beam_search beam 10; c4 squeezeformer streaming b32x10s per GPU greedy; c5
efficient_conformer streaming chunk 16, b64x5s per GPU, ctc_beam_search beam 20 + 4-gram LM.

Timing: W >= 3 warm-up steps; the timed region is exactly K steps, bracketed by CUDA events on the launching streams (barrier +
synchronize on both sides, max over ranks). `ms_per_step` / `value` are its mean; pick K so that the region lasts about a
second or more. The single-stream, CUDA-graph, e2e and kernel-profile figures beside it also time K steps each.

--dump-outputs DIR: after the timed steps, the results of the last one as a caller of the timed path receives them (decoded
ids, their lengths and scores; with N > 1 the gathered results of all ranks) go to DIR/<name>.npy as float64. Weights and
inputs are seeded, so two builds run with the same arguments can be compared output for output.
"""
import argparse
import json
import os
import statistics
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

VOCAB = 4233
METRIC = "utterances_per_sec"

# algorithmic GFLOP per utterance: SURVEY.md §8(d) / BASELINE.md §2 (2 * MAC of the GEMM-shaped work)
CONFIGS = {
    "c1": dict(model="deepspeech2", streaming=False, batch=1, seconds=5, decoder="ctc_greedy", gflop_per_utt=30.2,
               name="deepspeech2 non-streaming 1x5s fbank[1,498,80] ctc_greedy (BASELINE configs[0])"),
    "c2": dict(model="conformer", streaming=True, batch=32, seconds=10, decoder="ctc_greedy", gflop_per_utt=23.17,
               name="conformer-streaming b32x10s fbank[32,998,80] ctc_greedy (BASELINE configs[1])"),
    "c3": dict(model="conformer", streaming=False, batch=64, seconds=30, decoder="ctc_beam_search", beam=10, gflop_per_utt=76.8,
               name="conformer non-streaming b64x30s fbank[64,2998,80] ctc_beam_search beam 10 (BASELINE configs[2])"),
    "c4": dict(model="squeezeformer", streaming=True, batch=32, seconds=10, decoder="ctc_greedy", gflop_per_utt=19.0,
               name="squeezeformer-streaming b32x10s per GPU fbank[32,998,80] ctc_greedy (BASELINE configs[3] shard)"),
    # 494 frames = 4.96 s: the reference's forward_chunk cannot take an ODD number of subsampled frames in the last window of a
    # stream (efficient_conformer/encoder.py:390 concatenates full-rate caches with x2-repeated half-rate ones; 5.00 s = 498
    # frames would end on an 11-frame chunk and raise there), so both arms run the longest length it accepts
    "c5": dict(model="efficient_conformer", streaming=True, batch=64, seconds=5, frames=494, decoder="ctc_beam_search", beam=20,
               lm=True, chunked=True, gflop_per_utt=8.24,
               name="efficient_conformer streaming chunk 16 (67-frame windows, stride 64) b64x5s per GPU "
                    "ctc_beam_search beam 20 + 4-gram LM (BASELINE configs[4] shard)"),
}


def frames_of(seconds):
    return 1 + (16000 * seconds - 400) // 160  # kaldi snip-edges (audio_featurizer.py:125-136): 5 s 498, 10 s 998, 30 s 2998


def model_setup(conf):
    from ppasr_b200 import weights as W
    m = conf["model"]
    if m == "squeezeformer":
        cfg = W.SqueezeformerConfig(vocab_size=VOCAB, streaming=conf["streaming"])
        return cfg, W.init_squeezeformer_weights(cfg)
    if m == "efficient_conformer":
        cfg = W.EfficientConformerConfig(vocab_size=VOCAB, streaming=conf["streaming"])
        return cfg, W.init_efficient_conformer_weights(cfg)
    if m == "deepspeech2":
        cfg = W.DeepSpeech2Config(vocab_size=VOCAB, streaming=conf["streaming"])
        return cfg, W.init_deepspeech2_weights(cfg)
    cfg = W.ConformerConfig(vocab_size=VOCAB, streaming=conf["streaming"])
    return cfg, W.init_conformer_weights(cfg)


def make_oracle(conf, cfg, w):
    m = conf["model"]
    if m == "squeezeformer":
        from oracle.squeezeformer_oracle import SqueezeformerConf, SqueezeformerOracle
        return SqueezeformerOracle(SqueezeformerConf(**cfg.to_dict()), w)
    if m == "efficient_conformer":
        from oracle.efficient_conformer_oracle import EfficientConformerConf, EfficientConformerOracle
        return EfficientConformerOracle(EfficientConformerConf(**cfg.to_dict()), w)
    if m == "deepspeech2":
        from oracle.deepspeech2_oracle import DeepSpeech2Conf, DeepSpeech2Oracle
        return DeepSpeech2Oracle(DeepSpeech2Conf(**cfg.to_dict()), w)
    from oracle.conformer_oracle import ConformerConf, ConformerOracle
    return ConformerOracle(ConformerConf(**cfg.to_dict()), w)


def synthetic_lm(vocab, order=4):
    """Seeded synthetic character 4-gram LM over the synthetic vocabulary (SURVEY.md §8d: no LM ships with the reference)."""
    from ppasr_b200.decoders.ngram_lm import NGramLM
    rng = np.random.RandomState(0)
    V = len(vocab)
    sents = [[vocab[2 + int(z) % (V - 3)] for z in rng.zipf(1.3, size=rng.randint(5, 30))] for _ in range(20000)]
    return NGramLM.from_counts(sents, order=order)


def stream_windows(num_frames, window=67, stride=64, context=7):
    """predict.py:281-297 with is_end on the last call."""
    return [(cur, min(cur + window, num_frames)) for cur in range(0, num_frames - context + 1, stride)]


def peaks():
    fallback = {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "src": "fallback"}
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        d = json.load(open(p))
        return {"hbm_gbs": float(d["hbm_gbs"]), "bf16_tflops": float(d["bf16_tflops"]),
                "bf16_tflops_sustained": float(d.get("bf16_tflops_sustained", d["bf16_tflops"])), "src": "measured"}
    except (OSError, ValueError, KeyError, TypeError):  # absent or in another shape: the profiling guide's fallback numbers
        return fallback


def ncu_traffic(kernel, grid=None):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of `kernel` from the committed `ncu --set full` capture
    (profiles/ncu_traffic.json, written by scripts/ncu_summary.py); None when no capture of this kernel is committed.
    `grid`: CTAs of the launch being reported -- a capture taken at another grid size (same bytes per CTA: one CTA = four
    posterior rows / one row tile) is scaled by the ratio."""
    try:
        d = json.load(open(os.path.join(ROOT, "profiles", "ncu_traffic.json")))
        v = d.get(kernel)
        if not v:
            return None
        t = float(v["dram_bytes_per_launch"])
        if grid and v.get("grid_size"):
            t *= float(grid) / float(v["grid_size"])
        return t
    except (OSError, ValueError, KeyError, TypeError):
        return None


def host_cores():
    """Usable host cores: CPU affinity capped by the cgroup CPU quota (the GPU boxes expose 128 logical CPUs
    but a 16-CPU quota; running the CPU arm with 128 threads is 100x slower than with 16)."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        q, per = open("/sys/fs/cgroup/cpu.max").read().split()
        if q != "max":
            n = min(n, max(1, int(int(q) / int(per))))
    except Exception:
        pass
    return n


def pin_to_gpu_numa(index):
    """Bind this rank to the CPUs NVML reports as local to its GPU (8-GPU boxes: two sockets). Best effort."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(index)
        n = os.cpu_count() or 64
        words = pynvml.nvmlDeviceGetCpuAffinity(h, (n + 63) // 64)
        cpus = {64 * i + b for i, w in enumerate(words) for b in range(64) if (w >> b) & 1}
        cur = os.sched_getaffinity(0)
        use = (cpus & cur) or cur
        os.sched_setaffinity(0, use)
        return len(use)
    except Exception:
        return None


class ClockSampler(threading.Thread):
    """Samples SM clock / throttle reasons through NVML while the timed region runs."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index = index
        self.samples = []
        self.reasons = set()
        self.max_mhz = None
        self.stop_flag = False
        self.ok = False
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            self.ok = True
        except Exception:
            self.ok = False

    def run(self):
        if not self.ok:
            return
        nv = self.nv
        names = {
            getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8): "hw_slowdown",
            getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40): "hw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20): "sw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4): "sw_power_cap",
        }
        while not self.stop_flag:
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                try:
                    r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, nm in names.items():
                    if bit and (r & bit):
                        self.reasons.add(nm)
            except Exception:
                pass
            time.sleep(0.005)

    def result(self):
        if not self.ok or not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": ["unavailable"]}
        return {"sm_mhz": int(statistics.median(self.samples)), "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(self.samples)}


def dump_outputs(path, ids, out_lens, scores):
    """path/{ids,out_lens,scores}.npy in float64 (exact for the int32 ids and lengths). Only the first out_lens[b] ids of an
    utterance are defined; the rest of its row is written as -1 so that dumps of two builds compare element for element."""
    ids, out_lens, scores = (t.cpu().numpy() if hasattr(t, "cpu") else np.asarray(t) for t in (ids, out_lens, scores))
    ids = np.where(np.arange(ids.shape[1])[None, :] < out_lens[:, None], ids, -1)
    os.makedirs(path, exist_ok=True)
    for name, a in (("ids", ids), ("out_lens", out_lens), ("scores", scores)):
        np.save(os.path.join(path, name + ".npy"), np.asarray(a, dtype=np.float64))


def quantiles(xs):
    xs = sorted(xs)
    n = len(xs)
    q = lambda f: xs[min(n - 1, max(0, int(round(f * (n - 1)))))]
    return {"p10": q(0.1), "p50": statistics.median(xs), "p90": q(0.9), "repetitions": n}


# ----------------------------------------------------------------------------------------------------------------------
# CPU reference arm: the oracle restatement of the reference graph (PyTorch-CPU fp32) + the reference decoders' restatement.
# Paddle is not installable offline, so kind = "port"; the restatement is pinned to the reference's own code
# (tests/test_encoder_golden_cpu.py, tests/golden/greedy_golden.*).
# ----------------------------------------------------------------------------------------------------------------------
class CpuReference:
    def __init__(self, conf, cfg, weights, vocab):
        import torch
        self.torch = torch
        self.conf, self.cfg, self.vocab = conf, cfg, vocab
        self.orc = make_oracle(conf, cfg, weights)
        self.frames = conf.get("frames") or frames_of(conf["seconds"])
        self.scorer = None
        if conf.get("lm"):
            from ppasr_b200.decoders.ngram_lm import Scorer
            self.scorer = Scorer(2.2, 4.3, None, vocab, lm=synthetic_lm(vocab))
        # full per-GPU batch for the greedy configs; the pure-Python beam search restatement is ~1 s per 10 s utterance, so
        # the beam configs time a bounded sample of the batch (declared in `sample`)
        self.sample_b = conf["batch"] if conf["decoder"] == "ctc_greedy" else min(conf["batch"], 2)

    def probs(self, feats, lens):
        torch = self.torch
        if self.conf.get("chunked"):
            outs = []
            for b in range(feats.shape[0]):
                att, cnn, off, rows = torch.zeros(0, 0, 0, 0), torch.zeros(0, 0, 0, 0), 0, []
                for (a, e) in stream_windows(int(lens[b])):
                    p, att, cnn = self.orc.get_encoder_out_chunk(torch.from_numpy(feats[b:b + 1, a:e]), off, -16, att, cnn)
                    off += p.shape[1]
                    rows.append(p[0])
                outs.append(torch.cat(rows, 0).numpy())
            return outs
        p = self.orc.get_encoder_out(torch.from_numpy(feats), torch.tensor(lens))
        return [x for x in p.numpy()]

    def step(self, feats, lens):
        from oracle import decoders_oracle as DO
        ps = self.probs(feats, lens)
        if self.conf["decoder"] == "ctc_greedy":
            return DO.greedy_decoder_batch(ps, self.vocab)
        return [DO.ctc_beam_search_decoding(p, self.vocab, self.conf["beam"], 0.99, 40, ext_scorer=self.scorer)[0][1] for p in ps]

    def choose_threads(self, feats, lens):
        """3-point probe of the intra-op thread count (all usable cores, half, a quarter) on a 4-utterance slice."""
        torch = self.torch
        cores = 1 if self.conf["model"] == "deepspeech2" else host_cores()  # BASELINE configs[0]: single core
        cands = sorted({max(1, cores), max(1, cores // 2), max(1, cores // 4)}, reverse=True)
        if len(cands) == 1:
            torch.set_num_threads(cands[0])
            return cands[0], {}
        nb = min(4, feats.shape[0])
        f, l = feats[:nb], lens[:nb]
        probe = {}
        for n in cands:
            torch.set_num_threads(n)
            self.probs(f, l)
            t0 = time.perf_counter()
            self.probs(f, l)
            probe[n] = time.perf_counter() - t0
        best = min(probe, key=probe.get)
        torch.set_num_threads(best)
        return best, {str(k): round(v, 4) for k, v in probe.items()}

    def describe(self, n_steps):
        c = self.conf
        what = f"{self.sample_b} of {c['batch']} utterances x {c['seconds']} s per step" if self.sample_b != c["batch"] else \
            f"the full batch of {c['batch']} utterances x {c['seconds']} s per step"
        return (f"{what}, {n_steps} timed steps: PyTorch-CPU fp32 oracle restatement of the reference Paddle graph + "
                f"{c['decoder']} restatement (Paddle not installable offline; restatement pinned to the reference code, "
                "tests/test_encoder_golden_cpu.py)")


def run_reference(args, conf):
    import torch
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from ppasr_b200.weights import make_vocab, synthetic_fbank
    cfg, w = model_setup(conf)
    vocab = make_vocab(VOCAB)
    ref = CpuReference(conf, cfg, w, vocab)
    feats = synthetic_fbank(ref.sample_b, ref.frames, seed=1234)
    lens = [ref.frames] * ref.sample_b
    threads, probe = ref.choose_threads(feats, lens)
    W = max(1, args.warmup)
    K = max(1, args.steps)
    for _ in range(W):
        ref.step(feats, lens)
    times = []
    for _ in range(K):
        t0 = time.perf_counter()
        ref.step(feats, lens)
        times.append(time.perf_counter() - t0)
    dt = sum(times) / len(times)
    value = ref.sample_b / dt
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": "utt/s", "n_gpus": args.gpus, "steps": K,
        "warmup": W, "ms_per_step": dt * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": conf["name"], "rtf": dt / (ref.sample_b * conf["seconds"]), "batch_per_step": ref.sample_b,
                   "step_ms_quantiles": quantiles([t * 1e3 for t in times]), "thread_probe_s": probe},
        "cpu_baseline": {"value": value, "unit": "utt/s", "cores": torch.get_num_threads(), "kind": "port",
                         "sample": ref.describe(K)},
        "e2e": {"value": value, "unit": "utt/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


# ----------------------------------------------------------------------------------------------------------------------
# GPU arm
# ----------------------------------------------------------------------------------------------------------------------
class GpuWorkload:
    """One BASELINE config on one GPU: device-resident step (`value`), host-buffer step through the public API (`e2e`)."""

    def __init__(self, conf, cfg, weights, vocab, dev, rank, world):
        import torch
        from ppasr_b200.infer_utils.inference_predictor import InferencePredictor
        from ppasr_b200.weights import synthetic_fbank
        self.torch, self.conf, self.cfg, self.vocab, self.dev, self.rank, self.world = torch, conf, cfg, vocab, dev, rank, world
        self.B = conf["batch"]
        self.frames = conf.get("frames") or frames_of(conf["seconds"])
        configs = {"encoder_conf": cfg.to_dict(), "preprocess_conf": {"n_mels": 80}}
        self.pred = InferencePredictor(configs, conf["model"], streaming=conf["streaming"], weights=weights, device=dev.index)
        self.eng = self.pred.engine
        self.pipelined = conf["decoder"] == "ctc_greedy" and conf["model"] != "deepspeech2"
        npool = 16 if self.B * self.frames * 320 * 16 < (8 << 30) else 2
        if conf["model"] == "conformer" and not conf["streaming"]:
            npool = 3  # 64 x 2998 x 80 fp32 = 61 MB per batch: three distinct batches exceed the 126 MB L2
        self.host = torch.from_numpy(synthetic_fbank(self.B, self.frames, seed=1234 + rank)).pin_memory()
        self.pool = [self.host.to(dev)] + [torch.from_numpy(synthetic_fbank(self.B, self.frames, seed=5000 + 97 * rank + i)).to(dev)
                                            for i in range(npool - 1)]
        self.pool_bytes = sum(t.numel() * 4 for t in self.pool)
        self.dec = None
        if conf["decoder"] == "ctc_beam_search":
            from ppasr_b200.decoders.beam_search_decoder import BeamSearchDecoder
            kw = {}
            if conf.get("lm"):
                from ppasr_b200.decoders.ngram_lm import Scorer
                kw = dict(alpha=2.2, beta=4.3, ext_scorer=Scorer(2.2, 4.3, None, vocab, lm=synthetic_lm(vocab)))
            self.dec = BeamSearchDecoder(beam_size=conf["beam"], cutoff_prob=0.99, cutoff_top_n=40, vocab_list=vocab, **kw)
        self.windows = stream_windows(self.frames) if conf.get("chunked") else None
        self.Tp = self.eng.encode(self.pool[0]).Tp if not self.windows else None
        if self.windows:
            self.eng.stream_reset(self.B)
            self.Tp = sum(int(self.eng.lib.ppasr_b200_out_frames(self.eng._ctx, b - a)) for a, b in self.windows)

    # -- one step, sync-style (no pipeline): results stay on the device ------------------------------------------------
    def step_device(self, feats):
        eng, conf = self.eng, self.conf
        if self.windows:
            eng.stream_reset(self.B)
            st = self.dec._alloc_state(self.B, self.Tp)
            for (a, b) in self.windows:
                eng.encode_chunk(feats[:, a:b].contiguous(), -16)
                self.dec._advance(st, eng.ctc_probs(), None, self.Tp)
            return self.dec._results_device(st, self.B, self.Tp, self.Tp, 1)
        eng.encode(feats)
        if conf["decoder"] == "ctc_greedy":
            return eng.ctc_greedy(to_host=False)
        return self.dec.decode_device(eng.ctc_probs(), None, 1)

    def texts_from(self, res):
        from ppasr_b200.parallel import detokenize
        ids, lens = res[0], res[1]
        if ids.dim() == 3:
            ids, lens = ids[:, 0], lens[:, 0]
        return detokenize(ids.cpu().numpy(), np.maximum(lens.cpu().numpy(), 0), self.vocab)

    def step_e2e(self):
        """Host fbank in (pinned), texts out: H2D of the step's features and D2H of its ids inside."""
        if self.windows:
            eng = self.eng
            eng.stream_reset(self.B)
            st = self.dec._alloc_state(self.B, self.Tp)
            hn = self.host.numpy()
            for (a, b) in self.windows:
                eng.encode_chunk(hn[:, a:b], -16)      # host window -> device inside the call
                self.dec._advance(st, eng.ctc_probs(), None, self.Tp)
            return self.texts_from(self.dec._results_device(st, self.B, self.Tp, self.Tp, 1))
        self.eng.encode(self.host)                      # pinned host features -> device inside the call
        if self.conf["decoder"] == "ctc_greedy":
            return self.texts_from(self.eng.ctc_greedy(to_host=False))
        return self.texts_from(self.dec.decode_device(self.eng.ctc_probs(), None, 1))

    def h2d_bytes(self):
        return self.B * self.frames * 80 * 4

    def d2h_bytes(self):
        return self.B * self.Tp * 4 + self.B * 4


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--config", default=None, choices=sorted(CONFIGS),
                    help="BASELINE config to run (default c2 = configs[1], the config the headline metric is quoted on)")
    ap.add_argument("--model", default=None, choices=["conformer", "squeezeformer"], help="deprecated alias: squeezeformer = --config c4")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the results of the last timed step (ids, lens, scores) to DIR/<name>.npy as float64")
    args = ap.parse_args()
    if args.impl == "reference" and args.dump_outputs:
        ap.error("--dump-outputs writes the GPU path's results; the reference arm has none")
    cname = args.config or ("c4" if args.model == "squeezeformer" else "c2")
    conf = CONFIGS[cname]
    if args.impl == "reference":
        return run_reference(args, conf)

    import torch
    import torch.distributed as dist
    from ppasr_b200 import _lib as L
    from ppasr_b200.parallel import all_gather_records, all_gather_results, detokenize, unpack_records
    from ppasr_b200.weights import make_vocab

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    numa_cpus = pin_to_gpu_numa(local_rank) if world > 1 else None
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        # NCCL prints its version banner to stdout at the VERSION and WARN levels: send its log to stderr so that stdout
        # carries the one JSON line only
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
        dist.init_process_group("nccl", device_id=dev)
    W = max(3, args.warmup)
    K = max(1, args.steps)

    cfg, weights = model_setup(conf)
    vocab = make_vocab(VOCAB)
    wl = GpuWorkload(conf, cfg, weights, vocab, dev, rank, world)
    pred, eng, lib = wl.pred, wl.eng, L.load()
    B, Tp = wl.B, wl.Tp
    total_utts = B * world
    lmax = Tp
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)  # > 126 MB L2

    def gather(res):
        ids, ol, sc = res
        if ids.dim() == 3:
            ids, ol, sc = ids[:, 0].contiguous(), ol[:, 0].contiguous(), sc[:, 0].contiguous()
        return all_gather_results(ids, ol, sc, total_utts, lmax) if world > 1 else (ids, ol, sc)

    # ---- (a) single-stream: one batch at a time, L2 flushed between steps ----
    def step():
        return gather(wl.step_device(wl.pool[0]))

    for _ in range(W):
        step()
    torch.cuda.synchronize()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(K)]
    for k in range(K):
        flush.zero_()  # L2 flush between timed iterations (not inside the timed events)
        ev[k][0].record()
        step()
        ev[k][1].record()
    torch.cuda.synchronize()
    single = [a.elapsed_time(b) for a, b in ev]
    single_ms = sum(single) / K

    # ---- (a') the same single-batch step captured once as a CUDA graph and replayed (one graph launch per step) ----
    graph_info = None
    if wl.pipelined and world == 1:
        try:
            gs = torch.cuda.Stream(device=dev)
            gi = torch.empty((B, Tp), dtype=torch.int32, device=dev)
            gl = torch.empty((B,), dtype=torch.int32, device=dev)
            gc = torch.empty((B,), dtype=torch.float32, device=dev)
            torch.cuda.synchronize()
            eng.encode(wl.pool[0], stream=gs)
            eng.ctc_greedy_into(gi, gl, gc, stream=gs)      # once outside the capture on this stream
            gs.synchronize()
            want = (gi.clone(), gl.clone())
            eng.graph_begin(gs)
            eng.encode(wl.pool[0], stream=gs)
            eng.ctc_greedy_into(gi, gl, gc, stream=gs)
            nk = eng.graph_end(gs)
            gi.zero_()
            torch.cuda.synchronize()
            for _ in range(W):
                eng.graph_launch(gs)
            gs.synchronize()
            same = bool(torch.equal(gi, want[0]) and torch.equal(gl, want[1]))
            gev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(K)]
            with torch.cuda.stream(gs):
                for k in range(K):
                    flush.zero_()
                    gev[k][0].record(gs)
                    eng.graph_launch(gs)
                    gev[k][1].record(gs)
            gs.synchronize()
            gms = [a.elapsed_time(b) for a, b in gev]
            graph_info = {"ms_per_step": sum(gms) / K, "quantiles": quantiles(gms), "kernels_per_replay": nk,
                          "replay_matches_direct_run": same}
        except Exception as e:  # a driver / runtime without capture support for some launch attribute: report, do not fail
            graph_info = {"error": str(e)[:300]}
        torch.cuda.synchronize()

    # ---- (b) `value`: whole-job throughput, inputs device resident and cycling over a pool of distinct batches larger than
    #      L2 (no explicit flush). Greedy configs run the public throughput pipeline (several batches in flight on private
    #      streams); beam / chunked / DS2 configs run one batch at a time on the current stream. ----
    depth = int(os.environ.get("PPASR_B200_DEPTH", "4")) if wl.pipelined else 1
    pipe = pred.pipeline(depth=depth) if wl.pipelined else None
    pool = wl.pool

    # per pipeline slot: a zeroed record buffer and the gathered array (the all-gather is the only collective of the job)
    max_local = (total_utts + world - 1) // world
    rec_bufs, gat_bufs = {}, {}

    def gather_slot(ticket):
        ids, ol, sc = pipe.device_result(ticket)
        st = pipe.stream(ticket)
        key = st.cuda_stream
        if key not in rec_bufs:
            rec_bufs[key] = torch.zeros((max_local, lmax + 2), dtype=torch.int32, device=dev)
            gat_bufs[key] = torch.empty((world * max_local, lmax + 2), dtype=torch.int32, device=dev)
        with torch.cuda.stream(st):
            return all_gather_records(ids, ol, sc, total_utts, lmax, rec=rec_bufs[key], out=gat_bufs[key])

    def finish(ticket):
        if world > 1:
            return gather_slot(ticket)
        return pipe.device_result(ticket)

    def run_steps(n):
        """Runs n steps and returns what the last one gives its caller: (ids, out_lens, scores) device tensors, or the
        gathered records of all ranks when the pipeline runs with N > 1."""
        last = None
        if pipe is None:
            for i in range(n):
                last = gather(wl.step_device(pool[i % len(pool)]))
            return last
        pending = []
        for i in range(n):
            pending.append(pipe.submit(pool[i % len(pool)], to_host=False))
            if len(pending) == depth:
                last = finish(pending.pop(0))
        while pending:
            last = finish(pending.pop(0))
        return last

    def timed_rep(n):
        e0 = torch.cuda.Event(enable_timing=True)
        e1 = torch.cuda.Event(enable_timing=True)
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        e0.record()
        if pipe is not None:
            for sl in pipe.slots:
                sl["stream"].wait_event(e0)
        last = run_steps(n)
        if pipe is not None:
            for sl in pipe.slots:
                torch.cuda.current_stream().wait_stream(sl["stream"])
        e1.record()
        torch.cuda.synchronize()
        t = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)  # max over ranks
        return float(t.item()), last

    run_steps(max(W, 4))
    torch.cuda.synchronize()
    sampler = ClockSampler(local_rank)
    sampler.start()
    launches0 = lib.ppasr_b200_launch_count()
    timed_ms, last = timed_rep(K)
    launches1 = lib.ppasr_b200_launch_count()
    sampler.stop_flag = True
    ms = timed_ms / K
    value = total_utts / (ms * 1e-3)
    if args.dump_outputs and rank == 0:
        if pipe is not None and world > 1:
            last = unpack_records(last.cpu().numpy(), total_utts, world, lmax)
        dump_outputs(args.dump_outputs, *last)
    if pipe is not None:
        pipe.close()

    # ---- e2e through the public API with host buffers (H2D of the features, D2H of ids/lens/scores) ----
    # Greedy configs: DecodePipeline = the throughput-mode public API (the pinned H2D copy of batch i+1 overlaps the kernels of
    # batch i). Every step copies its own inputs in and its own results out. With N > 1 every rank contributes its shard to the
    # single all-gather (the gathered ids stay on every GPU), copies back and detokenises ITS OWN shard; rank 0, the consumer
    # of the whole job, additionally copies the gathered records back and detokenises all N x B utterances.
    brk = {"submit_ms": 0.0, "wait_d2h_ms": 0.0, "allgather_enqueue_ms": 0.0, "detok_ms": 0.0}
    pipe = pred.pipeline(depth=depth) if wl.pipelined else None
    gathered_pin = torch.empty((world * max_local, lmax + 2), dtype=torch.int32).pin_memory() if world > 1 and rank == 0 else None

    own_pin = (torch.empty((B, lmax), dtype=torch.int32).pin_memory(), torch.empty((B,), dtype=torch.int32).pin_memory()) \
        if world > 1 and rank != 0 else None

    def e2e_finish(ticket):
        t0 = time.perf_counter()
        if world > 1:
            dids, dol, dsc = pipe.device_result(ticket)      # device tensors (submitted with to_host=False)
            g = gather_slot(ticket)
            with torch.cuda.stream(pipe.stream(ticket)):
                if gathered_pin is not None:
                    gathered_pin.copy_(g, non_blocking=True)   # rank 0 consumes the whole job: ONE copy of the gathered records
                else:
                    own_pin[0].copy_(dids[:, :lmax], non_blocking=True)
                    own_pin[1].copy_(dol, non_blocking=True)
            t1 = time.perf_counter()
            pipe.stream(ticket).synchronize()
            if gathered_pin is not None:
                ids, ol, _ = unpack_records(gathered_pin.numpy(), total_utts, world, lmax)
            else:
                ids, ol = own_pin[0].numpy(), own_pin[1].numpy()
        else:
            t1 = time.perf_counter()
            ids, ol, _ = pipe.result(ticket)             # synchronises the slot stream; results in pinned host buffers
        t2 = time.perf_counter()
        texts = detokenize(ids, ol, vocab)   # rank 0: all N x B utterances; the other ranks: their own shard
        t3 = time.perf_counter()
        brk["allgather_enqueue_ms"] += (t1 - t0) * 1e3
        brk["wait_d2h_ms"] += (t2 - t1) * 1e3
        brk["detok_ms"] += (t3 - t2) * 1e3
        return texts

    def e2e_run(n):
        texts = None
        if pipe is None:
            for _ in range(n):
                res_texts = wl.step_e2e()
                texts = res_texts
            return texts
        pending = []
        for _ in range(n):
            t0 = time.perf_counter()
            pending.append(pipe.submit(wl.host, to_host=(world == 1)))
            brk["submit_ms"] += (time.perf_counter() - t0) * 1e3
            if len(pending) == depth:
                texts = e2e_finish(pending.pop(0))
        while pending:
            texts = e2e_finish(pending.pop(0))
        return texts

    e2e_run(4)
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    for k in brk:
        brk[k] = 0.0
    t0 = time.perf_counter()
    texts = e2e_run(K)
    torch.cuda.synchronize()
    t = torch.tensor([(time.perf_counter() - t0) / K * 1e3], device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    e2e_ms = float(t.item())
    if pipe is not None:
        pipe.close()
    brk = {k: v / K for k, v in brk.items()}

    # ---- roofline of the dominant kernel, measured live with CUDA events ----
    pk = peaks()
    roof = None
    prof_table = None
    if rank == 0:
        if conf["decoder"] == "ctc_beam_search":
            # the decode's HBM-bound kernel: the pruning scan of the posterior [B, T', V] fp32 (reads every byte once)
            if wl.windows:
                eng.stream_reset(B)
                eng.encode_chunk(wl.pool[0][:, wl.windows[0][0]:wl.windows[0][1]].contiguous(), -16)
            else:
                eng.encode(wl.pool[0])
            probs = eng.ctc_probs()
            rows = probs.shape[0] * probs.shape[1]
            ws = torch.empty(lib.ppasr_b200_beam_workspace_bytes(probs.shape[0], probs.shape[1]), dtype=torch.uint8, device=dev)
            prune = lambda: L.check(lib.ppasr_b200_op_ctc_prune(L.ptr(probs), rows, VOCAB, 0.99, 40, L.ptr(ws), L.stream_ptr()))
            prune()
            torch.cuda.synchronize()
            tot, n = 0.0, 10
            for _ in range(n):
                flush.zero_()
                e0 = torch.cuda.Event(enable_timing=True)
                e1 = torch.cuda.Event(enable_timing=True)
                e0.record()
                prune()
                e1.record()
                torch.cuda.synchronize()
                tot += e0.elapsed_time(e1)
            us = tot / n * 1e3
            nbytes = rows * VOCAB * 4.0
            ach = nbytes / (us * 1e-6) / 1e9
            roof = {"kernel": "ctc_prune", "bound": "hbm", "achieved": ach, "peak": pk["hbm_gbs"], "unit": "GB/s",
                    "frac": ach / pk["hbm_gbs"], "traffic": ncu_traffic("ctc_prune", rows),  # one CTA per posterior row "peak_source": pk["src"] + " (copy bandwidth)",
                    "us_per_launch": us, "algorithmic_bytes_per_launch": nbytes,
                    "rows_per_launch": rows, "note": "posterior [B,T',V] fp32 read once; L2 flushed before every timed launch"}
        elif conf["model"] != "deepspeech2":
            # like the `value` measurement: inputs cycle over the pool of distinct device-resident batches (larger than L2), no
            # explicit flush -- a 256 MiB flush would also evict the 70 MB of weights a serving process keeps L2 resident
            eng.profile_enable(True)
            for i in range(K):
                eng.encode(wl.pool[i % len(wl.pool)])
                eng.ctc_greedy(to_host=False)
            prof = eng.profile_read()
            eng.profile_enable(False)
            M = B * Tp
            D, FF = cfg.output_size, cfg.linear_units
            ffn_m = 0.75 if conf["model"] == "squeezeformer" else 1.0  # half of the squeezeformer blocks run at T'/2
            flops = {  # algorithmic FLOPs per launch (2*M*N*K)
                "ffn1_gemm": 2.0 * M * FF * D, "ffn2_gemm": 2.0 * M * D * FF, "qkv_gemm": 2.0 * M * 3 * D * D,
                "outproj_gemm": 2.0 * M * D * D, "pw1_glu_gemm": 2.0 * M * 2 * D * D, "pw2_gemm": 2.0 * M * D * D,
                "conv2_gemm": 2.0 * (B * Tp * 19) * D * 9 * D, "embed_gemm": 2.0 * M * D * 19 * D,
                "ctc_stats_gemm": 2.0 * M * VOCAB * D, "attention": 2.0 * B * 4 * Tp * Tp * (128 + 64),
                # fused_ffn: W1 + W2 GEMMs (+ the chained pointwise_conv2 in every second launch: averaged)
                "fused_ffn": (2.0 * M * D * FF * 2) * ffn_m + (0.5 * 2.0 * M * D * D if conf["model"] == "conformer" else 0.0),
                "fused_attn_out": 2.0 * M * D * D + 2.0 * M * 2 * D * D,
                "conv_front": 2.0 * (B * Tp * 19) * D * 9 * D,
            }
            total = sum(v[1] for v in prof.values())
            prof_table = {k: {"launches_per_step": v[0] // K, "us_per_launch": v[1] / v[0] * 1e3,
                              "share": v[1] / total} for k, v in sorted(prof.items(), key=lambda kv: -kv[1][1])}
            top = max((k for k in prof if k in flops), key=lambda k: prof[k][1])
            us_all = prof[top][1] / prof[top][0] * 1e3
            # second pass: event pairs around the dominant class ONLY, so the other ~70 launches of the step stay back to back
            # and the CPU-side event records do not open gaps in front of the timed kernel
            eng.profile_enable(True, only=top)
            for i in range(K):
                eng.encode(wl.pool[i % len(wl.pool)])
                eng.ctc_greedy(to_host=False)
            prof1 = eng.profile_read()
            eng.profile_enable(False)
            us = prof1[top][1] / prof1[top][0] * 1e3
            ach = flops[top] / (us * 1e-6) / 1e12
            roof = {"kernel": top, "bound": "tensor", "achieved": ach, "peak": pk["bf16_tflops"], "unit": "TFLOP/s",
                    "frac": ach / pk["bf16_tflops"], "traffic": ncu_traffic(top), "peak_source": pk["src"] + " (burst cuBLAS bf16)",
                    "us_per_launch": us, "us_per_launch_all_classes_timed": us_all, "share_of_step": prof[top][1] / total,
                    "algorithmic_flops_per_launch": flops[top],
                    "step_tensor_frac_sustained": (conf["gflop_per_utt"] * B / ms) / pk["bf16_tflops_sustained"],
                    "note": f"us_per_launch: CUDA-event pairs around the launches of this kernel class only, {K} single-batch steps "
                            "over distinct input batches (pool larger than L2, no flush; average over the plain and the "
                            "chained launches); shares: a first pass with pairs around every launch"}
            try:
                sms = torch.cuda.get_device_properties(dev).multi_processor_count
                ctas = (B * Tp + 127) // 128 * (2 if lib.ppasr_b200_get_ffn_split() == 1 else 1)
                if top == "fused_ffn":
                    roof.update({"ctas_per_launch": ctas, "sms": sms})
            except Exception:
                pass

    # ---- CPU baseline: the same CPU reference arm, bounded to ~10-20 s (rank 0, N = 1) ----
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        ref = CpuReference(conf, cfg, weights, vocab)
        f = wl.host[:ref.sample_b].numpy()
        lens = [wl.frames] * ref.sample_b
        threads, probe = ref.choose_threads(f, lens)
        ref.step(f, lens)
        t0 = time.perf_counter()
        n = 0
        while n < 2 or time.perf_counter() - t0 < 10.0:
            ref.step(f, lens)
            n += 1
            if n >= 50:
                break
        dt = (time.perf_counter() - t0) / n
        cpu = {"value": ref.sample_b / dt, "unit": "utt/s", "cores": torch.get_num_threads(), "kind": "port",
               "sample": ref.describe(n), "rtf": dt / (ref.sample_b * conf["seconds"]), "thread_probe_s": probe}

    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": "utt/s", "n_gpus": world, "steps": K, "warmup": W,
            "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "bf16" if conf["model"] != "deepspeech2" else "bf16 (recurrent weights) / f32 (state)",
            "data": "synthetic",
            "config": {"workload": conf["name"] + "; per GPU", "config": cname,
                       "global_batch": total_utts, "frames": wl.frames, "out_frames": Tp, "vocab": VOCAB,
                       "parallelism": f"dp{world} (batch sharded, one all-gather of ids)" if world > 1 else "single GPU",
                       "mode": (f"throughput: {depth} batches in flight ({depth} engines on {depth} CUDA streams per GPU)"
                                if wl.pipelined else "one batch at a time on one stream"),
                       "l2": f"inputs larger than L2: {len(pool)} distinct device-resident batches ({wl.pool_bytes / 1e6:.0f} MB) "
                             "cycled; no explicit flush",
                       "timed_region": {"steps": K, "total_s": timed_ms / 1e3},
                       "single_stream_ms_per_step": single_ms,
                       "single_stream_quantiles": quantiles(single),
                       "single_stream_note": "one batch at a time, 256 MiB memset L2 flush between steps (outside the events)",
                       "single_stream_cuda_graph": graph_info,
                       "rtf": ms * 1e-3 / (B * conf["seconds"]), "gflop_per_step_per_gpu": conf["gflop_per_utt"] * B,
                       "ffn_variant": {"single_stream": int(lib.ppasr_b200_get_ffn_split()),
                                       "pipeline": int(os.environ.get("PPASR_B200_FFN_PIPE", "2"))},
                       "numa_pinned_cpus": numa_cpus},
            "clocks": sampler.result(),
            "e2e": {"value": total_utts / (e2e_ms * 1e-3), "unit": "utt/s", "ms_per_step": e2e_ms,
                    "h2d_bytes_per_step": wl.h2d_bytes(), "d2h_bytes_per_step": wl.d2h_bytes(),
                    "host_ms_per_step_rank0": brk,
                    "api": (f"InferencePredictor.pipeline(depth={depth}).submit(host fbank)/result() + host detokenisation"
                            if wl.pipelined else "engine.encode/encode_chunk(host fbank) + decoder + D2H of the best ids + host detokenisation")},
            "gpu_launches": int(launches1 - launches0),
            "roofline": roof, "cpu_baseline": cpu, "kernel_profile": prof_table,
            "sample_text_len": len(texts[0]) if texts else 0,
        }
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
