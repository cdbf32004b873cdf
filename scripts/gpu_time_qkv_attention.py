"""Time the fused QKV projection + rel-pos attention (qkv_rel_attention_kernel) against the QKV GEMM + rel_attention_kernel
pair it replaces, through ppasr_b200_op_qkv_attention on the same inputs. The two are timed alternately, each with CUDA events
over many back-to-back launches after a warm-up; one JSON line per case with the median of the rounds.

    python scripts/gpu_time_qkv_attention.py [--iters 200] [--rounds 5] [--out timings/qkv_attention.jsonl]

The op's pair path also allocates its scratch q2 / kk / vt (stream-ordered) and clears the V^T padding, so `pair_us` is an
upper bound on the two kernels. A separate torch.profiler pass (after the event timing) gives the device time of each kernel
alone: `kernel_us` maps kernel name -> mean time per launch. The card's name, power limit and max SM clock are printed in the
same run.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from ppasr_b200 import _lib as L  # noqa: E402

D, H, POS_LD = 256, 4, 256


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return {"device": torch.cuda.get_device_name(0), "nvidia_smi": q[0] if q else "unavailable"}


def time_ms(fn, iters):
    for _ in range(5):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters


def case(lib, dev, name, B, T, ragged, iters, rounds):
    g = torch.Generator().manual_seed(B * 1000 + T)
    y = torch.randn(B * T, D, generator=g).to(torch.bfloat16).to(dev)
    wqkv = (torch.randn(3 * D, D, generator=g) / 16).to(torch.bfloat16).to(dev)
    bqkv = (torch.randn(3 * D, generator=g) * 0.1).to(dev)
    pu = (torch.randn(D, generator=g) * 0.3).to(dev)
    pv = (torch.randn(D, generator=g) * 0.3).to(dev)
    pos = torch.randn(T, POS_LD, generator=g).to(torch.bfloat16).to(dev)
    klens = (torch.randint(T // 4, T + 1, (B,), generator=g, dtype=torch.int32) if ragged
             else torch.full((B,), T, dtype=torch.int32)).to(dev)
    outs = [torch.empty(B * T, D, device=dev, dtype=torch.bfloat16) for _ in range(2)]

    def run(fused):
        L.check(lib.ppasr_b200_op_qkv_attention(L.ptr(y), L.ptr(wqkv), L.ptr(bqkv), L.ptr(pu), L.ptr(pv), L.ptr(pos), T,
                                                POS_LD, 0, 0, L.ptr(klens), B, T, L.ptr(outs[fused]), fused, L.stream_ptr()))

    fused_ms, pair_ms = [], []
    for _ in range(rounds):
        fused_ms.append(time_ms(lambda: run(1), iters))
        pair_ms.append(time_ms(lambda: run(0), iters))
    torch.cuda.synchronize()
    kernel_us = {}
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        for _ in range(20):
            run(1)
            run(0)
        torch.cuda.synchronize()
    for ev in prof.key_averages():
        if any(k in ev.key for k in ("qkv_rel_attention", "rel_attention_kernel", "EpiQKV")):
            kname = ("qkv_rel_attention_kernel" if "qkv_rel_attention" in ev.key
                    else "rel_attention_kernel" if "rel_attention_kernel" in ev.key else "qkv_gemm (EpiQKV)")
            dt = getattr(ev, "device_time_total", None) or getattr(ev, "cuda_time_total", 0.0)
            kernel_us[kname] = round(dt / max(ev.count, 1), 2)
    f, p = statistics.median(fused_ms), statistics.median(pair_ms)
    return {"case": name, "B": B, "T": T, "ragged": ragged, "fused_us": round(f * 1e3, 2), "pair_us": round(p * 1e3, 2),
            "fused_us_rounds": [round(x * 1e3, 2) for x in fused_ms], "pair_us_rounds": [round(x * 1e3, 2) for x in pair_ms],
            "speedup": round(p / f, 3), "kernel_us": kernel_us,
            "bit_identical": bool(torch.equal(outs[0].view(torch.int16), outs[1].view(torch.int16)))}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=200)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("needs a CUDA device")
    dev = torch.device("cuda:0")
    lib = L.load()
    rows = [dict(case="card", **card())]
    rows.append(case(lib, dev, "c2", 32, 248, False, a.iters, a.rounds))
    rows.append(case(lib, dev, "half_rate", 32, 124, False, a.iters, a.rounds))
    rows.append(case(lib, dev, "c2_ragged", 32, 248, True, a.iters, a.rounds))
    rows.append(dict(case="card_after", **card()))
    lines = [json.dumps(r) for r in rows]
    print("\n".join(lines), flush=True)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
