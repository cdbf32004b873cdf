"""Time grouped_attention_kernel (ppasr_b200_op_grouped_attention) from 64 to 1667 key groups, and one offline step of the
12-block Efficient Conformer at B = 8 x 60 s. CUDA events over many launches after a warm-up; one JSON line per case.

    python scripts/gpu_time_grouped_attention.py [--iters 50] [--out timings/grouped_attention.jsonl]

FLOPs are algorithmic, from shapes: 2 * B * H * Tg * Tgk * (384 + 192) for QK^T over [q+u | q+v] . [k | p] and P.V. Above 256
key groups (4 blocks of 64) the kernel scores every block twice (recompute path); `issued_tflops` counts that extra QK^T.
The card's name, power limit and max SM clock are read in the same run and printed with the numbers.
"""
import argparse
import json
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from ppasr_b200 import _lib as L  # noqa: E402


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


def op_case(lib, dev, layout, B, Tgk, iters):
    H = 4
    if layout == "offline":            # queries == keys (build_plan layout)
        T = 3 * Tgk
        Tg = Tgk
        k_pitch, vt_pitch = Tg, (Tg + 63) // 64 * 64
    else:                              # a 16-frame chunk against the cache (encode_chunk layout, max_len 5000)
        T, Tg = 16, 6
        k_pitch = vt_pitch = 1672
    q2g = (torch.randn(B, H, Tg, 384, device=dev) * 0.5).to(torch.bfloat16)
    kk = (torch.randn(B, H, k_pitch, 192, device=dev) * 0.5).to(torch.bfloat16)
    vt = torch.randn(B, H, 192, vt_pitch, device=dev).to(torch.bfloat16)
    pos = (torch.randn(Tgk, 768, device=dev) * 0.5).to(torch.bfloat16)
    out = torch.empty(B * T, 256, device=dev, dtype=torch.bfloat16)

    def run():
        L.check(lib.ppasr_b200_op_grouped_attention(L.ptr(q2g), L.ptr(kk), k_pitch, L.ptr(vt), vt_pitch, L.ptr(pos), L.ptr(out),
                                                    B, H, T, Tgk, None, L.stream_ptr()))

    ms = time_ms(run, iters)
    flops = 2.0 * B * H * Tg * Tgk * (384 + 192)
    nblk = (Tgk + 63) // 64
    issued = flops + (2.0 * B * H * Tg * Tgk * 384 if nblk > 4 else 0.0)
    return {"case": "op", "layout": layout, "B": B, "H": H, "query_groups": Tg, "key_groups": Tgk,
            "path": "resident" if nblk <= 4 else "recompute", "us": round(ms * 1e3, 2), "gflop": round(flops / 1e9, 3),
            "tflops": round(flops / ms / 1e9, 1), "issued_tflops": round(issued / ms / 1e9, 1)}


def model_case(dev, iters):
    from ppasr_b200.engine import ConformerEngine
    from ppasr_b200.weights import EfficientConformerConfig, init_efficient_conformer_weights, synthetic_fbank
    cfg = EfficientConformerConfig(num_blocks=12, vocab_size=4233, group_layer_idx=(0, 1, 2, 3), stride_layer_idx=3)
    eng = ConformerEngine(cfg, init_efficient_conformer_weights(cfg))
    B, T = 8, 6000                     # 8 x 60 s: T' = 1499 encoder frames, 500 key groups in the grouped blocks
    feats = torch.from_numpy(synthetic_fbank(B, T)).to(dev)
    lens = [T] * B
    ms = time_ms(lambda: eng.encode(feats, lens), iters)
    eng.close()
    return {"case": "model", "model": "efficient_conformer 12 blocks (grouped 0-3, stride 3)", "B": B, "feature_frames": T,
            "encoder_frames": ((T - 1) // 2 - 1) // 2, "ms_per_encode": round(ms, 3),
            "audio_s_per_s": round(B * T / 100.0 / (ms / 1e3), 1)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=50)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("needs a CUDA device")
    dev = torch.device("cuda:0")
    torch.manual_seed(0)
    lib = L.load()
    rows = [dict(case="card", **card())]
    for Tgk in (64, 128, 256, 257, 320, 512, 1024, 1667):
        rows.append(op_case(lib, dev, "offline", 8, Tgk, a.iters))
    for Tgk in (64, 256, 257, 512, 1024, 1667):
        rows.append(op_case(lib, dev, "streaming", 64, Tgk, a.iters))
    rows.append(model_case(dev, max(3, a.iters // 10)))
    rows.append(dict(case="card_after", **card()))
    lines = [json.dumps(r) for r in rows]
    print("\n".join(lines), flush=True)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
