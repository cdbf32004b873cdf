"""QKV projection + rel-pos attention of an offline block (ppasr_b200_op_qkv_attention): the fused kernel
(qkv_rel_attention_kernel, T' <= 256) gives the same bits as the QKV GEMM + rel_attention_kernel pair on the same inputs,
and both match an fp32 restatement of the reference attention (conformer/attention.py:76-84,198-262) within the op-level
2e-2 of max|.|."""
import pytest
import torch

D, H = 256, 4
POS_ROW0, POS_COL0, POS_LD = 5, 256, 512  # key 0 at row 5 of a two-layer positional table, second layer's columns


def restate(y, wqkv, bqkv, pos_u, pos_v, pos, klens, B, T):
    """fp32 restatement on any device: q / k / v = y W^T + b, S = ((q + u) k^T + (q + v) p^T) / sqrt(64), keys >= klen
    masked, softmax, A V."""
    qkv = y.float() @ wqkv.float().t() + bqkv
    q, k, v = qkv.view(B, T, 3, H, 64).permute(2, 0, 3, 1, 4).unbind(0)  # [B, H, T, 64] each
    p = pos[POS_ROW0:POS_ROW0 + T, POS_COL0:POS_COL0 + D].float().view(T, H, 64).transpose(0, 1)
    s = ((q + pos_u.view(H, 1, 64)) @ k.transpose(-1, -2) + (q + pos_v.view(H, 1, 64)) @ p.transpose(-1, -2)) / 8.0
    mask = torch.arange(T, device=y.device)[None, :] >= klens[:, None].to(y.device)
    s = s.masked_fill(mask[:, None, None, :], float("-inf"))
    a = torch.softmax(s, -1).masked_fill(mask[:, None, None, :], 0.0)
    return (a @ v).transpose(1, 2).reshape(B * T, D)


def make_inputs(B, T, device, seed):
    g = torch.Generator().manual_seed(seed)
    y = torch.randn(B * T, D, generator=g).to(torch.bfloat16)
    wqkv = (torch.randn(3 * D, D, generator=g) / 16).to(torch.bfloat16)
    bqkv = torch.randn(3 * D, generator=g) * 0.1
    pos_u = torch.randn(D, generator=g) * 0.3
    pos_v = torch.randn(D, generator=g) * 0.3
    pos = torch.randn(POS_ROW0 + 300, POS_LD, generator=g).to(torch.bfloat16)
    # ragged: one full-length utterance, the others end inside key block 0 or (T > 128) key block 1
    klens = torch.randint(1, T + 1, (B,), generator=g, dtype=torch.int32)
    klens[0] = T
    if B > 1:
        klens[1] = max(1, min(T, 77))
    if B > 2 and T > 128:
        klens[2] = 129 + (T - 129) // 2
    return [t.to(device) for t in (y, wqkv, bqkv, pos_u, pos_v, pos, klens)]


def run_op(lib, inputs, B, T, fused):
    from ppasr_b200 import _lib as L
    y, wqkv, bqkv, pos_u, pos_v, pos, klens = inputs
    out = torch.full((B * T, D), float("nan"), device=y.device, dtype=torch.bfloat16)
    L.check(lib.ppasr_b200_op_qkv_attention(L.ptr(y), L.ptr(wqkv), L.ptr(bqkv), L.ptr(pos_u), L.ptr(pos_v), L.ptr(pos),
                                            pos.shape[0], POS_LD, POS_ROW0, POS_COL0, L.ptr(klens), B, T, L.ptr(out), fused,
                                            L.stream_ptr()))
    torch.cuda.synchronize()
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("B", [1, 3, 32])
@pytest.mark.parametrize("T", [1, 16, 100, 128, 129, 200, 248, 256])
def test_fused_qkv_attention_bit_identical_to_gemm_pair(lib, cuda, B, T):
    inputs = make_inputs(B, T, cuda, seed=1000 * B + T)
    fused = run_op(lib, inputs, B, T, 1)
    pair = run_op(lib, inputs, B, T, 0)
    assert torch.equal(fused.view(torch.int16), pair.view(torch.int16))


@pytest.mark.gpu
@pytest.mark.parametrize("B,T", [(3, 248), (2, 129), (1, 16), (32, 256)])
def test_fused_qkv_attention_matches_fp32_restatement(lib, cuda, B, T):
    inputs = make_inputs(B, T, cuda, seed=7 * T + B)
    got = run_op(lib, inputs, B, T, 1)
    ref = restate(*inputs[:6], inputs[6], B, T)
    assert torch.isfinite(got.float()).all()
    err = (got.float() - ref).abs().max().item() / ref.abs().max().item()
    assert err < 2e-2, err


@pytest.mark.gpu
def test_fused_qkv_attention_refuses_more_than_256_frames(lib, cuda):
    from ppasr_b200 import _lib as L
    inputs = make_inputs(2, 257, cuda, seed=257)
    with pytest.raises(L.PPASRB200Error):
        run_op(lib, inputs, 2, 257, 1)
    pair = run_op(lib, inputs, 2, 257, 0)  # the pair has no such limit
    assert torch.isfinite(pair.float()).all()


def test_restatement_matches_per_row_softmax_cpu():
    """The restatement above, checked on CPU tensors against an explicit per-(utterance, head, query) loop."""
    B, T = 2, 9
    y, wqkv, bqkv, pos_u, pos_v, pos, klens = make_inputs(B, T, "cpu", seed=3)
    klens[1] = 4
    got = restate(y, wqkv, bqkv, pos_u, pos_v, pos, klens, B, T).view(B, T, H, 64)
    qkv = (y.double() @ wqkv.double().t() + bqkv.double()).view(B, T, 3 * D)
    pt = pos.double()[POS_ROW0:POS_ROW0 + T, POS_COL0:POS_COL0 + D]
    for b in range(B):
        n = int(klens[b])
        for h in range(H):
            sl = slice(h * 64, h * 64 + 64)
            q, k, v = qkv[b, :, sl], qkv[b, :n, D + h * 64:D + h * 64 + 64], qkv[b, :n, 2 * D + h * 64:2 * D + h * 64 + 64]
            for t in range(T):
                s = ((q[t] + pos_u.double()[sl]) @ k.t() + (q[t] + pos_v.double()[sl]) @ pt[:n, sl].t()) / 8.0
                ref = torch.softmax(s, 0) @ v
                assert torch.allclose(got[b, t, h].double(), ref, atol=1e-4, rtol=1e-4)
