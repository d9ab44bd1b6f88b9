"""The oracle's explicit dropout masks (oracle/restatement.py): the device-side restatement of the projection mask, the
keep factors block_forward / pair_forward take in place of torch's dropout, and where in the block they act.  These are
what the bench-step test (tests/test_gpu_bench_step.py) feeds the float64 oracle with the seed words the kernels drew."""
import pytest
import torch
import torch.nn.functional as F

from oracle import model_init
from oracle import restatement as R

WS = (4, 4, 2)


def _hash_keep(words, i, p_drop):
    """Keep factor of element i of csrc/dropout.cu, one element at a time in plain Python integers."""
    M = 0xFFFFFFFF

    def mix(x):
        x ^= x >> 16
        x = (x * 0x21F0AAAD) & M
        x ^= x >> 15
        x = (x * 0x735A2D97) & M
        return x ^ (x >> 15)

    s0, s1 = words[0] & M, words[1] & M
    q = i >> 2
    h = mix((s0 + (q & M) * 0x9E3779B1 + (q >> 32) * 0x85EBCA77) & M) ^ s1
    t = R._drop_threshold(p_drop)
    return 256.0 / (256 - t) if ((mix(h) >> (8 * (i & 3))) & 0xFF) >= t else 0.0


@pytest.mark.parametrize("p_drop", [0.1, 0.3, 1e-3])
@pytest.mark.parametrize("n0,n", [(0, 1), (0, 4099), (3, 17), (1021, 2050), (4096 + 2, 1)])
def test_projection_mask_torch_equals_numpy(n0, n, p_drop):
    words = [20261018, 1234567891]
    ref = R.elementwise_dropout_keep_factor(words, n0 + n, p_drop)[n0:]
    got = R.elementwise_dropout_keep_factor_torch(words, n0, n, p_drop)
    assert got.dtype == torch.float64 and got.shape == (n,)
    assert torch.equal(got, ref)


def test_projection_mask_beyond_32_bit_quad_index():
    """Element indices whose quad index needs more than 32 bits (the high word enters the hash on its own)."""
    words = [7, 2 ** 31 - 2]
    for n0 in (0, 2 ** 34 - 5, 3 * 2 ** 33 + 1):
        got = R.elementwise_dropout_keep_factor_torch(words, n0, 9, 0.1)
        assert got.tolist() == [_hash_keep(words, n0 + k, 0.1) for k in range(9)], n0


def test_projection_mask_rate():
    got = R.elementwise_dropout_keep_factor_torch([5, 6], 0, 1 << 20, 0.1)
    t = R._drop_threshold(0.1)
    assert set(got.unique().tolist()) == {0.0, 256.0 / (256 - t)}
    assert abs((got == 0).double().mean().item() - t / 256) < 3e-3


def _pair_case(seed=3, B=2, C=12, heads=2, dims=(8, 8, 6), I=8):
    torch.manual_seed(seed)
    sd = {k: v.double() for k, v in model_init.pair_state_dict(C, heads, 16, I, WS, down=True, merge_last_dim=True).items()
          if v.is_floating_point()}
    for k, v in sd.items():                     # biases and norm parameters away from their 0 / 1 initial values
        if k.endswith("bias") or k.endswith("norm.weight"):
            v.add_(0.1 * torch.randn_like(v))
    x = torch.randn(B, C, *dims, dtype=torch.float64)
    ps = [0.5 * torch.randn(B, I, C, dtype=torch.float64) for _ in range(2)]
    return sd, x, ps, heads, I


def _sub(sd, i):
    pre = f"swin_blocks.{i}."
    return {k[len(pre):]: v for k, v in sd.items() if k.startswith(pre)}


def test_block_keep_factors_layout():
    """Attention mask = dropout_keep_factor over (sample * window, head, query, key); projection mask = the elementwise
    mask over the block's [B,P,N,C] token tensor in row-major order."""
    sd, x, ps, heads, I = _pair_case(dims=(8, 6, 6))          # padded on every axis (R.pad_amounts): 12x8x8, P = 3*2*4
    words = [11, 22, 33, 44]
    B, C = x.shape[:2]
    P, N = 24, 32
    ak, pk = R.block_keep_factors(words, x.shape, WS, heads, I, 0.1, 0.3)
    assert torch.equal(ak, R.dropout_keep_factor(words[:2], B, P, heads, N, N + I, 0.1))
    assert torch.equal(pk, R.elementwise_dropout_keep_factor(words[2:], B * P * N * C, 0.3).reshape(B, P, N, C))
    assert R.block_keep_factors(words, x.shape, WS, heads, I, 0.0, 0.3)[0] is None
    assert R.block_keep_factors(words, x.shape, WS, heads, I, 0.1, 0.0)[1] is None


def test_all_ones_keep_factors_reproduce_no_dropout():
    sd, x, ps, heads, I = _pair_case()
    B, C = x.shape[:2]
    ones = (torch.ones(B, 12, heads, 32, 32 + I, dtype=torch.float64), torch.ones(B, 12, 32, C, dtype=torch.float64))   # P = 2*2*3
    for shift in ((0, 0, 0), (2, 2, 1)):
        ref = R.block_forward(_sub(sd, 0), x, ps[0], WS, shift, heads)
        # explicit factors take the place of the dropout whatever the rate says
        got = R.block_forward(_sub(sd, 0), x, ps[0], WS, shift, heads, 0.5, 0.5, attn_keep=ones[0], proj_keep=ones[1])
        assert torch.equal(got, ref)
    ref = R.pair_forward(sd, x, ps, WS, heads, True, True)
    got = R.pair_forward(sd, x, ps, WS, heads, True, True, 0.5, 0.5, keep=(ones, ones))
    assert torch.equal(got, ref)


def _block_by_hand(sd, x, p, ws, shift_cfg, heads, ak, pk):
    """Block forward with the two dropout sites written out: probabilities * ak, (o Wproj^T + bproj) * pk, then + shortcut."""
    dims, C = tuple(x.shape[2:]), x.shape[1]
    pads = R.pad_amounts(dims, ws)
    shift = R.effective_shift(dims, ws, shift_cfg)
    ids = R.region_ids(dims, ws, shift, pads) if any(shift) else None
    th, tw, td, tok = R.bias_tables(R.split_block_params(sd), ws, sd["pe.enc_content_h"].shape[1], p.shape[1])
    bias = R.dense_bias(th, tw, td, tok)
    xw = R.partition_tokens(x, ws, shift, pads)
    ln = F.layer_norm(xw, (C,), sd["attn_norm.weight"], sd["attn_norm.bias"], 1e-6)
    lp = F.layer_norm(p, (C,), sd["attn_norm.weight"], sd["attn_norm.bias"], 1e-6)
    dh = C // heads
    hd = lambda t: t.reshape(*t.shape[:-1], heads, dh).transpose(-2, -3)          # [..., h, n, dh]
    q, k, v = (hd(ln @ sd[f"attn.to_{n}.weight"].t()) for n in "qkv")
    kp, vp = (hd(lp @ sd[f"attn.to_{n}.weight"].t())[:, None] for n in "kv")          # [B,1,h,I,dh]
    Pw = q.shape[1]
    k = torch.cat([k, kp.expand(-1, Pw, -1, -1, -1)], dim=3)
    v = torch.cat([v, vp.expand(-1, Pw, -1, -1, -1)], dim=3)
    s = q @ k.transpose(-1, -2) * dh ** -0.5 + bias
    if ids is not None:
        t = torch.from_numpy(ids)
        m = (t[:, :, None] == t[:, None, :]).double()
        m = torch.cat([m, m.new_ones(Pw, m.shape[1], p.shape[1])], dim=2)
        s = s * m[None, :, None]
    o = (torch.softmax(s, dim=-1) * ak) @ v
    o = o.transpose(-2, -3).reshape(xw.shape)
    y = (o @ sd["attn.proj.weight"].t() + sd["attn.proj.bias"]) * pk + xw
    y = y + F.layer_norm(y, (C,), sd["mlp_norm.weight"], sd["mlp_norm.bias"], 1e-6) @ sd["mlp.weight"].t() + sd["mlp.bias"]
    return R.reverse_tokens(y, dims, ws, shift, pads)


@pytest.mark.parametrize("dims,shift", [((8, 8, 6), (2, 2, 1)), ((8, 6, 6), (0, 0, 0)), ((8, 6, 6), (2, 2, 1))])
def test_explicit_masks_match_hand_restatement(dims, shift):
    sd, x, ps, heads, I = _pair_case(dims=dims)
    words = [101, 202, 303, 404]
    ak, pk = R.block_keep_factors(words, x.shape, WS, heads, I, 0.3, 0.3)
    got = R.block_forward(_sub(sd, 1), x, ps[1], WS, shift, heads, attn_keep=ak, proj_keep=pk)
    ref = _block_by_hand(_sub(sd, 1), x, ps[1], WS, shift, heads, ak, pk)
    assert (got - ref).abs().max().item() < 1e-12
    plain = R.block_forward(_sub(sd, 1), x, ps[1], WS, shift, heads)
    assert (got - plain).abs().max().item() > 0.1                 # the masks do act
    # each site on its own
    one = torch.ones_like
    for a, b in ((ak, one(pk)), (one(ak), pk)):
        got = R.block_forward(_sub(sd, 1), x, ps[1], WS, shift, heads, attn_keep=a, proj_keep=b)
        assert (got - _block_by_hand(_sub(sd, 1), x, ps[1], WS, shift, heads, a, b)).abs().max().item() < 1e-12


def test_pair_forward_keep_per_block():
    """pair_forward hands block i the i-th (attn_keep, proj_keep) pair: same result as chaining block_forward by hand."""
    sd, x, ps, heads, I = _pair_case()
    keeps = [R.block_keep_factors([i, 2 * i + 1, 3 * i + 2, 4 * i + 3], x.shape, WS, heads, I, 0.2, 0.2) for i in (1, 2)]
    y = x
    for i, sh in enumerate(((0, 0, 0), (2, 2, 1))):
        y = R.block_forward(_sub(sd, i), y, ps[i], WS, sh, heads, attn_keep=keeps[i][0], proj_keep=keeps[i][1])
    y = R.patch_merging_forward({k[6:]: v for k, v in sd.items() if k.startswith("merge.")}, y, True)
    got = R.pair_forward(sd, x, ps, WS, heads, True, True, keep=keeps)
    assert torch.equal(got, y)
    swapped = R.pair_forward(sd, x, ps, WS, heads, True, True, keep=keeps[::-1])
    assert (swapped - y).abs().max().item() > 1e-3
