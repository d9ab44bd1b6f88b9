"""CPU-only checks of the product's host side: the C-ABI library loads and exports every symbol that
include/pwa.h declares, the C host logic (geometry / region ids / index maps) is bit-exact against the
golden vectors from the live reference, and the nn.Module mirror keeps the reference's state-dict keys.
No compute call that needs a GPU is made here."""
import ctypes
import os
import re

import numpy as np
import pytest
import torch

import pwa_b200
from oracle import restatement as R
from tests.util import golden_names, load_npz, load_block_case

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_exports_every_declared_symbol():
    hdr = open(os.path.join(ROOT, "include", "pwa.h")).read()
    declared = set(re.findall(r"\b(pwa_[a-z_0-9]+)\s*\(", hdr))
    assert declared, "no declarations parsed"
    lib = ctypes.CDLL(pwa_b200._lib.LIB_PATH)
    for name in sorted(declared):
        assert hasattr(lib, name), f"{name} declared in include/pwa.h but not exported"
    assert set(pwa_b200._lib.EXPORTED_SYMBOLS) == declared
    assert lib.pwa_version() == 100


@pytest.mark.parametrize("name", golden_names("geo_"))
def test_c_geometry_bit_exact_vs_reference(name):
    d = load_npz(name)
    m = [int(v) for v in d["meta"]]
    dims, ws, shift_cfg = tuple(m[0:3]), tuple(m[3:6]), tuple(m[6:9])
    g = pwa_b200.Geometry(dims, ws, shift_cfg)
    assert g.pads == tuple(int(v) for v in d["pads"])
    assert g.shift == tuple(int(v) for v in d["shift"])
    assert np.array_equal(g.index_map_host(0).astype(np.int64), d["index_map"])
    assert g.masked == ("mask_bits" in d)
    if g.masked:
        shape = tuple(int(v) for v in d["mask_shape"])
        ref = np.unpackbits(d["mask_bits"], axis=-1)[..., : shape[-1]].astype(bool)
        ids = g.region_ids_host()
        assert np.array_equal(ids[:, :, None] == ids[:, None, :], ref)
        # the free function with the reference's signature
        mask = pwa_b200.get_attn_mask(g.sp, ws, g.shift, g.pads)
        assert mask.dtype == torch.float32 and tuple(mask.shape) == shape
        assert np.array_equal(mask[0].numpy().astype(bool), ref)


def test_c_geometry_matches_oracle_on_bench_shapes():
    for dims in [(48, 48, 48), (24, 24, 24), (12, 12, 24), (64, 64, 64), (32, 32, 32), (16, 16, 32), (5, 9, 3)]:
        for ws, sh in [((8, 8, 4), (4, 4, 2)), ((8, 8, 4), (0, 0, 0)), ((4, 4, 2), (2, 2, 1))]:
            g = pwa_b200.Geometry(dims, ws, sh)
            pads = R.pad_amounts(dims, ws)
            shift = R.effective_shift(dims, ws, sh)
            assert g.pads == pads and g.shift == shift
            assert np.array_equal(g.index_map_host(0), R.gather_index(dims, ws, shift, pads))
            assert np.array_equal(g.index_map_host(1), R.gather_index(dims, ws, shift, pads, R.crop_lo(pads)))
            if g.masked:
                assert np.array_equal(g.region_ids_host(), R.region_ids(dims, ws, shift, pads))


def test_geometry_rejects_bad_arguments():
    with pytest.raises(pwa_b200._lib.PwaError):
        pwa_b200.Geometry((0, 8, 8), (4, 4, 2), (0, 0, 0))
    with pytest.raises(pwa_b200._lib.PwaError):
        pwa_b200.Geometry((8, 8, 8), (4, 4, 2), (4, 0, 0))


def test_state_dict_keys_and_shapes_match_reference():
    meta, sd, *_ = load_block_case("blk_w884_dh12_shift", torch.float32)
    blk = pwa_b200.SwinTransformerBlock(hidden_channels=meta["C"], window_size=meta["ws"],
                                        pos_bias_embed_dim=meta["E"], num_heads=meta["heads"], max_prompts=1,
                                        tokens_per_prompt=meta["I"], shift_size=meta["shift"])
    ours = blk.state_dict()
    assert set(ours.keys()) == set(sd.keys())
    for k in sd:
        assert tuple(ours[k].shape) == tuple(sd[k].shape), k
        assert ours[k].dtype == sd[k].dtype or not sd[k].is_floating_point(), k
    blk.load_state_dict(sd)            # reference checkpoints load unchanged
    assert torch.equal(blk.pe.relative_dist_h, sd["pe.relative_dist_h"])


def test_pair_state_dict_keys_match_reference():
    d = load_npz("pair_merge")
    ref_keys = {k[len("mld1.sd."):] for k in d if k.startswith("mld1.sd.")}
    pair = pwa_b200.ConsecutiveSwinBlocks(hidden_channels=12, num_heads=2, pos_bias_embed_dim=16, max_prompts=1,
                                          tokens_per_prompt=8, window_size=(4, 4, 2), down=True)
    assert set(pair.state_dict().keys()) == ref_keys
    names = [n for n, _ in pair.named_parameters_body()]
    assert any(n.startswith("reduction") for n in names) and any("to_q" in n for n in names)
    assert len(pair.named_parameters_bias_content()) == 12 and len(pair.named_parameters_bias_prompt_tokens()) == 4


def test_relative_pe_tables_match_reference():
    d = load_npz("pe_small")
    pe = pwa_b200.RelativePE(embed_dim=16, num_heads=3, max_abs_pos=(4, 4, 2), max_cap_dist=(4, 4, 2),
                             max_prompts=2, tokens_per_prompt=3).double()
    pe.load_state_dict({k[3:]: torch.from_numpy(v) for k, v in d.items() if k.startswith("sd.")})
    dense = pe(4, 4, 2, 6)
    assert tuple(dense.shape) == d["bias_prompt"].shape
    assert np.abs(dense.detach().numpy() - d["bias_prompt"]).max() < 1e-6
    assert np.abs(pe(4, 4, 2, 0).detach().numpy() - d["bias_content"]).max() < 1e-6
    with pytest.raises(RuntimeError):
        pe.tables(4, 4, 2, 5)          # dim_i must equal max_prompts * tokens_per_prompt


def test_no_cpu_fallback():
    blk = pwa_b200.SwinTransformerBlock(hidden_channels=12, window_size=(4, 4, 2), pos_bias_embed_dim=16,
                                        num_heads=4, max_prompts=1, tokens_per_prompt=8, shift_size=(0, 0, 0))
    with pytest.raises(RuntimeError, match="no CPU path"):
        blk(torch.zeros(1, 12, 8, 8, 4))
    with pytest.raises(ValueError, match="not compatible with the number of heads"):
        pwa_b200.WindowAttention(dim=10, num_heads=4)


def test_bench_reference_arm_prints_the_contract_line():
    """`bench.py --impl reference` (the CPU arm the driver runs next to ours) prints one JSON line with the contract keys."""
    import json
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    out = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1"],
                         capture_output=True, text=True, timeout=300, cwd=root)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["unit"] == "patches/s" and line["value"] > 0
    for key in ("metric", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "dtype", "data", "config",
                "cpu_baseline", "e2e"):
        assert key in line, key
    assert line["cpu_baseline"]["kind"] == "port" and line["cpu_baseline"]["cores"] >= 1
    assert line["e2e"]["h2d_bytes_per_step"] == 0 and line["e2e"]["d2h_bytes_per_step"] == 0
    assert line["steps"] == 1


def test_bench_rejects_zero_steps():
    import subprocess
    import sys
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "0"],
                         capture_output=True, text=True, timeout=300, cwd=ROOT)
    assert out.returncode == 2 and "--steps must be at least 1" in out.stderr
    assert out.stdout == ""


def test_bench_dump_outputs_budget_and_sample(tmp_path):
    """bench.dump_outputs: arrays that fit an even share of the byte budget are written whole as float32 (float64 stays
    float64), a larger one as the same sorted, seeded sample on every call, and the data stays within the budget."""
    import bench
    g = torch.Generator().manual_seed(3)
    arrays = {"loss": torch.tensor(2.5), "small": torch.arange(10, dtype=torch.bfloat16),
              "mid": torch.randn(2, 500, generator=g), "big": torch.randn(50, 100, generator=g, dtype=torch.float64)}
    budget = 12000
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), arrays, budget=budget)
    got = {k: np.load(tmp_path / "a" / f"{k}.npy") for k in arrays}
    assert sorted(os.listdir(tmp_path / "a")) == sorted(f"{k}.npy" for k in arrays)
    assert got["loss"].dtype == np.float32 and got["loss"].shape == () and got["loss"] == 2.5
    assert got["small"].dtype == np.float32 and np.array_equal(got["small"], np.arange(10, dtype=np.float32))
    assert got["mid"].dtype == np.float32 and np.array_equal(got["mid"], arrays["mid"].numpy())
    big, full = got["big"], arrays["big"].numpy().reshape(-1)
    assert big.dtype == np.float64 and big.ndim == 1 and 0 < big.size < full.size
    pos = {v: i for i, v in enumerate(full)}
    idx = np.array([pos[v] for v in big])
    assert np.all(np.diff(idx) > 0)                                   # distinct elements, in flat order
    assert sum(v.nbytes for v in got.values()) <= budget
    for k in arrays:
        assert np.array_equal(np.load(tmp_path / "b" / f"{k}.npy"), got[k])


def test_token_split_picks_a_divisor_near_72():
    """The weight-gradient GEMM slices the token axis into S batches: S divides T, lies in [32, 160] and is the divisor
    closest to 72; 0 (= single GEMM) when no such divisor exists."""
    from pwa_b200.functional import _token_split
    for T in (442368, 55296, 28672, 6912, 4 * 13824, 32 * 17, 160 * 1001):
        S = _token_split(T)
        assert S and T % S == 0 and 32 <= S <= 160, (T, S)
        assert all(abs(d - 72) >= abs(S - 72) for d in range(32, 161) if T % d == 0)
    assert _token_split(1000003) == 0 and _token_split(31) == 0


def test_dropout_mask_restatements_agree():
    """oracle: the numpy and the torch (device-agnostic, chunkable) restatements of the kernels' dropout hash mask."""
    for words, p_drop in (([123456789, 987654321], 0.25), ([31337, -5], 0.1), ([0, 0], 0.003)):
        a = R.dropout_keep_factor(words, 2, 3, 4, 6, 10, p_drop)
        b = R.dropout_keep_factor_torch(words, 0, 6, 4, 6, 10, p_drop).reshape(2, 3, 4, 6, 10)
        assert torch.equal(a, b)
        c = R.dropout_keep_factor_torch(words, 3, 3, 4, 6, 10, p_drop)
        assert torch.equal(a.reshape(6, 4, 6, 10)[3:], c)


@pytest.mark.parametrize("name,mode,dec_prompt", [("model_cfg1", 'self_supervised_learning_encoder', False),
                                                  ("model_cfg3_small", 'self_supervised_learning_all', True),
                                                  ("model_cfg4_small", 'downstream', True)])
def test_swin_unetr_state_dict_and_freeze_logic_match_reference(name, mode, dec_prompt):
    """MONAI-free SwinUnetR host (SURVEY §8f-3): exactly the reference model's state-dict keys and shapes (reference
    checkpoints load unchanged; incl. MONAI Convolution's child name `conv`) and the same set of trainable parameters per
    training mode (swin_unetr.py:21-40), recorded from the live reference by oracle/gen_golden_model.py."""
    from oracle import gen_golden_model as G
    d = load_npz(name)
    model = pwa_b200.SwinUnetR(G.model_conf(mode, dec_prompt=dec_prompt))
    ours = [f"{k}:{'x'.join(str(v) for v in t.shape)}" for k, t in model.state_dict().items()]
    assert sorted(ours) == sorted(str(s) for s in d["sd_keys"])
    assert sorted(n for n, p in model.named_parameters() if p.requires_grad) == [str(s) for s in d["trainable"]]
    if mode == 'downstream':
        assert sorted(id(p) for _, p in model.named_parameters_downstream()) == sorted(id(p) for p in model.parameters() if p.requires_grad)
