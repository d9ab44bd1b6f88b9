"""CPU-only checks of the deterministic siblings (include/pwa.h): they and their workspace size queries are exported, the
queries answer without a GPU, and the calls that must fail do so before touching the device: the deterministic attention
backward outside the tcgen05 envelope (PWA_ERR_UNSUPPORTED) and any sibling given a workspace smaller than its query
(PWA_ERR_ARG)."""
import ctypes

import pwa_b200
from pwa_b200 import _lib
from pwa_b200.functional import _shape_struct

L = _lib.lib
BF16, F16, F32 = _lib.PWA_BF16, _lib.PWA_F16, _lib.PWA_F32
SIBLINGS = ("pwa_attn_bwd", "pwa_ln_bwd2", "pwa_dropout_colsum", "pwa_colsum_rows", "pwa_bias_tables_bwd")


def test_siblings_and_size_queries_are_exported():
    lib = ctypes.CDLL(_lib.LIB_PATH)
    for name in SIBLINGS:
        for sym in (name + "_det", name + "_det_workspace_size"):
            assert hasattr(lib, sym), sym
            assert sym in _lib.EXPORTED_SYMBOLS


def _enc0(dh=12, I=64, heads=4, ws=(8, 8, 4)):
    return _shape_struct(4, 432, dh * heads, heads, I, ws, dh ** -0.5)


def test_attention_workspace_size_at_enc0():
    # 148 CTAs (a multiple of heads = 4): 37 slots; prompt dK and dV [37][B][I][C], then the table slots [37][heads][...]
    slots, B, I, C, h = 37, 4, 64, 48, 4
    floats = 2 * slots * B * I * C + slots * h * (8 * 8 + 8 * 8 + 4 * 4 + I)
    for dt in (BF16, F16):
        assert L.pwa_attn_bwd_det_workspace_size(ctypes.byref(_enc0()), dt) == 4 * floats


def test_attention_outside_the_envelope_is_unsupported():
    cases = [(_enc0(), F32), (_enc0(dh=8), BF16), (_enc0(I=48), BF16), (_enc0(ws=(4, 4, 2)), F16)]
    for s, dt in cases:
        assert L.pwa_attn_tc_supported(ctypes.byref(s), dt) == 0
        assert L.pwa_attn_bwd_det_workspace_size(ctypes.byref(s), dt) == -2
        null = [None] * 23
        assert L.pwa_attn_bwd_det(*null, None, 0, ctypes.byref(s), dt, None) == -2
        assert b"deterministic" in L.pwa_last_error()


def test_token_domain_workspace_sizes():
    rows = 442368
    # pwa_colsum_rows: at most 296 CTAs, one [C] slot each
    assert L.pwa_colsum_rows_det_workspace_size(rows, 48, BF16) == 296 * 48 * 4
    assert L.pwa_colsum_rows_det_workspace_size(0, 48, BF16) == 0
    # pwa_dropout_colsum: at most 148 * 8 CTAs
    assert L.pwa_dropout_colsum_det_workspace_size(rows, 48, BF16) == 148 * 8 * 48 * 4
    # pwa_ln_bwd2: four [blocks][C] slot arrays; bf16 C = 48 takes the bulk kernel (296 CTAs) when aligned, else the register
    # kernel (G = 16: 16 rows per CTA, 592 CTAs): the size covers both
    assert L.pwa_ln_bwd2_det_workspace_size(rows, 48, BF16) == 592 * 4 * 48 * 4
    assert L.pwa_ln_bwd2_det_workspace_size(rows, 48, F32) == 592 * 4 * 48 * 4
    a3 = ctypes.c_int32 * 3
    assert L.pwa_bias_tables_bwd_det_workspace_size(4, 64, a3(8, 8, 4), a3(8, 8, 4), 64) == 0
    for bad in (L.pwa_colsum_rows_det_workspace_size(rows, 12, BF16), L.pwa_dropout_colsum_det_workspace_size(rows, 6, F32),
                L.pwa_ln_bwd2_det_workspace_size(rows, 4096, BF16), L.pwa_ln_bwd2_det_workspace_size(-1, 48, BF16)):
        assert bad == -1


def test_small_workspace_is_an_argument_error():
    fake = ctypes.c_void_p(1 << 20)          # never dereferenced: the size check comes first
    rows, C = 4096, 48
    rc = L.pwa_ln_bwd2_det(*[fake] * 7, fake, fake, None, None, rows, C, BF16, fake, 16, None)
    assert rc == -1 and b"workspace" in L.pwa_last_error()
    rc = L.pwa_colsum_rows_det(fake, fake, rows, C, BF16, fake, 16, None)
    assert rc == -1 and b"workspace" in L.pwa_last_error()
    rc = L.pwa_dropout_colsum_det(fake, fake, rows, C, 0.1, fake, fake, BF16, fake, 16, None)
    assert rc == -1 and b"workspace" in L.pwa_last_error()
    s = _enc0()
    rc = L.pwa_attn_bwd_det(*[fake] * 23, fake, 1024, ctypes.byref(s), BF16, None)
    assert rc == -1 and b"workspace" in L.pwa_last_error()


def test_module_imports_without_gpu():
    assert pwa_b200._lib.lib.pwa_version() == 100
