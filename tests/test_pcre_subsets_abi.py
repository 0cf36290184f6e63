"""CPU-only checks of chromo_pcre_subsets_workspace_floats: the replay layout has no Embedding / Pairwise block, so the
workspace grows by at most 96 kB per variant in BF16 with the default configuration (i_max 8)."""
import ctypes

from _util import KWS
from chromoformer_b200 import ChromoformerClassifier, _lib


def _cfg(i_max=8, reg=None):
    m = ChromoformerClassifier(7, 128, 128, dict(KWS[0]), dict(KWS[1]), dict(reg or KWS[2]), i_max=i_max)
    return _lib.Config.from_buffer_copy(m._cfg)


def test_workspace_per_variant():
    lib = _lib.load()
    cfg = _cfg()
    n = lambda B, V, f: lib.chromo_pcre_subsets_workspace_floats(ctypes.byref(cfg), B, V, f)
    for B in (1, 64, 4096):
        for V0, V1 in ((1024, 2048), (65536, 131072)):
            grow = (n(B, V1, _lib.F_BF16) - n(B, V0, _lib.F_BF16)) * 4 / (V1 - V0)
            assert 0 < grow <= 96 * 1024, (B, V0, grow)
    # FP32 keeps the layer-by-layer Regulation buffers (about 0.5 MB per variant); a deletion workspace needs a full
    # forward layout per variant
    fp32 = (n(64, 2048, 0) - n(64, 1024, 0)) * 4 / 1024
    assert 0.4e6 < fp32 < 0.6e6, fp32
    bf16 = (n(64, 2048, _lib.F_BF16) - n(64, 1024, _lib.F_BF16)) * 4 / 1024
    dele = lib.chromo_pcre_deletion_workspace_floats(ctypes.byref(cfg), 64, _lib.F_BF16) * 4 / (64 * 9)
    print(f"bytes per variant: BF16 {bf16:.0f}, FP32 {fp32:.0f}; deletion {dele:.0f}")
    assert dele > 10 * bf16


def test_workspace_argument_errors():
    lib = _lib.load()
    cfg = _cfg()
    assert lib.chromo_pcre_subsets_workspace_floats(ctypes.byref(cfg), 0, 4, 0) == -1
    assert lib.chromo_pcre_subsets_workspace_floats(ctypes.byref(cfg), 4, 0, 0) == -1
    assert lib.chromo_pcre_subsets_workspace_floats(ctypes.byref(cfg), 4, 1 << 30, 0) == -1
    assert lib.chromo_pcre_subsets_workspace_floats(ctypes.byref(cfg), 4, 4, 0) > 0
