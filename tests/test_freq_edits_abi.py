"""CPU-only checks of chromo_freq_edits_workspace_floats and of the argument errors of chromo_freq_edits (they are
reported before anything touches a device), and that the workspace bounds of the other entry points did not move."""
import ctypes

from _util import KWS
from chromoformer_b200 import ChromoformerClassifier, _lib

EINVAL, ENOMEM = -1, -2
F_REGONLY = 8


def _cfg(i_max=8, reg=None):
    m = ChromoformerClassifier(7, 128, 128, dict(KWS[0]), dict(KWS[1]), dict(reg or KWS[2]), i_max=i_max)
    return _lib.Config.from_buffer_copy(m._cfg)


def test_workspace_is_the_subsets_bound_plus_the_drop_words():
    lib = _lib.load()
    for i_max in (8, 16):
        cfg = _cfg(i_max)
        for f in (0, _lib.F_BF16, _lib.F_BF16 | _lib.F_DENSE):
            for B in (1, 64, 4096):
                for V in (1, 3, 4, 1023, 65536):
                    sub = lib.chromo_pcre_subsets_workspace_floats(ctypes.byref(cfg), B, V, f)
                    got = lib.chromo_freq_edits_workspace_floats(ctypes.byref(cfg), B, V, f)
                    assert got == sub + (V + 3) // 4 * 4, (i_max, f, B, V)


def test_workspace_argument_errors():
    lib = _lib.load()
    cfg = _cfg()
    assert lib.chromo_freq_edits_workspace_floats(ctypes.byref(cfg), 0, 4, 0) == EINVAL
    assert lib.chromo_freq_edits_workspace_floats(ctypes.byref(cfg), 4, 0, 0) == EINVAL
    assert lib.chromo_freq_edits_workspace_floats(ctypes.byref(cfg), 4, 1 << 30, 0) == EINVAL
    assert b"chromo_freq_edits" in lib.chromo_last_error()
    assert lib.chromo_freq_edits_workspace_floats(ctypes.byref(cfg), 4, 4, 0) > 0


def _call(lib, cfg, batch, gene, freq, logits, var_logits, ws, ws_floats, flags, V=1):
    return lib.chromo_freq_edits(ctypes.byref(cfg), 1, ctypes.byref(batch), gene, freq, V, logits, var_logits, ws,
                                 ws_floats, flags, None)


def test_flag_and_pointer_errors():
    """Unsupported flags, null pointers and variants < 1 are CHROMO_EINVAL with a message, a short workspace
    CHROMO_ENOMEM, all before any device access (every pointer here is a dummy host address)."""
    lib = _lib.load()
    cfg = _cfg()
    batch = _lib.Batch()
    batch.batch = 2
    for r in range(cfg.n_res):
        for name in ("x_p", "x_pcre", "mask_p", "mask_pcre", "imask", "pos_enc"):
            getattr(batch, name)[r] = 16
    batch.freq = 16
    big = 1 << 40
    for flags in (_lib.F_TRAINING, _lib.F_BF16 | _lib.F_TRAINING, F_REGONLY, _lib.F_BWD_HEAD_REG, _lib.F_BWD_REST,
                  _lib.F_FREQ_GRAD, 1 << 10):
        assert _call(lib, cfg, batch, 16, 16, 16, 16, 16, big, flags) == EINVAL, flags
        assert b"inference only" in lib.chromo_last_error()
    for args in ((None, 16, 16, 16), (16, None, 16, 16), (16, 16, 16, None)):
        g, f, lg, vl = args
        assert _call(lib, cfg, batch, g, f, lg, vl, 16, big, _lib.F_BF16) == EINVAL, args
        assert b"null" in lib.chromo_last_error()
    assert _call(lib, cfg, batch, 16, 16, None, 16, 16, big, 0) == EINVAL
    assert _call(lib, cfg, batch, 16, 16, 16, 16, None, big, 0) == EINVAL
    assert _call(lib, cfg, batch, 16, 16, 16, 16, 16, big, 0, V=0) == EINVAL
    assert b"variants" in lib.chromo_last_error()
    for f in (0, _lib.F_BF16):
        need = lib.chromo_freq_edits_workspace_floats(ctypes.byref(cfg), 2, 5, f)
        assert _call(lib, cfg, batch, 16, 16, 16, 16, 16, need - 1, f, V=5) == ENOMEM
        assert b"workspace too small" in lib.chromo_last_error()
        assert str(need).encode() in lib.chromo_last_error()


def test_other_workspaces_unchanged():
    """The freq-edit entry point leaves the forward, deletion, subsets and occlusion workspaces as they were (values of
    the parent revision for the default configuration, i_max 8 and 16)."""
    lib = _lib.load()
    got = []
    for i_max in (8, 16):
        cfg = _cfg(i_max)
        for f in (0, _lib.F_BF16):
            for B in (1, 64, 4096):
                got.append((i_max, f, B, lib.chromo_workspace_floats(ctypes.byref(cfg), B, f),
                            lib.chromo_pcre_deletion_workspace_floats(ctypes.byref(cfg), B, f),
                            lib.chromo_pcre_subsets_workspace_floats(ctypes.byref(cfg), B, 3 * B, f),
                            lib.chromo_pcre_occlusion_workspace_floats(ctypes.byref(cfg), B, 3 * B, f)))
    assert got == EXPECTED, got


# (i_max, flags, batch, chromo_workspace_floats, chromo_pcre_deletion_workspace_floats,
#  chromo_pcre_subsets_workspace_floats and chromo_pcre_occlusion_workspace_floats with 3 * batch variants)
EXPECTED = [
    (8, 0, 1, 1952992, 3671672, 2009660, 2011968), (8, 0, 64, 15800320, 129629040, 24612432, 24760080),
    (8, 0, 4096, 909475840, 8191859712, 1474335744, 1483785216), (8, 2, 1, 8154748, 9875704, 8160108, 8162416),
    (8, 2, 64, 22008796, 135900992, 22260764, 22408412), (8, 2, 4096, 916120520, 8202472664, 932160036, 941609508),
    (16, 0, 1, 2149088, 9024544, 2329472, 2331780), (16, 0, 64, 29235200, 471426544, 46456656, 46604304),
    (16, 0, 4096, 1766653952, 30068669440, 2870596608, 2880046080),
    (16, 2, 1, 8350940, 15231560, 8360464, 8362772), (16, 2, 64, 35450528, 477885456, 35970840, 36118488),
    (16, 2, 4096, 1773733596, 30091252200, 1806944752, 1816394224),
]
