"""CPU check of the chromo_input_grads_t binding: the ctypes mirror has the size and member offsets the C compiler gives
the header's struct, and F_FREQ_GRAD is the header's CHROMO_F_FREQ_GRAD."""
import ctypes
import os
import shutil
import subprocess

import pytest

from _util import ROOT
from chromoformer_b200 import _lib

_PROBE = r"""
#include <stddef.h>
#include <stdio.h>
#include "chromoformer_b200.h"
int main(void) {
    printf("%d %zu %zu %zu %zu\n", CHROMO_F_FREQ_GRAD, sizeof(chromo_input_grads_t),
           offsetof(chromo_input_grads_t, x_p), offsetof(chromo_input_grads_t, x_pcre),
           offsetof(chromo_input_grads_t, freq));
    return 0;
}
"""


def test_input_grads_struct_matches_header(tmp_path):
    cc = shutil.which("cc") or shutil.which("gcc")
    if cc is None:
        pytest.skip("no C compiler")
    src, exe = tmp_path / "probe.c", tmp_path / "probe"
    src.write_text(_PROBE)
    subprocess.check_call([cc, "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)])
    flag, size, off_xp, off_xpcre, off_freq = map(int, subprocess.check_output([str(exe)]).split())
    G = _lib.InputGrads
    assert flag == _lib.F_FREQ_GRAD == 128
    assert ctypes.sizeof(G) == size
    assert (G.x_p.offset, G.x_pcre.offset, G.freq.offset) == (off_xp, off_xpcre, off_freq)
    # the new member trails the struct: callers built against the two-array layout see unchanged offsets
    assert off_freq == 2 * _lib.MAX_RES * ctypes.sizeof(ctypes.c_void_p)
