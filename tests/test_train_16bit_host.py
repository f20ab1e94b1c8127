"""16-bit logits on the training entry (`d3pm_train_desc.logits_dtype`): argument checks and the descriptor layout, without
a GPU."""
import ctypes
import os
import shutil
import subprocess

import pytest
import torch

import d3pm_b200
from d3pm_b200 import _lib, ops, train

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _desc(K, dtype, pitch=None, B=3, N=1024):
    """A forward-only descriptor on fake, non-null, 16-byte aligned pointers: every check passes up to the one a test
    wants to see fail, and none of them touches the device."""
    d = _lib.TrainDesc()
    d.logits = d.x0 = d.x_t = d.t = d.coef_table = d.tok_main = d.tok_aux = 16
    d.B, d.N, d.K, d.T = B, N, K, 100
    d.pitch = K if pitch is None else pitch
    d.backward = 0
    d.logits_dtype = dtype
    return d


def test_16bit_training_arguments_are_checked_before_any_launch():
    lib = d3pm_b200.load_library()
    for bad in (3, -1, 99):
        assert lib.d3pm_train_rows(ctypes.byref(_desc(1024, bad))) == -1
        assert b"logits_dtype" in lib.d3pm_last_error()
    for dtype in (_lib.LOGITS_F16, _lib.LOGITS_BF16):
        assert lib.d3pm_train_rows(ctypes.byref(_desc(1024, dtype, pitch=1028))) == -2  # 16-bit rows: pitch % 8
        d = _desc(1024, dtype)
        d.backward, d.grad, d.w_main, d.w_aux, d.pitch_grad = 1, 16, 16, 16, 1028
        assert lib.d3pm_train_rows(ctypes.byref(d)) == -2                                # ... and pitch_grad % 8
        assert lib.d3pm_train_rows(ctypes.byref(_desc(64, dtype))) == -3                 # not a stream-kernel codebook
        assert lib.d3pm_train_rows(ctypes.byref(_desc(1024, dtype, B=1))) == -3          # fewer than 2048 rows
        d = _desc(1024, dtype)
        d.x0_recon = 16                                                                  # one arg-max output of two
        assert lib.d3pm_train_rows(ctypes.byref(d)) == -3
        assert b"cast to float" in lib.d3pm_last_error()
    # float32 rows keep their old rules: pitch % 4 suffices
    assert lib.d3pm_train_rows(ctypes.byref(_desc(1024, _lib.LOGITS_F32, pitch=1030))) == -2


def test_python_mirror_of_the_stream_predicate():
    def rows(B, N, K, pitch=None):
        base = torch.empty(B, N, pitch or K, dtype=torch.float16)
        return base[..., :K], pitch or K
    assert train.stream_takes_16bit(*rows(2, 1024, 4096))
    assert train.stream_takes_16bit(*rows(3, 1024, 1024, pitch=1032))
    assert not train.stream_takes_16bit(*rows(2, 1024, 1024, pitch=1028))
    assert not train.stream_takes_16bit(*rows(1, 1024, 2048))
    assert not train.stream_takes_16bit(*rows(4, 1024, 64))
    assert set(ops.STREAM_CODEBOOKS) == {1024, 2048, 4096}


def test_16bit_logit_rows_are_zero_copy_for_the_reference_layout():
    for dtype in (torch.float16, torch.bfloat16):
        x = torch.zeros(2, 16, 1024, dtype=dtype)  # [B, N, K] storage, handed on as its [B, K, N] view
        rows, pitch = train._logit_rows(x.permute(0, 2, 1))
        assert rows.dtype == dtype and pitch == 1024 and rows.data_ptr() == x.data_ptr()


@pytest.mark.skipif(shutil.which("cc") is None, reason="needs a C compiler")
def test_train_desc_layout_matches_the_header(tmp_path):
    src = tmp_path / "layout.c"
    src.write_text('#include <stddef.h>\n#include <stdio.h>\n#include "d3pm_b200.h"\n'
                   'int main(void) { printf("%zu %zu %zu\\n", offsetof(d3pm_train_desc, stream), '
                   'offsetof(d3pm_train_desc, logits_dtype), sizeof(d3pm_train_desc)); return 0; }\n')
    exe = tmp_path / "layout"
    subprocess.run(["cc", "-I", os.path.join(ROOT, "include"), "-o", str(exe), str(src)], check=True)
    got = [int(v) for v in subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout.split()]
    assert got == [_lib.TrainDesc.stream.offset, _lib.TrainDesc.logits_dtype.offset, ctypes.sizeof(_lib.TrainDesc)]
