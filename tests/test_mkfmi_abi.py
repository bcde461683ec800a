"""kj_mkfmi without a GPU: argument errors are reported before anything else, and a valid request fails with KJ_ERR_NO_DEVICE
(there is no CPU fallback)."""
import ctypes as C
import pytest


def _opts(kb, e=3, alphabet=None):
    return kb.KjMkfmiOpts(e, alphabet, 0)


def test_mkfmi_argument_errors(built, tmp_path):
    import kaiju_b200 as kb
    L = kb.lib(); st = kb.KjMkfmiStats()
    faa = tmp_path / "a.faa"; faa.write_text(">a\nMKVLA\n")
    assert L.kj_mkfmi(None, b"x", C.byref(_opts(kb)), 0, C.byref(st)) == -1
    assert L.kj_mkfmi(str(faa).encode(), None, C.byref(_opts(kb)), 0, C.byref(st)) == -1
    assert L.kj_mkfmi(str(faa).encode(), b"x", C.byref(_opts(kb, e=17)), 0, C.byref(st)) == -1
    assert L.kj_mkfmi(str(faa).encode(), b"x", C.byref(_opts(kb, alphabet=b"AC*")), 0, C.byref(st)) == -1
    assert L.kj_mkfmi(str(faa).encode(), b"x", C.byref(_opts(kb, alphabet=b"ACA")), 0, C.byref(st)) == -1
    assert L.kj_mkfmi(str(faa).encode(), b"x", C.byref(_opts(kb, alphabet=b"ABCDEFGHIJKLMNOPQRSTUVWXY")), 0, C.byref(st)) == -5
    assert b"24 letters" in L.kj_last_error()
    assert L.kj_mkfmi(str(faa).encode(), b"x", C.byref(_opts(kb, alphabet=b"DNA")), 0, C.byref(st)) == -5


def test_mkfmi_no_cpu_fallback(built, tmp_path):
    import torch
    import kaiju_b200 as kb
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    faa = tmp_path / "a.faa"; faa.write_text(">a\nMKVLA\n")
    with pytest.raises(kb.KaijuError) as e:
        kb.build_index(str(faa), str(tmp_path / "a"))
    assert "-4" in str(e.value) and not (tmp_path / "a.fmi").exists()
