"""CPU: the final-observation calls of the C-ABI without a device: the NULL handle and the binding."""
from spacefortress_b200 import _lib


def test_final_obs_calls_reject_a_null_handle():
    L = _lib.lib()
    assert L.sf_set_final_obs(None, None, None, None) == _lib.SF_ERR_INVALID
    assert b"handle" in L.sf_last_error()
    assert L.sf_final_obs_enabled(None) == -1


def test_the_binding_exports_both_calls():
    L = _lib.lib()
    for name in ("sf_set_final_obs", "sf_final_obs_enabled"):
        assert name in _lib.EXPORTED_SYMBOLS and hasattr(L, name), name
    src = open(_lib.os.path.join(_lib.HERE, "..", "include", "sf_b200.h")).read()
    assert "int sf_set_final_obs(sf_handle* h, uint8_t* d_frames, float* d_rows, int32_t* d_final_step);" in src
    assert "int sf_final_obs_enabled(const sf_handle* h);" in src
