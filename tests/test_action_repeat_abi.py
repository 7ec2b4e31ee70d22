"""CPU: the action-repeat setter and getter of the C-ABI check their handle without a device."""
from spacefortress_b200 import _lib


def test_action_repeat_calls_reject_a_null_handle():
    L = _lib.lib()
    assert L.sf_set_action_repeat(None, 2) == _lib.SF_ERR_INVALID
    assert b"handle" in L.sf_last_error()
    assert L.sf_action_repeat(None) == -1


def test_the_limit_is_one_episode():
    src = open(_lib.os.path.join(_lib.HERE, "..", "include", "sf_b200.h")).read()
    assert "#define SF_MAX_ACTION_REPEAT %d" % _lib.MAX_ACTION_REPEAT in src
    assert _lib.MAX_ACTION_REPEAT == 5295  # ceil(180000 / 34) ticks: game.cpp:487-489
