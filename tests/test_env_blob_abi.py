"""CPU: the env-blob constants of the ctypes binding are the header's."""
import os
import re

from spacefortress_b200 import _lib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_env_blob_constants_match_the_header():
    src = open(os.path.join(ROOT, "include", "sf_b200.h")).read()
    defs = dict(re.findall(r"#define\s+(SF_ENV_BLOB_\w+)\s+(\w+)", src))
    assert int(defs["SF_ENV_BLOB_BYTES"]) == _lib.ENV_BLOB_BYTES
    assert int(defs["SF_ENV_BLOB_VERSION"]) == _lib.ENV_BLOB_VERSION
    assert _lib.ENV_BLOB_BYTES % 16 == 0
