"""CPU: the variant builds the tools make still compile. Each probe of csrc/sf_probe.cuh exports its reader and the
product library exports neither (the probes are build variants, never part of the product); a build with another
granule of the host-buffer delta updates exports the whole C-ABI."""
import ctypes as C
import os
from concurrent.futures import ThreadPoolExecutor

import pytest

from spacefortress_b200 import _lib, build

PROBES = {"-DSF_BARRIER_TIMING": "sf_barrier_cycles", "-DSF_TIMELINE": "sf_timeline"}


@pytest.fixture(scope="module")
def nvcc():
    if os.environ.get("SF_SKIP_NVCC_BUILD") == "1":
        pytest.skip("SF_SKIP_NVCC_BUILD=1")
    try:
        return build._nvcc()
    except RuntimeError:
        pytest.skip("nvcc not found")


def test_probe_variants_build_and_export_their_readers(nvcc, tmp_path):
    outs = {d: str(tmp_path / ("libsf%s.so" % d.lower().replace("-dsf", ""))) for d in PROBES}
    with ThreadPoolExecutor(len(PROBES)) as ex:
        for f in [ex.submit(build.build, out=outs[d], defs=d) for d in PROBES]:
            f.result()
    for d, reader in PROBES.items():
        L = C.CDLL(outs[d])
        for name in PROBES.values():
            assert hasattr(L, name) == (name == reader), (d, name)
    product = C.CDLL(build.build())
    for name in PROBES.values():
        assert not hasattr(product, name), name


def test_delta_granule_is_a_build_define(nvcc, tmp_path):
    """The granule of the host-buffer delta updates is fixed when the library is built: a variant with another granule
    (tools/gpu_host_step_ranks.py) compiles and exports the whole C-ABI, and the product library has no run-time knob
    that names it."""
    out = str(tmp_path / "libsf_granule32.so")
    build.build(out=out, defs="-DSF_DELTA_GRANULE=32")
    L = C.CDLL(out)
    assert [s for s in _lib.EXPORTED_SYMBOLS if not hasattr(L, s)] == []
    with open(build.build(), "rb") as f:
        assert b"SF_DELTA_GRANULE" not in f.read()
