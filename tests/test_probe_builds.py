"""CPU: the probe builds of csrc/sf_probe.cuh still compile, each exports its reader, and the product library exports
neither (the probes are build variants, never part of the product)."""
import ctypes as C
import os
from concurrent.futures import ThreadPoolExecutor

import pytest

from spacefortress_b200 import build

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
