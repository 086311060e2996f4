"""The batch-from-device entry points of include/csg.h are exported by libcsg.so (no GPU needed)."""
import ctypes as C

import pytest

NEW = ("csg_prove_many_device", "csg_build_traces_many_rescue", "csg_build_traces_many_schnorr",
       "csg_build_traces_many_merkle_update", "csg_build_traces_many_transaction")


@pytest.mark.parametrize("name", NEW)
def test_exported(csg, name):
    assert hasattr(C.CDLL(str(csg.LIB_PATH)), name)
    assert callable(getattr(csg.lib(), name))
