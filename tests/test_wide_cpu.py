"""The wide kernels without a GPU: built for sm_100a within the register budget of one 512-thread CTA per SM, carried
inside the library, and the getter that says whether a context runs them is exported."""
import os
import re
import shutil
import subprocess

import pytest

import pmdi_b200  # noqa: F401
from pmdi_b200 import capi

CUBIN = os.path.join(os.path.dirname(capi.LIB_PATH), "pmdi_sweep_wide.cubin")
WIDE_KERNELS = ["k_eval_row_wide", "k_sweep_pool_wide", "k_sweep_pool_wide_dbg", "k_sweep_spec_wide",
                "k_sweep_spec_wide_dbg"]


def test_wide_module_holds_the_wide_kernels_and_ships_in_the_library():
    capi.build()
    tool = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    if not os.path.exists(tool):
        pytest.skip("cuobjdump not available")
    out = subprocess.run([tool, "--dump-resource-usage", CUBIN], capture_output=True, text=True).stdout
    # nothing else: a kernel next to them shares their non-inlined device functions
    assert sorted(re.findall(r"Function (\w+):", out)) == WIDE_KERNELS
    for k in WIDE_KERNELS:
        m = re.search(r"Function %s:\s*\n\s*REG:(\d+) STACK:(\d+)" % k, out)
        assert m, f"{k} not found in {CUBIN}"
        assert int(m.group(1)) <= 128, (k, m.group(1))
    blob = open(capi.LIB_PATH, "rb").read()
    assert open(CUBIN, "rb").read() in blob


def test_is_wide_is_exported():
    header = open(os.path.join(capi.INCLUDE, "pmdi_cuda.h")).read()
    assert re.search(r"int pmdi_ctx_is_wide\(const pmdi_ctx\* ctx, int32_t\* wide\);", header)
    assert "pmdi_ctx_is_wide" in capi.EXPORTS
    assert hasattr(capi.lib(), "pmdi_ctx_is_wide")
    assert capi.lib().pmdi_ctx_is_wide(None, None) == 1
