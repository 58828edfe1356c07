"""The C-ABI library loads on a CPU-only box, exports every symbol include/tcmcmc.h declares, its
structs have the layout the Python binding assumes, and compute entry points fail loudly (no CPU
fallback) when there is no CUDA device."""
import ctypes as C
import os
import re
import subprocess

import numpy as np
import pytest

from conftest import ROOT
from transcriptioncycleinference_b200 import _lib, constructs

HEADER = os.path.join(ROOT, "include", "tcmcmc.h")


def _declared_functions():
    src = open(HEADER).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(tc_[a-z0-9_]+)\s*\(", src)))


def test_every_declared_symbol_is_exported():
    L = _lib.load()
    names = _declared_functions()
    assert len(names) >= 14
    for n in names:
        assert hasattr(L, n), "libtcmcmc.so does not export %s" % n
    assert sorted(_lib.EXPORTS) == names


def test_version_and_defaults():
    L = _lib.load()
    assert L.tc_version() == 100
    o = _lib.default_opts()
    # mcmcstat defaults + the reference's configuration (TranscriptionCycleMCMC.m:263-270)
    assert (o.nsimu, o.burnintime, o.adaptint, o.ntry, o.updatesigma) == (20000, 10000, 100, 2, 1)
    assert (o.drscale, o.qcovadj, o.burnin_scale, o.N0, o.S20, o.sigma2_0) == (5.0, 1e-8, 10.0, 1.0, 1.0, 1.0)
    assert o.adascale == 0.0 and o.n_burn == 10000 and o.store_chain == 0 and o.algo == _lib.ALGO_TOEPLITZ
    assert o.layout == 0                      # TC_LAYOUT_AUTO: the large-series layout only when the regular one does not fit


def test_struct_layouts_match_header(tmp_path):
    """sizeof/offsetof and the TC_EINVAL / TC_LAYOUT_* values from a C compile of the header == the ctypes mirror."""
    src = tmp_path / "sz.c"
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "tcmcmc.h"\nint main(){printf("%zu %zu %zu %zu %zu %zu %zu %d\\n",'
                   'sizeof(tc_construct),sizeof(tc_mcmc_opts),sizeof(tc_replay),sizeof(tc_device_info),'
                   'offsetof(tc_mcmc_opts,drscale),offsetof(tc_mcmc_opts,seed),offsetof(tc_construct,pp7_loopn),TC_NCOUNTERS);'
                   'printf("%d %d %d %d %d\\n",TC_EINVAL,TC_LAYOUT_AUTO,TC_LAYOUT_BIG,TC_LAYOUT_WARP,TC_LAYOUT_CTA);return 0;}\n')
    exe = tmp_path / "sz"
    subprocess.check_call(["/usr/bin/gcc" if os.path.exists("/usr/bin/gcc") else "gcc", "-I", os.path.join(ROOT, "include"),
                           "-o", str(exe), str(src)])
    vals = [int(x) for x in subprocess.check_output([str(exe)]).split()]
    assert vals[0] == C.sizeof(_lib.Construct)
    assert vals[1] == C.sizeof(_lib.McmcOpts)
    assert vals[2] == C.sizeof(_lib.Replay)
    assert vals[3] == C.sizeof(_lib.DeviceInfo)
    assert vals[4] == _lib.McmcOpts.drscale.offset and vals[5] == _lib.McmcOpts.seed.offset
    assert vals[6] == _lib.Construct.pp7_loopn.offset
    assert vals[7] == _lib.NCOUNTERS
    assert vals[8:] == [_lib.TC_EINVAL, _lib.LAYOUT_AUTO, _lib.LAYOUT_BIG, _lib.LAYOUT_WARP, _lib.LAYOUT_CTA]


def test_no_cpu_fallback_without_device(cells_npz):
    """On a box without a GPU the product path must fail loudly, not compute on the CPU."""
    if _lib.device_count() > 0:
        pytest.skip("a CUDA device is present")
    from transcriptioncycleinference_b200.engine import Cells
    with pytest.raises(_lib.TcError) as e:
        Cells.from_packed(cells_npz["N"][:2], cells_npz["off"][:3], cells_npz["t"], cells_npz["ms2"], cells_npz["pp7"])
    assert e.value.code == -2 and "no CPU fallback" in str(e.value)
    with pytest.raises(_lib.TcError):
        _lib.measure_fp64_peak(0)
    from transcriptioncycleinference_b200 import mcmc
    with pytest.raises(RuntimeError):
        mcmc.TranscriptionCycleMCMC("fileDir", "/nonexistent")


def test_product_does_not_import_oracle():
    """oracle/ is test infrastructure: nothing under the product package may reference it."""
    pkg = os.path.join(ROOT, "transcriptioncycleinference_b200")
    for dp, _, fs in os.walk(pkg):
        for f in fs:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                txt = open(os.path.join(dp, f)).read()
                assert not re.search(r"^\s*(from|import)\s+oracle\b", txt, flags=re.M), f
                assert "tc_oracle" not in txt and "libtcoracle" not in txt, f


def test_construct_validation_messages():
    c = constructs.to_c("P2P-MS2v5-LacZ-PP7v4")
    assert c.nsets == 1 and abs(c.ms2_end[0] - 1.299) < 1e-15
