"""include/dronenav.h is a C header and libdronenav.so a C library: a plain C99 program (tests/c_abi/demo.c, gcc -std=c99
-pedantic -Werror, no CUDA headers, no C++) loads it, resolves every entry point, and -- on a GPU -- steps environments
through dn_step_host with malloc'ed host buffers; the per-step sums it prints are checked against the batched oracle."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from tests.conftest import ROOT

SRC = os.path.join(ROOT, "tests", "c_abi", "demo.c")


@pytest.fixture(scope="module")
def demo(built_lib, tmp_path_factory):
    # compiled outside the repository tree, which may be read-only where the suite runs
    exe = str(tmp_path_factory.mktemp("c_abi") / "demo")
    subprocess.run(["gcc", "-std=c99", "-pedantic", "-Wall", "-Wextra", "-Werror", "-O1", "-I", os.path.join(ROOT, "include"),
                    "-o", exe, SRC, "-ldl", "-lm"], check=True)
    from drl_dronenavigation_b200 import _lib
    return exe, _lib.LIB_PATH


def test_header_compiles_as_c99_and_every_symbol_resolves(demo):
    exe, lib = demo
    from drl_dronenavigation_b200 import _lib
    out = subprocess.run([exe, lib, "symbols"], check=True, capture_output=True, text=True).stdout.split()
    sizes = dict(zip(out[2::2], out[3::2]))
    assert int(out[1]) == _lib.DN_ABI_VERSION
    # the C compiler's struct sizes are the ones the ctypes mirror uses
    assert int(sizes["sizeof(dn_config)"]) == C.sizeof(_lib.dn_config)
    assert int(sizes["sizeof(dn_step_io)"]) == C.sizeof(_lib.dn_step_io)
    assert int(sizes["sizeof(dn_state_view)"]) == C.sizeof(_lib.dn_state_view)
    assert int(sizes["sizeof(dn_stats)"]) == C.sizeof(_lib.dn_stats)


@pytest.mark.gpu
def test_plain_c_host_steps_environments_through_dn_step_host(demo):
    from oracle.batched_oracle import BatchedOracle
    exe, lib = demo
    # 64 envs x 30 control steps with LCG seed 31: every discrete decision of this run keeps a margin of > 1e-3 to its threshold
    # in the oracle (50x the FP32 drift), so the open-loop comparison cannot be upset by an FP32 / FP64 near-tie
    N, T, seed = 64, 30, 31
    lines = subprocess.run([exe, lib, "step", str(N), str(T), str(seed)], check=True, capture_output=True, text=True).stdout.strip().split("\n")
    assert len(lines) == T + 1 and lines[-1].startswith("episodes")
    B = BatchedOracle(N, "circle", pyb_freq=240, ctrl_freq=30)
    lcg = seed
    total_done = 0
    for t in range(T):
        a = np.empty(4 * N, np.float32)
        for i in range(4 * N):
            lcg = (1103515245 * lcg + 12345) & 0x7fffffff
            a[i] = np.float32(0.092227 + 0.004 * (lcg / 1073741824.0 - 1.0))
        obs, rew, bits, found, *_ = B.step(a.reshape(N, 4))
        tt, rsum, dsum, fsum, osum = lines[t].split()
        assert int(tt) == t
        assert B.margin.min() > 1e-3 and min(B.rew_margin.min(), B.gimbal_margin.min()) > 5e-4
        assert int(dsum) == int((bits != 0).sum()) and int(fsum) == int(found.sum())
        assert abs(float(rsum) - float(rew.sum())) < 1e-3 * N
        assert abs(float(osum) - float(obs.astype(np.float64).sum())) < 1e-3 * N
        total_done += int((bits != 0).sum())
    assert total_done > 100 and int(lines[-1].split()[1]) == total_done and int(lines[-1].split()[5]) >= T
