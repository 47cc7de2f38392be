"""All GPUs of one box behind one C ABI (include/ismpc_b200_multigpu.h, host/MPCSolverMultiGpu.hpp): the library loads
and exports what its header declares, the C++ face compiles with plain g++, shards are the contiguous ranges of SURVEY
8(e), and on the GPU a group gives bit for bit what one handle gives -- tick by tick through host buffers, and as a
resident closed loop with the final gather (NCCL all-gather when the box has two or more GPUs, host copies otherwise)."""
import ctypes as C
import os
import re
import subprocess
import tempfile

import numpy as np
import pytest

from quadruped_gait_generation_ismpc_b200 import abi, binding, sharding, synth

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "ismpc_b200_multigpu.h")


def test_multigpu_library_exports_every_declared_symbol():
    declared = set(re.findall(r"\b(ismpc_group_[a-z_0-9]+)\s*\(", open(HEADER).read()))
    assert declared == set(binding.MG_EXPORTS)
    L = binding.mglib()
    for s in declared:
        assert hasattr(L, s), "missing export %s" % s
    needed = subprocess.check_output(["readelf", "-d", binding.MG_LIB_PATH], text=True)
    libs = re.findall(r"NEEDED.*\[(.*?)\]", needed)
    assert "libismpc_b200.so" in libs and any(x.startswith("libnccl") for x in libs), libs


def test_group_shards_are_the_contiguous_ranges_of_the_survey():
    """ismpc_group_shard == sharding.shard_range (what bench.py --gpus N and the gloo tests use); no GPU needed: the
    arithmetic is exported as a free function of (n_total, group size, rank) -- checked through a C driver."""
    src = r'''
#include <stdio.h>
#include "ismpc_b200_multigpu.h"
int main(void) { return ismpc_group_shard(0, 10, 0, 0, 0) == ISMPC_ERR_ARG ? 0 : 1; }
'''
    with tempfile.TemporaryDirectory() as d:
        open(os.path.join(d, "t.c"), "w").write(src)
        libdir = os.path.dirname(binding.LIB_PATH)
        subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), os.path.join(d, "t.c"), "-o", os.path.join(d, "t"),
                               "-L" + libdir, "-lismpc_b200_mg", "-lismpc_b200", "-Wl,-rpath," + libdir])
        assert subprocess.run([os.path.join(d, "t")]).returncode == 0      # NULL group is refused, nothing dereferenced
    for n, G in ((1024, 8), (1000, 8), (7, 8), (65536, 8), (5, 2)):
        cover = []
        for r in range(G):
            lo, hi = sharding.shard_range(n, r, G)
            cover += list(range(lo, hi))
        assert cover == list(range(n))


def _build_example(d):
    exe = os.path.join(d, "multigpu_example")
    libdir = os.path.dirname(binding.LIB_PATH)
    subprocess.check_call(["g++", "-std=c++17", "-Wall", "-Wextra", "-Werror", "-O1", "-o", exe,
                           os.path.join(ROOT, "tests", "cpp", "multigpu_example.cpp"),
                           "-L" + libdir, "-lismpc_b200_mg", "-lismpc_b200", "-Wl,-rpath," + libdir])
    return exe


def test_multigpu_example_compiles_with_plain_gpp_and_fails_loudly_without_gpu():
    import torch
    with tempfile.TemporaryDirectory() as d:
        exe = _build_example(d)
        if torch.cuda.is_available():
            pytest.skip("GPU present")
        r = subprocess.run([exe, "8", "3", "host", "0"], capture_output=True, text=True)
        assert r.returncode == 2 and "ismpc_group_create" in r.stderr
    with pytest.raises(binding.IsmpcError):
        binding.Group([0], 8, binding.GATHER_HOST)


def _devices():
    import torch
    return list(range(torch.cuda.device_count()))


@pytest.mark.gpu
@pytest.mark.parametrize("layout", ["one", "two_shards_host_gather", "all_gpus_nccl"])
def test_group_equals_single_handle(handle, layout):
    """Tick through host buffers and resident closed loop (scatter / rollout with pushes / gather) == one handle."""
    devs = _devices()
    if layout == "one":
        devices, mode = [0], binding.GATHER_NCCL
    elif layout == "two_shards_host_gather":
        devices, mode = [0, 0, 0], binding.GATHER_HOST          # three shards on one device: the sharding logic without NCCL
    else:
        if len(devs) < 2:
            pytest.skip("needs two GPUs")
        devices, mode = devs, binding.GATHER_NCCL
    model = abi.formc_model()
    n = 203                                                     # not a multiple of the group size
    state, walk, inst, plan = synth.formc_batch(n, seed=71, k0_cap=300)
    push = synth.push_batch(n, seed=72, formc=True)
    push["ct0"] = 10; push["ct1"] = 24
    handle.formc_set_model(model); handle.formc_prepare_gait(35, 10)
    ref = handle.formc_solve_batch(state, walk, inst, plan, want_primal=False, want_active=False)
    ref_roll = handle.formc_rollout(state, walk, inst, plan, 60, push=push, want_traj=False)
    g = binding.Group(devices, (n + len(devices) - 1) // len(devices), mode)
    try:
        g.formc_configure(model, 35, 10, plan)
        out = g.formc_solve_batch(state, walk, inst)
        assert out.tobytes() == ref["out"].tobytes()
        # packed tick records, constants resident per shard: pageable buffers (staged) and pinned ones (in place)
        g.formc_set_instances(inst)
        tick = abi.pack_ticks(state, walk)
        assert g.formc_solve_batch_packed(tick).tobytes() == ref["out"].tobytes()
        t_pin = binding.PinnedBuffer(tick.nbytes, fill=tick); o_pin = binding.PinnedBuffer(n * abi.FORMC_OUT.itemsize)
        try:
            g.formc_solve_batch_packed_raw(n, t_pin.ptr, o_pin.ptr)
            assert o_pin.array.tobytes() == ref["out"].tobytes()
        finally:
            t_pin.close(); o_pin.close()
        g.formc_scatter(state, walk, inst, push)
        g.formc_rollout(25); g.formc_rollout(35)               # two calls: the pushes belong to the first
        r = g.formc_gather()
        assert r["state"].tobytes() == ref_roll["state"].tobytes()
        assert r["walk"].tobytes() == ref_roll["walk"].tobytes()
        assert np.array_equal(r["status"], ref_roll["status"])
        cover = []
        for k in range(len(devices)):
            a, c = g.shard(n, k)
            assert (a, a + c) == sharding.shard_range(n, k, len(devices))
            cover += list(range(a, a + c))
        assert cover == list(range(n))
        assert g.kernel_launches > 0
    finally:
        g.close()


@pytest.mark.gpu
def test_multigpu_example_runs():
    """host/MPCSolverMultiGpu.hpp from plain C++: the tick-by-tick loop through host buffers and the resident closed loop
    end at the same CoM (the same ticks, 1e-12), on every GPU of the box (NCCL gather with two or more, host otherwise)."""
    devs = _devices()
    with tempfile.TemporaryDirectory() as d:
        exe = _build_example(d)
        args = [exe, "37", "40"] + (["nccl"] + [str(x) for x in devs] if len(devs) >= 2 else ["host", "0", "0"])
        out = subprocess.check_output(args, text=True, env=dict(os.environ, NCCL_DEBUG="WARN"))
    rows = np.array([[float(x) for x in ln.split()] for ln in out.strip().splitlines() if ln[:1].isdigit()])   # (NCCL may print a banner)
    # (status 16 = ISMPC_ST_XY_SKIPPED on flight-phase ticks -- lambda_0 = 0, MPCSolver.cpp:322 -- is not a failure)
    assert rows.shape == (37, 8) and ((rows[:, 7].astype(int) & abi.ST_FAIL_MASK) == 0).all()
    assert np.abs(rows[:, 1:4] - rows[:, 4:7]).max() <= 1e-12
    # (sanity of the run itself: the CoM moved forward and stayed near its target height -- the gait has a flight phase of
    # F_ds = 10 samples with f = 0, MPCSolver.cpp:223-243, during which the CoM falls by up to g (0.1 s)^2 / 2 = 4.9 cm)
    assert np.abs(rows[:, 3] - 0.69).max() < 6e-2 and rows[:, 1].max() > 0.0
