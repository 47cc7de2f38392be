"""SASS goldens of kernels that must not change: compile a source of the library with its flags, read each kernel's SASS
with cuobjdump, hash it, and compare against a golden file only when the nvcc is the one the file was recorded with
(another nvcc may schedule differently)."""
import hashlib
import json
import os
import re
import shutil
import subprocess

import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(os.path.dirname(HERE), "quadruped_gait_generation_ismpc_b200", "csrc")
FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17", "-Xcompiler", "-fPIC", "--fmad=true"]


def _nvcc():
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(nvcc):
        pytest.skip("no nvcc")
    return nvcc


def compile_sass(source, tmp_path, extra=()):
    """Compiles csrc/<source> with the library's flags (plus extra).  Returns ({kernel symbol: SASS lines}, nvcc's
    stderr)."""
    nvcc = _nvcc()
    obj = str(tmp_path / (os.path.splitext(source)[0] + ".o"))
    r = subprocess.run([nvcc, *FLAGS, *extra, "-c", os.path.join(CSRC, source), "-o", obj], capture_output=True,
                       text=True, check=True)
    out = subprocess.run([os.path.join(os.path.dirname(nvcc), "cuobjdump"), "-sass", obj], capture_output=True, text=True,
                         check=True).stdout
    funcs, cur = {}, None
    for line in out.splitlines():
        m = re.match(r"\s*Function : (\S+)", line)
        if m:
            cur = m.group(1); funcs[cur] = []
        elif cur and line.strip() and not line.strip().startswith("."):
            funcs[cur].append(line.strip())
    return funcs, r.stderr


def digest(lines):
    return hashlib.sha256("\n".join(lines).encode()).hexdigest()


def golden(name):
    """tests/golden/<name>: {"nvcc": version, "kernels": {name: digest}}."""
    return json.load(open(os.path.join(HERE, "golden", name)))


def skip_unless_recorded_nvcc(gold):
    version = re.search(r"release \S+, V(\S+)", subprocess.run([_nvcc(), "--version"], capture_output=True,
                                                                text=True).stdout).group(1)
    if version != gold["nvcc"]:
        pytest.skip("SASS recorded with nvcc %s, this is %s" % (gold["nvcc"], version))
