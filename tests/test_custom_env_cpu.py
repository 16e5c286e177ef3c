"""Custom env plug-in (SURVEY 8 row f4), host side: a user's CUDA-C env file is compiled for
sm_100a with the reference's three compile-time constants and exposes its extern "C"
kernels by name.  Compilation needs nvcc only (no GPU); launching is in
tests/test_gpu_custom_env.py."""
import os
import re
import subprocess

import pytest

from warp_drive_b200.utils import custom_kernels as ck
from warp_drive_b200.utils.env_registrar import EnvironmentRegistrar

HERE = os.path.dirname(os.path.abspath(__file__))
COUNTER_CU = os.path.join(HERE, "custom_env", "counter_env_step.cu")


def test_compile_user_env_file_for_sm100a(tmp_path, monkeypatch):
    monkeypatch.setenv("WDB_KERNEL_CACHE", str(tmp_path))
    cubin = ck.compile_module(COUNTER_CU, n_envs=8, n_agents=5, blocks_per_env=1)
    assert ck.kernel_names(cubin) == ["CudaCounterEnvReset", "CudaCounterEnvStep"]
    elf = subprocess.run(["cuobjdump", "--list-elf", cubin], capture_output=True, text=True).stdout
    assert set(re.findall(r"sm_\d+a?", elf)) == {"sm_100a"}
    # cached by content + shape: same inputs -> same file, new shape -> new file
    assert ck.compile_module(COUNTER_CU, 8, 5, 1) == cubin
    assert ck.compile_module(COUNTER_CU, 16, 5, 1) != cubin


def test_compile_from_source_text_and_nvcc_errors_surface(tmp_path, monkeypatch):
    monkeypatch.setenv("WDB_KERNEL_CACHE", str(tmp_path))
    code = 'extern "C" __global__ void CudaTinyStep(float *x) {\n' \
           '  x[wdb_env::agent_index()] += wkNumberEnvs; }\n'
    assert ck.kernel_names(ck.compile_module(code, 4, 3)) == ["CudaTinyStep"]
    with pytest.raises(RuntimeError, match="nvcc failed"):
        ck.compile_module('extern "C" __global__ void Broken(float *x) { x[0] = y; }\n', 4, 3)
    with pytest.raises(FileNotFoundError):
        ck.compile_module(str(tmp_path / "missing.cu"), 4, 3)


def test_registrar_keeps_custom_source_paths():
    reg = EnvironmentRegistrar()
    assert reg.get_cuda_env_src_path("CounterEnv") is None
    reg.add_cuda_env_src_path("CounterEnv", COUNTER_CU)
    assert reg.get_cuda_env_src_path("counterenv") == COUNTER_CU
    with pytest.raises(AssertionError):
        reg.add_cuda_env_src_path("Bad", "/tmp/not_cuda.py")


def test_marshal_follows_pycuda_rules():
    import ctypes

    import numpy as np

    assert isinstance(ck.marshal(np.int32(3)), ctypes.c_int)
    assert isinstance(ck.marshal(np.float32(3)), ctypes.c_float)
    assert isinstance(ck.marshal(True), ctypes.c_bool)
    assert isinstance(ck.marshal(np.float64(1)), ctypes.c_double)
    import torch

    with pytest.raises(RuntimeError, match="CUDA tensors"):
        ck.marshal(torch.zeros(2))
    with pytest.raises(TypeError):
        ck.marshal("x")
