"""CPU tests: the C-ABI library loads and exports every symbol include/wfcrl_b200.h declares; no compute without a GPU."""
import ctypes as C
import os
import re
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _declared_symbols():
    text = open(os.path.join(ROOT, "include", "wfcrl_b200.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(wf_[a-z_0-9]+)\s*\(", text)))


def test_header_and_binding_agree():
    from wfcrl_b200 import _lib

    declared = _declared_symbols()
    assert len(declared) >= 14
    assert sorted(_lib.SYMBOLS.keys()) == declared


def test_library_exports_every_declared_symbol():
    from wfcrl_b200 import _lib

    lib = _lib.load()
    for name in _declared_symbols():
        assert hasattr(lib, name), name
    assert b"sm_100a" in lib.wf_version()


def test_default_config_matches_reference_case_yaml():
    """wf_default_config needs no GPU: values of case.yaml:30-39,52-60,84-89 and the env defaults."""
    from wfcrl_b200 import _lib

    lib = _lib.load()
    cfg = _lib.WfConfig()
    assert lib.wf_default_config(C.byref(cfg)) == 0
    assert (cfg.air_density, cfg.turbulence_intensity, cfg.wind_shear, cfg.wind_veer) == (1.225, 0.06, 0.12, 0.0)
    assert (cfg.alpha, cfg.beta, cfg.ka, cfg.kb, cfg.ad, cfg.bd, cfg.dm) == (0.58, 0.077, 0.38, 0.004, 0.0, 0.0, 1.0)
    assert (cfg.ch_initial, cfg.ch_constant, cfg.ch_ai, cfg.ch_downstream) == (0.1, 0.5, 0.8, -0.32)
    assert (cfg.yaw_lo, cfg.yaw_hi, cfg.yaw_step, cfg.load_coef, cfg.dt, cfg.actuator_rate) == (-40, 40, 5, 0.1, 60, 0.3)
    assert (cfg.rotor_diameter, cfg.hub_height, cfg.tsr, cfg.pP) == (126.0, 90.0, 8.0, 1.88)
    assert cfg.table_len == 51
    from oracle.floris_oracle import turbine_tables
    ws, ct, _pw = turbine_tables()
    assert np.array_equal(np.array(cfg.table_ws[:51]), ws) and np.array_equal(np.array(cfg.table_ct[:51]), ct)


def test_no_cpu_fallback():
    """Without a CUDA device the product must fail loudly, never compute on the CPU."""
    import torch

    if torch.cuda.is_available():
        pytest.skip("CUDA device present")
    from wfcrl_b200 import _lib
    from wfcrl_b200.backend import FlorisBatch

    with pytest.raises(_lib.WfError):
        FlorisBatch([0.0, 500.0], [0.0, 0.0], 2)
    lib = _lib.load()
    cfg = _lib.WfConfig()
    lib.wf_default_config(C.byref(cfg))
    cfg.num_turbines, cfg.num_envs, cfg.max_iter = 2, 1, 10
    lx = np.array([0.0, 500.0])
    handle = C.c_void_p()
    rc = lib.wf_create(C.byref(cfg), lx.ctypes.data_as(C.c_void_p), lx.ctypes.data_as(C.c_void_p), C.byref(handle))
    assert rc == 2 and b"no CPU fallback" in lib.wf_last_error()  # WF_ERR_CUDA


def test_invalid_arguments_are_reported_not_thrown():
    from wfcrl_b200 import _lib

    lib = _lib.load()
    assert lib.wf_default_config(None) == 1
    cfg = _lib.WfConfig()
    lib.wf_default_config(C.byref(cfg))
    cfg.num_turbines, cfg.num_envs = 500, 1
    lx = np.zeros(500)
    handle = C.c_void_p()
    assert lib.wf_create(C.byref(cfg), lx.ctypes.data_as(C.c_void_p), lx.ctypes.data_as(C.c_void_p),
                         C.byref(handle)) == 1
    assert b"num_turbines" in lib.wf_last_error()
    ptr = lambda a: a.ctypes.data_as(C.c_void_p)  # noqa: E731
    cfg.num_turbines = 3
    bad = np.array([0.0, np.nan, 500.0])
    assert lib.wf_create(C.byref(cfg), ptr(bad), ptr(np.zeros(3)), C.byref(handle)) == 1
    assert b"layout" in lib.wf_last_error()
    cfg.kernel = 7
    assert lib.wf_create(C.byref(cfg), ptr(np.zeros(3)), ptr(np.zeros(3)), C.byref(handle)) == 1
    assert b"kernel" in lib.wf_last_error()
    lib.wf_default_config(C.byref(cfg))
    cfg.num_turbines, cfg.num_envs = 3, 1
    cfg.table_ws[5] = cfg.table_ws[4]
    assert lib.wf_create(C.byref(cfg), ptr(np.zeros(3)), ptr(np.zeros(3)), C.byref(handle)) == 1
    assert b"strictly increasing" in lib.wf_last_error()
    lib.wf_default_config(C.byref(cfg))
    cfg.num_turbines, cfg.num_envs, cfg.hub_height = 3, 1, 50.0
    assert lib.wf_create(C.byref(cfg), ptr(np.zeros(3)), ptr(np.zeros(3)), C.byref(handle)) == 1
    assert b"hub_height" in lib.wf_last_error()


def test_product_never_imports_the_oracle():
    """The oracle is test infrastructure: nothing under wfcrl_b200/ may import it."""
    pkg = os.path.join(ROOT, "wfcrl_b200")
    for dirpath, _dirs, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                text = open(os.path.join(dirpath, f)).read()
                assert "import oracle" not in text and "from oracle" not in text, f
                assert "floris_oracle" not in text and "env_oracle" not in text, f


def test_version_string_carries_the_hash_of_the_sources():
    """wf_version() names the sources the binary was built from; build() rebuilds on any difference (no GPU needed)."""
    from wfcrl_b200 import _lib, build

    assert build.library_hash() == build.source_hash()
    version = _lib.load().wf_version().decode()
    assert version.startswith("wfcrl_b200 ") and version.endswith("wfcrl_b200-src-sha256:" + build.source_hash())
    assert _lib.binary_matches_source()


def test_compiled_code_is_a_function_of_the_sources(monkeypatch, tmp_path):
    """The source hash stands for the binary: the sources select no code by a macro from outside (their only conditional
    is on the hash itself), and no environment variable the package reads changes the nvcc command."""
    from wfcrl_b200 import build

    for f in sorted(os.listdir(build.CSRC)):
        if f.endswith((".cu", ".cuh", ".h")):
            for line in open(os.path.join(build.CSRC, f)):
                if re.match(r"\s*#\s*(if|elif)", line):
                    assert "WF_SOURCE_HASH" in line, (f, line)

    names = set()
    for dirpath, _dirs, files in os.walk(os.path.join(ROOT, "wfcrl_b200")):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                names.update(re.findall(r"\bWFCRL_[A-Z0-9_]*[A-Z0-9]\b", open(os.path.join(dirpath, f)).read()))
    names.update({"WFCRL_NVCC_FLAGS", "WFCRL_DEBUG"})

    src_hash = build.source_hash()
    # every file the build writes goes to tmp_path (source_hash() would follow HERE there)
    monkeypatch.setattr(build, "source_hash", lambda: src_hash)
    monkeypatch.setattr(build, "HERE", str(tmp_path))
    monkeypatch.setattr(build, "BAKED", str(tmp_path / "wf_fast_baked.inc"))
    monkeypatch.setattr(build, "LIB", str(tmp_path / "libwfcrl_b200.so"))
    monkeypatch.setattr(build, "_nvcc", lambda: "nvcc")
    calls = []

    def run(cmd, **_kw):
        calls.append(list(cmd))
        if "-o" in cmd:
            open(cmd[cmd.index("-o") + 1], "w").close()
        return subprocess.CompletedProcess(cmd, 0, stdout="", stderr="")

    monkeypatch.setattr(subprocess, "run", run)

    def library_command(env):
        for k in [k for k in os.environ if k.startswith("WFCRL_")]:
            monkeypatch.delenv(k)
        for k, v in env.items():
            monkeypatch.setenv(k, v)
        calls.clear()
        build.build_library(force=True)
        return calls[-1]

    plain = library_command({})
    assert plain[-len(build.SOURCES):] == [os.path.join(build.CSRC, s) for s in build.SOURCES]
    assert f'-DWF_SOURCE_HASH="{src_hash}"' in plain
    assert library_command({k: "-DWF_OUTSIDE_SWITCH=1 -O0" for k in names}) == plain
