"""Staged host path of a strict FP32 handle with many re-solved envs.  The FP64 re-solve's results come back to the host as
compact records; the first 160 are copied with every step and the rest only when more envs were re-solved.  That second
copy and the scatter of its records must give the device-resident step's results bit for bit."""
import numpy as np
import pytest

from tests._util import layout

pytestmark = pytest.mark.gpu

EAGER_RECORDS = 160  # records copied with every step (wf_api.cu: step_host_impl)


def test_staged_host_step_with_many_resolved_envs(cuda_device, monkeypatch):
    import torch

    from wfcrl_b200.backend import FlorisBatch

    lx, ly = layout("Turb32_Row5_")
    B, T = 1024, len(lx)
    rng = np.random.default_rng(7)
    # Rotor speeds just above cut-in (2.5 m/s), where the power curve rises steeply from 0: the FP32 kernel hands such
    # envs to the FP64 re-solve.  A quarter of the envs get ordinary winds and stay with FP32.
    ws = rng.uniform(2.6, 2.8, B)
    ws[::4] = np.clip(8 * rng.weibull(8, B // 4), 3, 28)
    wd = np.clip(rng.normal(270, 20, B) % 360, 0, 360)
    dev, host = (FlorisBatch(lx, ly, B, precision="f32", kernel="fast", max_iter=100) for _ in range(2))
    for fb in (dev, host):
        fb.reset(ws, wd, host_trig=True)
    monkeypatch.setenv("WFCRL_B200_HOST_PATH", "staged")
    for k in range(3):
        a = rng.uniform(-2, 2, (B, T)).astype(np.float32)
        want = dev.step(torch.as_tensor(a, device="cuda"))
        got = host.step_host(torch.as_tensor(a))
        torch.cuda.synchronize()
        resolved = host.get_state("ambiguous")
        assert int(resolved.sum()) > EAGER_RECORDS, (k, int(resolved.sum()))
        assert np.array_equal(resolved, dev.get_state("ambiguous")), k
        for key, v in want.items():
            assert torch.equal(v.cpu(), got[key]), (k, key)
    dev.close()
    host.close()
