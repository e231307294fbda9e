"""Layout pools of mixed turbine counts (wf_set_layouts_sized): one handle of T = 80 turbines whose envs run farms of 1, 7,
32 and 80 turbines.  Every env must compute, bit for bit, what a handle created with its farm alone computes, in its first
n columns; its padding columns must read exactly 0, in the outputs and in the yaw / accumulator state."""
import ctypes as C

import numpy as np
import pytest

from tests._util import layout, sample_winds

pytestmark = pytest.mark.gpu

POOL = ["Turb1_Row1_", "Ablaincourt_", "Turb32_Row5_", "HornsRev1_"]
COUNTS = [1, 7, 32, 80]
T = 80
PER_TURBINE = ("yaw", "wind_speed", "wind_direction", "power", "load")
PER_ENV = ("reward", "freewind", "truncated")
# (precision, strict, interface mode, vortex table)
MODES = {
    "f64_fast_table": ("f64", True, False, True),
    "f64_fast_direct": ("f64", True, False, False),
    "f32_strict": ("f32", True, False, True),
    "f32_relaxed": ("f32", False, False, True),
    "interface": ("f64", True, True, True),
}


@pytest.fixture(scope="module")
def farms():
    return [layout(n) for n in POOL]


def make_mixed(farms, B, **kw):
    from wfcrl_b200.backend import FlorisBatch

    fb = FlorisBatch(*farms[-1], B, **kw)
    fb.set_mixed_layouts([f[0] for f in farms], [f[1] for f in farms])
    return fb


def assert_rows_equal(pool_out, ref_out, rows, n, where):
    """Env rows `rows` of the pool against the same rows of a single-layout handle of n turbines; padding is 0."""
    import torch

    trows = torch.as_tensor(rows, device="cuda")
    for key in PER_TURBINE:
        p = pool_out[key][trows]
        assert torch.equal(p[:, :n], ref_out[key][trows]), (where, key)
        assert not bool(p[:, n:].any()), (where, key, "padding")
    for key in PER_ENV:
        assert torch.equal(pool_out[key][trows], ref_out[key][trows]), (where, key)


def assert_state_equal(pool, ref, rows, n, where, names=("xs", "ys", "order", "ambiguous")):
    for name in names:
        p, r = pool.get_state(name)[rows], ref.get_state(name)[rows]
        if p.ndim == 2:
            p = p[:, :n]
        assert np.array_equal(p, r), (where, name)


def assert_padding_state_zero(fb, counts):
    for name in ("yaw", "acc", "acc_prev"):
        v = fb.get_state(name)
        for b, n in enumerate(counts):
            assert not v[b, n:].any(), (name, b, n)


@pytest.mark.parametrize("mode", list(MODES))
def test_mixed_pool_equals_single_layout_handles(cuda_device, monkeypatch, farms, mode):
    import torch

    from wfcrl_b200.backend import FlorisBatch

    precision, strict, interface, table = MODES[mode]
    if table:
        monkeypatch.delenv("WFCRL_B200_NO_VTAB", raising=False)
    else:
        monkeypatch.setenv("WFCRL_B200_NO_VTAB", "1")
    B = 1024 if mode == "f32_strict" else 256  # enough envs for the guard band to flag some
    kw = dict(precision=precision, kernel="fast", max_iter=50, strict=strict, reward_shaper="step")
    pool = make_mixed(farms, B, **kw)
    refs = [FlorisBatch(lx, ly, B, **kw) for lx, ly in farms]
    ids = np.arange(B) % len(farms)
    pool.assign_layouts(None, ids)
    counts = np.array(COUNTS)[ids]
    assert np.array_equal(pool.get_state("turbine_count"), counts)
    ws, wd = sample_winds(B, seed=5)
    for fb in [pool] + refs:
        fb.reset(ws, wd, host_trig=True)
    rng = np.random.default_rng(11)
    flagged = np.zeros(len(farms), dtype=int)
    for k in range(4):
        if interface:
            cmd = rng.uniform(-20, 20, (B, T))  # commands in padding columns are ignored
            outs = [pool.update_command(torch.as_tensor(cmd, device="cuda"))]
            outs += [fb.update_command(torch.as_tensor(np.ascontiguousarray(cmd[:, :n]), device="cuda"))
                     for fb, n in zip(refs, COUNTS)]
        else:
            act = rng.uniform(-5, 5, (B, T)).astype(np.float32)  # actions in padding columns are ignored
            outs = [pool.step(torch.as_tensor(act, device="cuda"))]
            outs += [fb.step(torch.as_tensor(np.ascontiguousarray(act[:, :n]), device="cuda"))
                     for fb, n in zip(refs, COUNTS)]
        torch.cuda.synchronize()
        amb = pool.get_state("ambiguous")
        for lay, n in enumerate(COUNTS):
            rows = ids == lay
            flagged[lay] += int(amb[rows].sum())
            assert_rows_equal(outs[0], outs[1 + lay], rows, n, (k, lay))
            assert_state_equal(pool, refs[lay], rows, n, (k, lay))
        assert_padding_state_zero(pool, counts)
    xs, order = pool.get_state("xs"), pool.get_state("order")
    for b, n in enumerate(counts):
        assert not xs[b, n:].any() and np.array_equal(order[b, n:], np.arange(n, T))
    if mode == "f32_strict":
        # the FP64 re-solve ran for pool envs of the 7-, 32- and 80-turbine farms: W = 8 warps per env in the pool
        # against W = 1, 4 and 8 in the single-layout handles
        assert (flagged[1:] > 0).all(), flagged
    for fb in [pool] + refs:
        fb.close()


@pytest.mark.parametrize("precision", ["f32", "f64"])
def test_autoreset_with_layout_sampling_equals_fresh_handles(cuda_device, farms, precision):
    import torch

    from wfcrl_b200.backend import FlorisBatch

    B, L_ep = 256, 4
    kw = dict(precision=precision, kernel="fast", max_iter=L_ep)
    pool = make_mixed(farms, B, **kw)
    pool.assign_layouts(None, 3)  # every env starts on the 80-turbine farm
    ws, wd = sample_winds(B, seed=3)
    pool.reset(ws, wd, host_trig=False)
    pool.set_layout_sampling(True)
    pool.set_autoreset(True, seed=41, env_id_offset=0)
    rng = np.random.default_rng(2)
    act = lambda: torch.as_tensor(rng.uniform(-5, 5, (B, T)).astype(np.float32), device="cuda")  # noqa: E731
    while not bool(pool.step(act())["truncated"].any()):
        pass
    pool.autoreset_finish()
    torch.cuda.synchronize()
    ids = pool.get_state("layout_id")
    assert set(ids.tolist()) == {0, 1, 2, 3}  # envs moved from 80 turbines to every other count
    counts = np.array(COUNTS)[ids]
    assert np.array_equal(pool.get_state("turbine_count"), counts)
    assert_padding_state_zero(pool, counts)
    refs = [FlorisBatch(lx, ly, B, **kw) for lx, ly in farms]
    for fb in refs:
        fb.reset(pool.get_state("ws"), pool.get_state("wd"), host_trig=False)
    for k in range(L_ep - 1):
        for lay, n in enumerate(COUNTS):
            rows = ids == lay
            assert_state_equal(pool, refs[lay], rows, n, (k, lay), names=("xs", "ys", "order"))
            if k == 0:  # the start observation (reward and truncated still belong to the finished episode)
                trows = torch.as_tensor(rows, device="cuda")
                for key in PER_TURBINE:
                    p = pool.out[key][trows]
                    assert torch.equal(p[:, :n], refs[lay].out[key][trows]) and not bool(p[:, n:].any()), (lay, key)
            else:
                assert_rows_equal(pool.out, refs[lay].out, rows, n, (k, lay))
        a = act()
        pool.step(a)
        for fb, n in zip(refs, COUNTS):
            fb.step(a[:, :n].contiguous())
        torch.cuda.synchronize()
        assert_padding_state_zero(pool, counts)
    for fb in [pool] + refs:
        fb.close()


def test_assign_from_80_to_7_turbines_zeroes_the_padding_state(cuda_device, farms):
    import torch

    B = 64
    pool = make_mixed(farms, B, precision="f32", kernel="fast", max_iter=50)
    pool.assign_layouts(None, 3)
    pool.reset(*sample_winds(B, seed=1))
    rng = np.random.default_rng(0)
    for _ in range(3):
        pool.step(torch.as_tensor(rng.uniform(-5, 5, (B, T)).astype(np.float32), device="cuda"))
    before = {name: pool.get_state(name) for name in ("yaw", "acc", "acc_prev")}
    assert all(v[:, 7:].any() for v in before.values())
    moved = np.arange(0, B, 2)
    pool.assign_layouts(moved, 1)
    for name, old in before.items():
        now = pool.get_state(name)
        assert not now[moved, 7:].any(), name
        assert np.array_equal(now[moved, :7], old[moved, :7]), name  # the env's own columns are kept
        assert np.array_equal(now[1::2], old[1::2]), name  # envs not listed are untouched
    pool.close()


@pytest.mark.parametrize("route", ["zero_copy", "staged"])
def test_step_host_equals_device_path(cuda_device, monkeypatch, farms, route):
    import torch

    monkeypatch.setenv("WFCRL_B200_HOST_PATH", route)
    B = 2048  # the staged route runs in chunks from 2048 envs, and strict FP32 flags some envs: compact records
    kw = dict(precision="f32", kernel="fast", max_iter=50, reward_shaper="step")
    a, b = make_mixed(farms, B, **kw), make_mixed(farms, B, **kw)
    ids = np.arange(B) % 4
    for fb in (a, b):
        fb.assign_layouts(None, ids)
        fb.reset(*sample_winds(B, seed=8))
    rng = np.random.default_rng(3)
    n_flagged = 0
    for k in range(3):
        act = torch.as_tensor(rng.uniform(-5, 5, (B, T)).astype(np.float32))
        host = a.step_host(act.pin_memory())
        dev = b.step(act.cuda())
        torch.cuda.synchronize()
        n_flagged += int(b.get_state("ambiguous").sum())
        for key in PER_TURBINE + PER_ENV:
            assert torch.equal(host[key], dev[key].cpu()), (k, key)
    assert n_flagged > 0
    a.close()
    b.close()


def test_checkpoint_resumes_bit_for_bit(cuda_device, farms):
    import torch

    B = 64
    kw = dict(precision="f64", kernel="fast", max_iter=40, reward_shaper="step")
    a = make_mixed(farms, B, **kw)
    a.assign_layouts(None, np.arange(B) % 4)
    a.reset(*sample_winds(B, seed=9))
    rng = np.random.default_rng(4)
    acts = [torch.as_tensor(rng.uniform(-5, 5, (B, T)).astype(np.float32), device="cuda") for _ in range(6)]
    for act in acts[:3]:
        a.step(act)
    sd = a.state_dict()
    b = make_mixed(farms, B, **kw)
    b.load_state_dict(sd)
    for name in ("layout_id", "turbine_count", "xs", "ys", "order", "cs", "yaw", "acc"):
        assert np.array_equal(a.get_state(name), b.get_state(name)), name
    for act in acts[3:]:
        oa = {k: v.clone() for k, v in a.step(act).items()}
        ob = b.step(act)
        torch.cuda.synchronize()
        for key in PER_TURBINE + PER_ENV:
            assert torch.equal(oa[key], ob[key]), key
    a.close()
    b.close()


def test_sized_call_with_full_counts_equals_set_layouts(cuda_device):
    import torch

    from wfcrl_b200.backend import FlorisBatch

    farms = [layout("Turb32_Row5_"), layout("Turb_TCRWP_")]
    B = 256
    kw = dict(precision="f32", kernel="fast", max_iter=50)
    a, b = FlorisBatch(*farms[0], B, **kw), FlorisBatch(*farms[0], B, **kw)
    a.set_layouts([f[0] for f in farms], [f[1] for f in farms])
    b.set_mixed_layouts([f[0] for f in farms], [f[1] for f in farms])
    for fb in (a, b):
        fb.assign_layouts(None, np.arange(B) % 2)
        fb.reset(*sample_winds(B, seed=6))
    rng = np.random.default_rng(5)
    for _ in range(3):
        act = torch.as_tensor(rng.uniform(-5, 5, (B, 32)).astype(np.float32), device="cuda")
        oa = {k: v.clone() for k, v in a.step(act).items()}
        ob = b.step(act)
        torch.cuda.synchronize()
        for key in PER_TURBINE + PER_ENV:
            assert torch.equal(oa[key], ob[key]), key
    for name in ("xs", "ys", "order", "xi", "yi", "turbine_count"):
        assert np.array_equal(a.get_state(name), b.get_state(name)), name
    a.close()
    b.close()


def test_rejections(cuda_device, farms):
    from wfcrl_b200.backend import FlorisBatch

    ptr = lambda a: a.ctypes.data_as(C.c_void_p)  # noqa: E731
    B = 8
    fb = make_mixed(farms, B, precision="f64", kernel="fast")
    lib, h = fb.lib, fb.handle
    fb.assign_layouts(None, np.arange(B) % 4)
    before = fb.get_state("layout_id")
    x = np.zeros((2, T))
    x[:, :7] = np.arange(7) * 500.0
    for bad_count in (0, T + 1, -3):
        counts = np.array([7, bad_count], dtype=np.int32)
        assert lib.wf_set_layouts_sized(h, 2, ptr(counts), ptr(x), ptr(x)) == 1
        assert b"turbine count" in lib.wf_last_error()
    counts = np.array([7, 7], dtype=np.int32)
    bad = x.copy()
    bad[1, 3] = np.nan
    assert lib.wf_set_layouts_sized(h, 2, ptr(counts), ptr(bad), ptr(x)) == 1 and b"finite" in lib.wf_last_error()
    beyond = x.copy()
    beyond[:, 7:] = np.nan  # entries beyond a layout's count are ignored
    assert np.array_equal(fb.get_state("layout_id"), before)  # the rejected calls changed nothing
    assert lib.wf_set_layouts_sized(h, 2, ptr(counts), ptr(beyond), ptr(beyond)) == 0
    assert (fb.get_state("turbine_count") == 7).all()
    # read-only count, nonzero padding state
    state = np.full(B, 7, dtype=np.int32)
    assert lib.wf_set_state(h, b"turbine_count", ptr(state), state.nbytes) == 1
    yaw = np.zeros((B, T))
    yaw[5, 7] = 1.0
    assert lib.wf_set_state(h, b"yaw", ptr(yaw), yaw.nbytes) == 1 and b"env 5" in lib.wf_last_error()
    acc = np.zeros((B, T), dtype=np.float32)
    acc[2, 79] = 0.5
    for name in (b"acc", b"acc_prev"):
        assert lib.wf_set_state(h, name, ptr(acc), acc.nbytes) == 1 and b"env 2" in lib.wf_last_error()
    yaw[5, 7] = 0.0
    yaw[5, 6] = 1.0
    assert lib.wf_set_state(h, b"yaw", ptr(yaw), yaw.nbytes) == 0
    fb.close()
    # basic-kernel (incl. the 5x5 grid) and multi-agent handles refuse padding
    counts = np.array([80, 7], dtype=np.int32)
    x = np.zeros((2, T))
    x[0], x[1, :7] = farms[3][0], farms[1][0]
    y = np.zeros((2, T))
    y[0], y[1, :7] = farms[3][1], farms[1][1]
    for kw in (dict(kernel="basic"), dict(kernel="basic", config_overrides={"turbine_grid_points": 5}),
               dict(kernel="fast", multi_agent=True)):
        fb = FlorisBatch(*farms[3], 4, precision="f64", **kw)
        assert fb.lib.wf_set_layouts_sized(fb.handle, 2, ptr(counts), ptr(x), ptr(y)) == 1, kw
        assert b"not supported" in fb.lib.wf_last_error(), kw
        assert (fb.get_state("turbine_count") == 80).all()
        fb.close()


def test_vec_env_pad_turbines(cuda_device):
    import torch

    from wfcrl_b200 import environments as envs

    ids = [n + "Floris" for n in POOL]
    B = 16
    env = envs.make_vec(ids, B, precision="f64", pad_turbines=True, max_num_steps=20)
    assert env.num_turbines == T
    assert env.observation_space["wind_speed"].low.min() == 0
    obs = env.reset(seed=3)
    counts = np.array(COUNTS)[np.arange(B) % 4]
    assert env.turbine_counts.cpu().numpy().tolist() == counts.tolist()
    assert obs["turbine_mask"].shape == (B, T) and obs["turbine_mask"].dtype == torch.bool
    assert np.array_equal(obs["turbine_mask"].cpu().numpy(), np.arange(T)[None, :] < counts[:, None])
    for k in ("yaw", "wind_speed", "wind_direction"):
        assert obs[k].shape == (B, T)
    singles = [envs.make_vec(i, B, precision="f64", max_num_steps=20) for i in ids]
    for e in singles:  # same global ids: env g of the single batch draws env g's winds
        e.reset(seed=3)
    rng = np.random.default_rng(1)
    for _ in range(3):
        act = rng.uniform(-5, 5, (B, T)).astype(np.float32)
        obs, reward, _, _, info = env.step(torch.as_tensor(act, device="cuda"))
        reward = reward.clone()
        for lay, (e, n) in enumerate(zip(singles, COUNTS)):
            rows = torch.as_tensor(np.arange(B) % 4 == lay, device="cuda")
            _, r1, _, _, i1 = e.step(torch.as_tensor(np.ascontiguousarray(act[:, :n]), device="cuda"))
            assert torch.equal(reward[rows], r1[rows]), lay
            assert torch.equal(info["power"][rows][:, :n], i1["power"][rows]), lay
    for e in [env] + singles:
        e.close()
