"""Layout pool (wf_set_layouts / wf_assign_layouts / wf_set_layout_sampling): a handle whose envs run different farms of one
turbine count.  Every env must compute, bit for bit, what a single-layout handle of its farm computes; the library's layout
draws must follow their stated formula; checkpoints must carry the layout ids."""
import ctypes as C

import numpy as np
import pytest

from oracle.env_oracle import philox4x32_10
from tests._util import layout, sample_winds

pytestmark = pytest.mark.gpu

OUT_KEYS = ("yaw", "wind_speed", "wind_direction", "power", "load", "reward", "freewind", "truncated")


def rotated_hornsrev():
    """HornsRev1 rotated by 17 degrees about a far point: same turbine count, another bounding-box centre."""
    x, y = layout("HornsRev1_")
    c, s = np.cos(np.radians(17.0)), np.sin(np.radians(17.0))
    return 1500.0 + c * x - s * y, -800.0 + s * x + c * y


def pool_of(names):
    return [layout(n) if isinstance(n, str) else n for n in names]


PAIRS = {
    "row5_tcrwp": ["Turb32_Row5_", "Turb_TCRWP_"],
    "turb6_rows": ["Turb6_Row2_", "Turb6_Row1_"],
    "hornsrev_rotated": ["HornsRev1_", rotated_hornsrev()],
}
# (precision, kernel, strict, multi_agent, interface mode, vortex table)
MODES = {
    "f64_fast_table": ("f64", "fast", True, False, False, True),
    "f64_fast_direct": ("f64", "fast", True, False, False, False),
    "f64_basic": ("f64", "basic", True, False, False, True),
    "f32_strict": ("f32", "fast", True, False, False, True),
    "f32_relaxed": ("f32", "fast", False, False, False, True),
    "multi_agent": ("f32", "fast", True, True, False, True),
    "interface": ("f64", "fast", True, False, True, True),
}


def _u53(a, b):
    return float(((int(a) >> 5) << 26) | (int(b) >> 6)) / 9007199254740992.0


def drawn_layout(seed, gid, episode, n_layouts):
    """The layout id the library draws for (seed, global env id, episode index): draw word 2 of the wind sampler."""
    r2 = philox4x32_10((gid & 0xFFFFFFFF, gid >> 32, episode, 2), (seed & 0xFFFFFFFF, seed >> 32))
    return int(np.floor(_u53(r2[0], r2[1]) * n_layouts))


def make_pool(layouts, B, **kw):
    from wfcrl_b200.backend import FlorisBatch

    lx, ly = layouts[0]
    fb = FlorisBatch(lx, ly, B, **kw)
    fb.set_layouts([p[0] for p in layouts], [p[1] for p in layouts])
    return fb


@pytest.mark.parametrize("mode", list(MODES))
@pytest.mark.parametrize("pair", list(PAIRS))
def test_pool_equals_single_layout_handles(cuda_device, monkeypatch, pair, mode):
    import torch

    from wfcrl_b200.backend import FlorisBatch

    precision, kernel, strict, multi_agent, interface, table = MODES[mode]
    if table:
        monkeypatch.delenv("WFCRL_B200_NO_VTAB", raising=False)
    else:
        monkeypatch.setenv("WFCRL_B200_NO_VTAB", "1")
    layouts = pool_of(PAIRS[pair])
    T = len(layouts[0][0])
    B = 1024 if mode == "f32_strict" else 256  # enough envs for the guard band to flag some
    kw = dict(precision=precision, kernel=kernel, max_iter=50, strict=strict, multi_agent=multi_agent,
              reward_shaper="step")
    pool = make_pool(layouts, B, **kw)
    refs = [FlorisBatch(lx, ly, B, **kw) for lx, ly in layouts]
    ids = np.arange(B) % 2
    pool.assign_layouts(None, ids)
    ws, wd = sample_winds(B, seed=5, tie_every=3 if pair == "turb6_rows" else 0)
    for fb in [pool] + refs:
        fb.reset(ws, wd, host_trig=True)
    rng = np.random.default_rng(11)
    n_flagged = 0
    for k in range(4):
        if interface:
            cmd = torch.as_tensor(rng.uniform(-20, 20, (B, T)), device="cuda")
            outs = [fb.update_command(cmd) for fb in [pool] + refs]
        else:
            act = torch.as_tensor(rng.uniform(-5, 5, (B, T)).astype(np.float32), device="cuda")
            outs = [fb.step(act) for fb in [pool] + refs]
        torch.cuda.synchronize()
        states = {name: [fb.get_state(name) for fb in [pool] + refs] for name in ("ambiguous", "xs", "order")}
        n_flagged += int(states["ambiguous"][0].sum())
        for lay in range(2):
            rows = torch.as_tensor(ids == lay, device="cuda")
            for key in OUT_KEYS:
                assert torch.equal(outs[0][key][rows], outs[1 + lay][key][rows]), (k, lay, key)
            for name, vals in states.items():
                assert np.array_equal(vals[0][ids == lay], vals[1 + lay][ids == lay]), (k, lay, name)
    if mode == "f32_strict":
        assert n_flagged > 0  # the FP64 re-solve path ran for pool envs
    for fb in [pool] + refs:
        fb.close()


def _sampling_pool(B, L=3, **kw):
    names = ["Turb6_Row2_", "Turb6_Row1_", (layout("Turb6_Row2_")[1], layout("Turb6_Row2_")[0])][:L]
    fb = make_pool(pool_of(names), B, precision=kw.pop("precision", "f64"), kernel="fast", **kw)
    fb.set_layout_sampling(True)
    return fb


def test_sampled_ids_follow_the_formula(cuda_device):
    import torch

    B, L, seed, off = 64, 3, 0x1234567890ABCDEF, (1 << 32) - 5  # the global ids cross the 32-bit word boundary
    fb = _sampling_pool(B, L, max_iter=4)
    # wf_reset_sampled, two episodes: episode index before the call is the counter word
    for _ in range(2):
        ep = fb.get_state("episode")
        fb.reset_sampled(None, seed, off)
        got = fb.get_state("layout_id")
        assert [drawn_layout(seed, off + b, int(ep[b]), L) for b in range(B)] == got.tolist()
    # in-kernel auto-resets over two episodes
    fb.set_autoreset(True, seed=seed + 1, env_id_offset=off)
    act = torch.zeros(B, 6, dtype=torch.float32, device="cuda")
    n = 0
    for _ in range(8):
        out = fb.step(act)
        torch.cuda.synchronize()
        if bool(out["truncated"].any()):
            ep = fb.get_state("episode")
            fb.autoreset_finish()
            got = fb.get_state("layout_id")
            assert [drawn_layout(seed + 1, off + b, int(ep[b]), L) for b in range(B)] == got.tolist()
            n += 1
    assert n == 2
    fb.close()


def test_sampling_leaves_winds_and_ti_alone(cuda_device):
    B = 256
    on = _sampling_pool(B)
    off = _sampling_pool(B)
    off.set_layout_sampling(False)
    for rep in range(3):
        for fb in (on, off):
            fb.reset_sampled(None, 99, 7, turbulence_intensity_range=(0.04, 0.12))
        for name in ("ws", "wd", "ti_ambient", "episode"):
            assert np.array_equal(on.get_state(name), off.get_state(name)), (rep, name)
    assert (off.get_state("layout_id") == 0).all() and len(set(on.get_state("layout_id").tolist())) == 3
    on.close()
    off.close()


def test_shards_reproduce_the_single_batch(cuda_device):
    B = 128
    full = _sampling_pool(B)
    halves = [_sampling_pool(B // 2) for _ in range(2)]
    for _ in range(2):
        full.reset_sampled(None, 5, 0)
        for h, fb in enumerate(halves):
            fb.reset_sampled(None, 5, h * B // 2)
        for name in ("layout_id", "ws", "wd", "xs", "order"):
            joined = np.concatenate([fb.get_state(name) for fb in halves])
            assert np.array_equal(full.get_state(name), joined), name
    for fb in [full] + halves:
        fb.close()


def test_sampled_id_frequencies(cuda_device):
    from scipy.stats import chisquare

    B, L = 8192, 3
    fb = _sampling_pool(B, L)
    counts = np.zeros(L)
    for _ in range(4):
        fb.reset_sampled(None, 2024, 0, warmup_solves=0)
        counts += np.bincount(fb.get_state("layout_id"), minlength=L)
    assert counts.sum() == 4 * B
    assert chisquare(counts).pvalue > 1e-4, counts
    fb.close()


@pytest.mark.parametrize("precision", ["f32", "f64"])
def test_autoreset_geometry_and_steps_equal_fresh_handle(cuda_device, precision):
    import torch

    from wfcrl_b200.backend import FlorisBatch

    layouts = pool_of(["Turb32_Row5_", "Turb_TCRWP_"])
    B, T, L_ep = 128, 32, 4
    kw = dict(precision=precision, kernel="fast", max_iter=L_ep)
    pool = make_pool(layouts, B, **kw)
    pool.set_layout_sampling(True)
    ws, wd = sample_winds(B, seed=3)
    pool.reset(ws, wd, host_trig=False)
    pool.set_autoreset(True, seed=41, env_id_offset=0)
    act = torch.zeros(B, T, dtype=torch.float32, device="cuda")
    while not bool(pool.step(act)["truncated"].any()):
        pass
    pool.autoreset_finish()
    torch.cuda.synchronize()
    ids = pool.get_state("layout_id")
    assert set(ids.tolist()) == {0, 1}
    refs = [FlorisBatch(lx, ly, B, **kw) for lx, ly in layouts]
    for fb in refs:
        fb.reset(pool.get_state("ws"), pool.get_state("wd"), host_trig=False)
    outs = [pool.out] + [fb.out for fb in refs]
    rng = np.random.default_rng(2)
    for k in range(L_ep - 1):
        # after the reset: the start observation (reward and truncated still belong to the finished episode's last step)
        keys = ("yaw", "wind_speed", "wind_direction", "freewind", "power", "load") if k == 0 else OUT_KEYS
        for lay in range(2):
            rows = ids == lay
            trows = torch.as_tensor(rows, device="cuda")
            for name in ("xs", "ys", "order", "cs"):
                assert np.array_equal(pool.get_state(name)[rows], refs[lay].get_state(name)[rows]), (k, lay, name)
            for key in keys:
                assert torch.equal(outs[0][key][trows], outs[1 + lay][key][trows]), (k, lay, key)
        act = torch.as_tensor(rng.uniform(-5, 5, (B, T)).astype(np.float32), device="cuda")
        for fb in [pool] + refs:
            fb.step(act)
        torch.cuda.synchronize()
    for fb in [pool] + refs:
        fb.close()


def test_checkpoint_resumes_mixed_layouts(cuda_device):
    import torch

    layouts = pool_of(["HornsRev1_", rotated_hornsrev()])
    B, T = 64, 80
    kw = dict(precision="f64", kernel="fast", max_iter=40, reward_shaper="step")
    a = make_pool(layouts, B, **kw)
    a.assign_layouts(np.arange(0, B, 3), 1)
    ws, wd = sample_winds(B, seed=9)
    a.reset(ws, wd, host_trig=True)
    rng = np.random.default_rng(4)
    acts = [torch.as_tensor(rng.uniform(-5, 5, (B, T)).astype(np.float32), device="cuda") for _ in range(6)]
    for act in acts[:3]:
        a.step(act)
    sd = a.state_dict()
    assert (sd["layout_id"] == (np.arange(B) % 3 == 0)).all()
    b = make_pool(layouts, B, **kw)
    b.load_state_dict(sd)
    for name in ("layout_id", "xs", "ys", "order", "xi", "yi", "cs"):
        assert np.array_equal(a.get_state(name), b.get_state(name)), name
    for act in acts[3:]:
        oa = {k: v.clone() for k, v in a.step(act).items()}
        ob = b.step(act)
        torch.cuda.synchronize()
        for key in OUT_KEYS:
            assert torch.equal(oa[key], ob[key]), key
    # a dict saved before the layout pool existed restores every env to layout 0
    del sd["layout_id"]
    b.load_state_dict(sd)
    assert (b.get_state("layout_id") == 0).all()
    a.close()
    b.close()


def test_invalid_pool_calls_are_rejected(cuda_device):
    from wfcrl_b200 import _lib

    layouts = pool_of(["Turb6_Row2_", "Turb6_Row1_"])
    B = 8
    fb = make_pool(layouts, B, precision="f64", kernel="fast")
    lib, h = fb.lib, fb.handle
    ptr = lambda a: a.ctypes.data_as(C.c_void_p)  # noqa: E731
    x = np.zeros((2, 6))
    assert lib.wf_set_layouts(h, 0, ptr(x), ptr(x)) == 1 and b"n_layouts" in lib.wf_last_error()
    bad = x.copy()
    bad[1, 3] = np.inf
    assert lib.wf_set_layouts(h, 2, ptr(bad), ptr(x)) == 1 and b"finite" in lib.wf_last_error()
    with pytest.raises(ValueError):
        fb.set_layouts(np.zeros((2, 5)), np.zeros((2, 5)))  # wrong turbine count: caught before the C call
    env_ids = np.array([0, B], dtype=np.int32)
    lids = np.array([1, 0], dtype=np.int32)
    assert lib.wf_assign_layouts(h, ptr(env_ids), 2, ptr(lids), None) == 1 and b"env id" in lib.wf_last_error()
    env_ids[1] = 1
    lids[0] = 2
    assert lib.wf_assign_layouts(h, ptr(env_ids), 2, ptr(lids), None) == 1 and b"layout id" in lib.wf_last_error()
    lids[0] = -1
    assert lib.wf_assign_layouts(h, ptr(env_ids), 2, ptr(lids), None) == 1
    assert (fb.get_state("layout_id") == 0).all()  # a rejected call changes nothing
    state = np.zeros(B, dtype=np.int32)
    assert lib.wf_set_state(h, b"layout_id", ptr(state), state.nbytes) == 1
    assert b"wf_assign_layouts" in lib.wf_last_error()
    with pytest.raises(_lib.WfError):
        fb.set_state("layout_id", 1)
    fb.close()


def test_vec_env_cycle_sample_and_options(cuda_device):
    """VecWindFarmEnv / make_vec over a list of env ids: cycle assignment by global id, host draws for reset(seed=...),
    explicit ids through options, library draws at auto-resets."""
    import torch

    from wfcrl_b200 import environments as envs

    B, off = 16, 5
    env = envs.make_vec(["Turb6_Row2_Floris", "Turb6_Row1_Floris"], B, precision="f64", max_num_steps=3,
                        env_id_offset=off)
    env.reset(seed=1)
    assert env.layout_ids.cpu().tolist() == [(off + b) % 2 for b in range(B)]
    env.reset(options={"layout": 1, "wind_speed": 8.0, "wind_direction": 270.0}, env_ids=[0, 3])
    ids = env.layout_ids.cpu().numpy()
    assert ids[0] == 1 and ids[3] == 1 and ids[1] == (off + 1) % 2
    env.close()

    env = envs.make_vec(["Turb6_Row2_Floris", "Turb6_Row1_Floris"], B, precision="f64", max_num_steps=3,
                        env_id_offset=off, layout_assignment="sample")
    env.reset(seed=7)
    want = [np.random.default_rng((7 + off + b, 2)).integers(2) for b in range(B)]
    assert env.layout_ids.cpu().tolist() == want
    env.reset(options={"layout": np.arange(B) % 2})  # library path: the given ids are kept
    assert env.layout_ids.cpu().tolist() == (np.arange(B) % 2).tolist()
    act = torch.zeros(B, 6, dtype=torch.float32, device="cuda")
    ep = env.backend.get_state("episode")
    for _ in range(2):
        env.step(act)
    assert env.layout_ids.cpu().tolist() == [drawn_layout(7, off + b, int(ep[b]), 2) for b in range(B)]
    env.close()
