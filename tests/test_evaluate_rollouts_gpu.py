"""Rollout evaluation (wf_evaluate_rollouts / evaluate_rollouts / best_sequence / cem_plan): K open-loop action sequences of H
steps per env evaluated from the current state without stepping.  Row (b, k, h) of every output must equal, bit for bit,
row b of what the (h+1)-th of H successive steps with candidate k's actions would write on the same handle in the same
state; rows after a candidate's truncating step read 0; nothing a step or get_state can see may change."""
import ctypes as C

import numpy as np
import pytest

from tests._util import layout, sample_winds
from tests.test_evaluate_actions_gpu import MODES, OUTPUTS, STATE, _actions, _env_vars, _warm

pytestmark = pytest.mark.gpu


def _check_against_steps(fb, act):
    """The reference loop: state_dict -> step(act[:, k, h]) for h = 0..H-1 -> load_state_dict, with an evaluation in the
    same state before each candidate (load_state_dict leaves the vortex table stale: both routes are covered).  Rows after
    an env's truncating step must be 0.  Returns the flagged rows per step h."""
    import torch

    B, K, H, _ = act.shape
    flagged = np.zeros(H, dtype=np.int64)
    for k in range(K):
        ev = {key: v.clone() for key, v in fb.evaluate_rollouts(act).items()}
        sd = fb.state_dict()
        done = torch.zeros(B, dtype=torch.bool, device="cuda")
        for h in range(H):
            out = fb.step(act[:, k, h].contiguous())
            torch.cuda.synchronize()
            for key in OUTPUTS:
                ref = out[key]
                expect = torch.where(done.view((B,) + (1,) * (ref.dim() - 1)), torch.zeros_like(ref), ref)
                assert torch.equal(ev[key][:, k, h], expect), (k, h, key)
            amb = torch.as_tensor(fb.get_state("ambiguous").astype(bool), device="cuda") & ~done
            assert torch.equal(ev["ambiguous"][:, k, h], amb), (k, h)
            flagged[h] += int(amb.sum())
            done |= out["truncated"].bool()
        fb.load_state_dict(sd)
    return flagged


@pytest.mark.parametrize("KH", [(1, 1), (3, 5), (6, 2)])
@pytest.mark.parametrize("name", ["Ablaincourt_", "Turb32_Row5_", "HornsRev1_"])
@pytest.mark.parametrize("mode", list(MODES))
def test_equals_steps(cuda_device, monkeypatch, mode, name, KH):
    from wfcrl_b200.backend import FlorisBatch

    precision, strict, table, baked = MODES[mode]
    _env_vars(monkeypatch, table, baked)
    lx, ly = layout(name)
    (K, H), T, B = KH, len(lx), 64
    fb = FlorisBatch(lx, ly, B, precision=precision, kernel="fast", max_iter=1000, strict=strict, reward_shaper="step")
    ws, wd = sample_winds(B, seed=T + K, tie_every=5)
    fb.reset(ws, wd, host_trig=True)
    rng = np.random.default_rng(K * H)
    _warm(fb, rng)
    _check_against_steps(fb, _actions(rng, (B, K, H, T)))
    fb.close()


SEMANTICS = {
    "discrete": dict(continuous_control=False),
    "reference_pct": dict(reward_shaper="reference", shaper_reference=0.4),
    "step_pct": dict(reward_shaper="step"),
    "load_coef": dict(load_coef=0.7),
    "constraint": dict(),
    "multi_agent": dict(multi_agent=True),
}


@pytest.mark.parametrize("precision", ["f64", "f32"])
@pytest.mark.parametrize("case", list(SEMANTICS))
def test_env_semantics(cuda_device, monkeypatch, case, precision):
    import torch

    from wfcrl_b200.backend import FlorisBatch

    _env_vars(monkeypatch, True)
    lx, ly = layout("Turb6_Row2_" if case == "multi_agent" else "Ablaincourt_")
    T, B, K, H = len(lx), 64, 3, 4
    kw = SEMANTICS[case]
    continuous = kw.get("continuous_control", True)
    fb = FlorisBatch(lx, ly, B, precision=precision, kernel="fast", max_iter=1000, **kw)
    ws, wd = sample_winds(B, seed=len(case))
    fb.reset(ws, wd, host_trig=True)
    rng = np.random.default_rng(len(case))
    _warm(fb, rng, continuous=continuous)
    act = _actions(rng, (B, K, H, T), continuous)
    if case == "step_pct":
        assert np.all(fb.get_state("shaper_ref") != 0)
    if case == "constraint":
        # acc just below the limit 0.1 * rate * dt * (num_moves + 1) in half the envs (0 in the others), and full-step
        # actions: step 0 moves, and its |a| = yaw_step lifts acc over the next step's limit, so that the constraint first
        # fires at h = 1 in the first half and not at all in the second
        limit = 0.1 * fb.cfg.actuator_rate * fb.cfg.dt
        assert fb.cfg.yaw_step > limit
        act = torch.where(act >= 0, 6.0, -6.0)
        acc = fb.get_state("acc")
        acc[: B // 2] = (limit * (fb.get_state("num_moves")[: B // 2] + 1) * (1 - 1e-3))[:, None]
        acc[B // 2:] = 0.0
        fb.set_state("acc", acc)
        ev = fb.evaluate_rollouts(act)
        torch.cuda.synchronize()
        yaw0 = torch.as_tensor(fb.get_state("yaw"), device="cuda")[:, None, :]
        moved0 = ev["yaw"][:, :, 0].double() != yaw0
        moved1 = ev["yaw"][:, :, 1] != ev["yaw"][:, :, 0]
        assert bool(moved0[: B // 2].any()) and not bool(moved1[: B // 2].any()) and bool(moved1[B // 2:].any())
    if case == "multi_agent":  # per-agent staleness: acc_prev differs from acc, and is carried from step to step
        acc_prev = fb.get_state("acc_prev")
        acc_prev[::2] = 1e4
        fb.set_state("acc_prev", acc_prev)
        assert not np.array_equal(fb.get_state("acc"), fb.get_state("acc_prev"))
    _check_against_steps(fb, act)
    fb.close()


def test_strict_flagged_rows_equal_the_resolve(cuda_device, monkeypatch):
    """Rows a strict FP32 handle flags at h > 0 (winds at the foot of the power curve) equal the re-solved steps, and the
    StepPercentage chain runs through the re-solve's double reward."""
    from wfcrl_b200.backend import FlorisBatch

    _env_vars(monkeypatch, True)
    lx, ly = layout("Turb32_Row5_")
    T, B, K, H = len(lx), 512, 3, 3
    rng = np.random.default_rng(3)
    ws, wd = sample_winds(B, seed=3)
    ws[: B // 2] = rng.uniform(3.0, 4.5, B // 2)
    fb = FlorisBatch(lx, ly, B, precision="f32", kernel="fast", max_iter=1000, reward_shaper="step")
    fb.reset(ws, wd, host_trig=True)
    for _ in range(2):
        fb.step(_actions(rng, (B, T)))
    flagged = _check_against_steps(fb, _actions(rng, (B, K, H, T)))
    assert flagged[1:].sum() > 0, flagged
    fb.close()


@pytest.mark.parametrize("mode", ["f64_table", "f32_strict"])
def test_truncation(cuda_device, monkeypatch, mode):
    import torch

    from wfcrl_b200.backend import FlorisBatch

    precision, strict, table, _ = MODES[mode]
    _env_vars(monkeypatch, table)
    lx, ly = layout("Turb6_Row2_")
    T, B, K, H, max_iter = len(lx), 128, 3, 5, 40
    ws, wd = sample_winds(B, seed=4)
    rng = np.random.default_rng(4)
    kw = dict(precision=precision, kernel="fast", max_iter=max_iter, strict=strict, reward_shaper="step")
    fb = FlorisBatch(lx, ly, B, **kw)
    fb.reset(ws, wd, host_trig=True)
    fb.step(_actions(rng, (B, T)))
    num_iter = np.full(B, max_iter - 3, dtype=np.int32)  # step h = 2 truncates
    num_iter[B // 2:] = max_iter + 2  # already past max_iter: never truncates
    fb.set_state("num_iter", num_iter)
    act = _actions(rng, (B, K, H, T))
    ev = {k: v.clone() for k, v in fb.evaluate_rollouts(act).items()}
    torch.cuda.synchronize()
    first = slice(0, B // 2)
    assert bool(ev["truncated"][first, :, 2].all()) and not bool(ev["truncated"][first][:, :, [0, 1, 3, 4]].any())
    for key, v in ev.items():
        assert not bool(v[first, :, 3:].any()), key
    assert not bool(ev["truncated"][B // 2:].any()) and bool((ev["wind_speed"][B // 2:] > 0).all())
    _check_against_steps(fb, act)
    fb.close()

    # with the auto-reset armed nothing is marked or reset: twin handles stay equal over later steps
    twins = [FlorisBatch(lx, ly, B, **kw) for _ in range(2)]
    acts = [_actions(rng, (B, T)) for _ in range(3)]
    for fb in twins:
        fb.reset(ws, wd, host_trig=True)
        fb.set_autoreset(True, seed=9)
        fb.step(acts[0])
        fb.set_state("num_iter", max_iter - 3)
    twins[0].evaluate_rollouts(act)
    for fb in twins:
        fb.autoreset_finish()
    torch.cuda.synchronize()
    for name in STATE:
        assert np.array_equal(twins[0].get_state(name), twins[1].get_state(name)), name
    for a in acts[1:]:
        outs = [{k: v.clone() for k, v in fb.step(a).items()} for fb in twins]
        torch.cuda.synchronize()
        for key in OUTPUTS:
            assert torch.equal(outs[0][key], outs[1][key]), key
    for fb in twins:
        fb.close()


@pytest.mark.parametrize("mode", ["f64_table", "f32_strict"])
def test_state_untouched(cuda_device, monkeypatch, mode):
    import torch

    from wfcrl_b200.backend import FlorisBatch

    precision, strict, table, _ = MODES[mode]
    _env_vars(monkeypatch, table)
    lx, ly = layout("Turb32_Row5_")
    T, B, K, H = len(lx), 512, 3, 4
    rng = np.random.default_rng(8)
    ws, wd = sample_winds(B, seed=8)
    ws[: B // 2] = rng.uniform(3.0, 4.5, B // 2)
    kw = dict(precision=precision, kernel="fast", max_iter=20, strict=strict, reward_shaper="step")
    twins = [FlorisBatch(lx, ly, B, **kw) for _ in range(2)]
    for fb in twins:
        fb.reset(ws, wd, host_trig=True)
        fb.set_autoreset(True, seed=5)
    acts = [_actions(rng, (B, T)) for _ in range(4)]
    for fb in twins:
        fb.step(acts[0])
    torch.cuda.synchronize()
    before = {name: twins[0].get_state(name).tobytes() for name in STATE}
    cand = _actions(rng, (B, K, H, T))
    twins[0].evaluate_rollouts(cand)
    torch.cuda.synchronize()
    for name in STATE:
        assert twins[0].get_state(name).tobytes() == before[name], name
    for act in acts[1:]:
        outs = [{k: v.clone() for k, v in fb.step(act).items()} for fb in twins]
        twins[0].evaluate_rollouts(cand)
        torch.cuda.synchronize()
        for key in outs[0]:
            assert torch.equal(outs[0][key], outs[1][key]), key
        for name in STATE:
            assert np.array_equal(twins[0].get_state(name), twins[1].get_state(name)), name
    for fb in twins:
        fb.close()


@pytest.mark.parametrize("precision", ["f64", "f32"])
def test_mixed_pool_padding(cuda_device, monkeypatch, precision):
    import torch

    from wfcrl_b200.backend import FlorisBatch

    _env_vars(monkeypatch, True)
    farms = [layout("Ablaincourt_"), layout("Turb32_Row5_")]
    counts = [len(f[0]) for f in farms]
    T, B, K, H = max(counts), 128, 2, 3
    pool = FlorisBatch(*farms[-1], B, precision=precision, kernel="fast", max_iter=1000, reward_shaper="step")
    pool.set_mixed_layouts([f[0] for f in farms], [f[1] for f in farms])
    ids = np.arange(B) % 2
    pool.assign_layouts(None, ids)
    ws, wd = sample_winds(B, seed=2)
    pool.reset(ws, wd, host_trig=True)
    rng = np.random.default_rng(2)
    _warm(pool, rng)
    act = rng.uniform(-6, 6, (B, K, H, T)).astype(np.float32)
    for b in range(B):
        act[b, :, :, counts[ids[b]]:] = np.nan  # ignored
    act = torch.as_tensor(act, device="cuda")
    ev = pool.evaluate_rollouts(act)
    torch.cuda.synchronize()
    for lay, n in enumerate(counts):
        rows = torch.as_tensor(np.flatnonzero(ids == lay), device="cuda")
        for key in ("yaw", "wind_speed", "wind_direction", "power", "load"):
            assert not bool(ev[key][rows][:, :, :, n:].any()), key
    _check_against_steps(pool, act)
    pool.close()


@pytest.mark.parametrize("mode", ["f64_table", "f32_strict"])
def test_first_call_on_a_non_blocking_stream(cuda_device, monkeypatch, mode):
    import torch

    from wfcrl_b200.backend import FlorisBatch

    precision, strict, table, _ = MODES[mode]
    _env_vars(monkeypatch, table)
    lx, ly = layout("Turb32_Row5_")
    T, B, K, H = len(lx), 1024, 3, 4
    rng = np.random.default_rng(12)
    ws, wd = sample_winds(B, seed=12)
    ws[: B // 2] = rng.uniform(3.0, 4.5, B // 2)
    kw = dict(precision=precision, kernel="fast", max_iter=1000, strict=strict, reward_shaper="step")
    twins = [FlorisBatch(lx, ly, B, **kw) for _ in range(2)]
    for fb in twins:
        fb.reset(ws, wd, host_trig=True)
    act = _actions(rng, (B, K, H, T))
    ref = {k: v.clone() for k, v in twins[1].evaluate_rollouts(act).items()}
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        got = {k: v.clone() for k, v in twins[0].evaluate_rollouts(act).items()}
    torch.cuda.synchronize()
    if precision == "f32":
        assert int(ref["ambiguous"].sum()) > 0
    for key in ref:
        assert torch.equal(got[key], ref[key]), key
    for fb in twins:
        fb.close()


def test_launch_counts_scratch_sharing_and_refusals(cuda_device, monkeypatch):
    import torch

    from wfcrl_b200.backend import FlorisBatch
    from wfcrl_b200.vector_env import VecWindFarmEnv

    _env_vars(monkeypatch, True)
    lx, ly = layout("Turb32_Row5_")
    T, B = len(lx), 256
    rng = np.random.default_rng(7)
    act = _actions(rng, (B, 4, 3, T))
    yaw = torch.as_tensor(rng.uniform(-40, 40, (B, 4, T)), device="cuda")
    ws, wd = sample_winds(B, seed=7)
    ws[: B // 2] = rng.uniform(3.0, 4.5, B // 2)  # a strict handle flags rows: the shared fix list and yaw rows are used
    for precision, strict, launches in (("f64", True, 1), ("f32", True, 2), ("f32", False, 1)):
        kw = dict(precision=precision, kernel="fast", max_iter=1000, strict=strict, reward_shaper="step")
        fb, ref = FlorisBatch(lx, ly, B, **kw), FlorisBatch(lx, ly, B, **kw)
        for h in (fb, ref):
            h.reset(ws, wd, host_trig=True)
            h.step(act[:, 0, 0].contiguous())  # a non-zero StepPercentage reference
        expect = {k: v.clone() for k, v in ref.evaluate_rollouts(act).items()}
        expect_act = {k: v.clone() for k, v in ref.evaluate_actions(act[:, :, 0].contiguous()).items()}
        expect_yaw = {k: v.clone() for k, v in ref.evaluate_yaw(yaw).items()}
        torch.cuda.synchronize()
        if precision == "f32" and strict:
            assert int(expect["ambiguous"][:, :, 1:].sum()) > 0
        # H = 1 is evaluate_actions, bit for bit
        h1 = ref.evaluate_rollouts(act[:, :, :1].contiguous())
        for key in expect_act:
            assert torch.equal(h1[key][:, :, 0], expect_act[key]), key
        # the three entry points share the scratch: interleaved with growing K*H, each result equals a fresh handle's
        for K, H in ((1, 1), (1, 2), (2, 2), (2, 3), (3, 3), (4, 3)):
            got = {k: v.clone() for k, v in fb.evaluate_rollouts(act[:, :K, :H].contiguous()).items()}
            got_act = {k: v.clone() for k, v in fb.evaluate_actions(act[:, :K, 0].contiguous()).items()}
            got_yaw = {k: v.clone() for k, v in fb.evaluate_yaw(yaw[:, :K].contiguous()).items()}
            torch.cuda.synchronize()
            for key in got:  # the rows of a candidate do not depend on K or H
                assert torch.equal(got[key], expect[key][:, :K, :H]), (precision, K, H, key)
                assert torch.equal(got_act[key], expect_act[key][:, :K]), (precision, K, key)
            for key in got_yaw:
                assert torch.equal(got_yaw[key], expect_yaw[key][:, :K]), (precision, K, key)
        # evaluate_actions keeps buffers of its own: a rollout evaluation does not overwrite its results
        views = fb.evaluate_actions(act[:, :2, 0].contiguous())
        kept = {k: v.clone() for k, v in views.items()}
        fb.evaluate_rollouts(act)
        torch.cuda.synchronize()
        for key in kept:
            assert torch.equal(views[key], kept[key]), key
        for K, H, fields, n in ((3, 1, None, launches), (2, 3, None, launches + 1), (2, 3, ("truncated",), launches)):
            n0 = fb.launch_count()
            if fields is None:
                fb.evaluate_rollouts(act[:, :K, :H].contiguous())
            else:
                fb.evaluate_rollouts(act[:, :K, :H].contiguous(), fields)
            assert fb.launch_count() - n0 == n, (precision, strict, K, H, fields)
        lib, h, st = fb.lib, fb.handle, fb._stream()
        p = C.c_void_p(act.data_ptr())
        out = C.byref(fb._out_struct)
        n0 = fb.launch_count()
        assert lib.wf_evaluate_rollouts(h, p, 0, 2, out, None, st) == 1 and b"K" in lib.wf_last_error()
        assert lib.wf_evaluate_rollouts(h, p, -1, 2, out, None, st) == 1
        assert lib.wf_evaluate_rollouts(h, p, 2, 0, out, None, st) == 1 and b"H" in lib.wf_last_error()
        assert lib.wf_evaluate_rollouts(h, p, 2, -3, out, None, st) == 1
        assert lib.wf_evaluate_rollouts(h, None, 1, 1, out, None, st) == 1 and b"NULL" in lib.wf_last_error()
        assert lib.wf_evaluate_rollouts(h, p, 1, 1, None, None, st) == 1 and b"NULL" in lib.wf_last_error()
        assert lib.wf_evaluate_rollouts(h, p, 2**16, 2**31 // B // 2**16 + 1, out, None, st) == 1
        assert b"2^31" in lib.wf_last_error()
        assert fb.launch_count() == n0
        with pytest.raises(ValueError):
            fb.evaluate_rollouts(torch.zeros(B, 2, 0, T, dtype=torch.float32, device="cuda"))
        with pytest.raises(ValueError):
            fb.evaluate_rollouts(act[:, :, 0].contiguous())
        with pytest.raises(ValueError):
            fb.evaluate_rollouts(act, ("reward", "obs"))
        with pytest.raises(TypeError):
            fb.evaluate_rollouts(act.double())
        fb.close()
        ref.close()
    basic = FlorisBatch(lx, ly, B, precision="f64", kernel="basic", max_iter=1000)
    n0 = basic.launch_count()
    with pytest.raises(Exception, match="WF_KERNEL_FAST"):
        basic.evaluate_rollouts(act)
    assert basic.launch_count() == n0
    basic.close()
    series = np.stack([np.full(20, 8.0), np.linspace(260, 280, 20)], 1)
    env = VecWindFarmEnv("Turb6_Row2_", B, precision="f64", wind_time_series=series)
    env.reset(seed=0)
    n0 = env.backend.launch_count()
    with pytest.raises(ValueError, match="time-series"):
        env.evaluate_rollouts(_actions(rng, (B, 2, 2, env.num_turbines)))
    assert env.backend.launch_count() == n0
    env.close()


@pytest.mark.parametrize("copy_outputs", [False, True])
def test_vector_env(cuda_device, monkeypatch, copy_outputs):
    import torch

    from wfcrl_b200.vector_env import VecWindFarmEnv

    _env_vars(monkeypatch, True)
    B, K, H, steps = 32, 3, 4, 6
    kw = dict(precision="f32", pad_turbines=True, copy_outputs=copy_outputs, max_num_steps=steps)
    env = VecWindFarmEnv(["Turb6_Row2_", "Ablaincourt_"], B, **kw)
    env.reset(seed=3)
    T = env.num_turbines
    rng = np.random.default_rng(3)
    for _ in range(3):
        env.step(_actions(rng, (B, T)))
    countdowns = list(env._countdowns)
    cand = _actions(rng, (B, K, H, T))
    joint = {k: v.clone() for k, v in env.backend.evaluate_rollouts(cand).items()}
    obs, reward, term, trunc, info = env.evaluate_rollouts({"yaw": cand})
    assert obs["yaw"].shape == (B, K, H, T) and obs["freewind_measurements"].shape == (B, K, H, 2)
    assert obs["turbine_mask"].shape == (B, K, H, T) and info["load"].shape == (B, K, H, T, 4)
    assert reward.shape == term.shape == trunc.shape == info["valid"].shape == (B, K, H) and not bool(term.any())
    assert torch.equal(obs["yaw"], joint["yaw"]) and torch.equal(reward, joint["reward"])
    assert torch.equal(trunc, joint["truncated"].bool()) and torch.equal(info["power"], joint["power"])
    h_trunc = countdowns[0] - 1  # every env was reset together: one cohort, truncating at step h_trunc < H
    assert len(countdowns) == 1 and 0 <= h_trunc < H - 1
    assert bool(trunc[:, :, h_trunc].all()) and int(trunc.sum()) == B * K
    assert torch.equal(info["valid"], (torch.arange(H, device="cuda") <= h_trunc).expand(B, K, H))
    assert (obs["yaw"].data_ptr() == env.backend.evaluate_rollouts(cand)["yaw"].data_ptr()) != copy_outputs
    obs2, reward2, _, trunc2, info2 = env.evaluate_rollouts(cand, observations=False)
    assert obs2 is None and info2["power"] is None and info2["load"] is None
    assert torch.equal(reward2, joint["reward"]) and torch.equal(info2["valid"], info["valid"])
    assert env._countdowns == countdowns
    env.close()


def test_multi_agent_split(cuda_device, monkeypatch):
    import torch

    from wfcrl_b200.vector_env import VecMAWindFarmEnv

    _env_vars(monkeypatch, True)
    B, K, H = 16, 3, 2
    env = VecMAWindFarmEnv("Turb6_Row2_", B, precision="f64")
    env.reset(seed=1)
    T = env.num_turbines
    cand = _actions(np.random.default_rng(1), (B, K, H, T))
    joint = {key: v.clone() for key, v in env.backend.evaluate_rollouts(cand).items()}
    per_agent = {a: {"yaw": cand[:, :, :, i]} for a, i in env.agent_name_mapping.items()}
    for actions in (cand, per_agent):
        obs, reward, term, trunc, info = env.evaluate_rollouts(actions)
        for a, i in env.agent_name_mapping.items():
            assert torch.equal(obs[a]["yaw"], joint["yaw"][:, :, :, i])
            assert torch.equal(obs[a]["wind_speed"], joint["wind_speed"][:, :, :, i])
            assert torch.equal(reward[a], joint["reward"]) and torch.equal(trunc[a], joint["truncated"].bool())
            assert torch.equal(info[a]["power"], joint["power"][:, :, :, i])
            assert torch.equal(info[a]["load"], joint["load"][:, :, :, i]) and bool(info[a]["valid"].all())
    obs, reward, _, _, info = env.evaluate_rollouts(cand, observations=False)
    assert obs is None and all(info[a]["power"] is None for a in env.possible_agents)
    env.close()


@pytest.mark.parametrize("precision", ["f64", "f32"])
def test_cem_plan(cuda_device, monkeypatch, precision):
    import torch

    from wfcrl_b200.planning import best_sequence, cem_plan
    from wfcrl_b200.vector_env import VecWindFarmEnv

    _env_vars(monkeypatch, True)
    B, H = 64, 4
    env = VecWindFarmEnv("Turb32_Row5_", B, precision=precision, max_num_steps=50)
    env.reset(seed=5)
    T = env.num_turbines
    env.step(_actions(np.random.default_rng(5), (B, T)))
    runs = []
    for _ in range(2):
        gen = torch.Generator(device="cuda")
        gen.manual_seed(123)
        runs.append(cem_plan(env, H, samples=16, iterations=3, gamma=0.9, generator=gen))
    action, ret, seq = runs[0]
    for a, b in zip(runs[0], runs[1]):  # a seeded call repeats exactly
        assert torch.equal(a, b)
    assert action.shape == (B, T) and ret.shape == (B,) and seq.shape == (B, H, T) and ret.dtype == torch.float64
    assert torch.equal(action, seq[:, 0])
    # the return is what a fresh evaluation of the returned sequence gives, and never below the all-zero sequence's
    _, again, _ = best_sequence(env, seq[:, None], gamma=0.9)
    assert torch.equal(again, ret)
    _, zero, _ = best_sequence(env, torch.zeros(B, 1, H, T, device="cuda"), gamma=0.9)
    assert bool((ret >= zero).all())
    # stepping the planned first action gives the row-0 predicted reward
    predicted = env.evaluate_rollouts(seq[:, None].contiguous(), observations=False)[1][:, 0, 0].clone()
    _obs, reward, _term, _trunc, _info = env.step(action)
    assert torch.equal(reward, predicted)
    env.close()
