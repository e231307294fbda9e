"""Action evaluation (wf_evaluate_actions / evaluate_actions / greedy_lookahead): K candidate actions per env evaluated from
the current state without stepping.  Row (b, k) of every output must equal, bit for bit, row b of what wf_step with
candidate k would write on the same handle in the same state, and nothing a step or get_state can see may change."""
import ctypes as C

import numpy as np
import pytest

from tests._util import layout, sample_winds

pytestmark = pytest.mark.gpu

# (precision, strict, vortex table, baked FP32 kernel)
MODES = {
    "f64_table": ("f64", True, True, True),
    "f64_direct": ("f64", True, False, True),
    "f32_strict": ("f32", True, True, True),
    "f32_strict_generic": ("f32", True, True, False),
    "f32_relaxed": ("f32", False, True, True),
}
STATE = ("yaw", "acc", "acc_prev", "num_iter", "num_moves", "nonfinite", "episode", "ambiguous", "ep_return", "ep_len",
         "fin_sum", "fin_sumsq", "fin_n", "fin_len", "ws", "wd", "ws_norm", "shaper_ref", "ti_ambient", "order", "xs", "ys",
         "xi", "yi", "cs", "layout_id", "turbine_count")
OUTPUTS = ("yaw", "wind_speed", "wind_direction", "power", "load", "reward", "freewind", "truncated")


def _env_vars(monkeypatch, table, baked=True):
    if table:
        monkeypatch.delenv("WFCRL_B200_NO_VTAB", raising=False)
    else:
        monkeypatch.setenv("WFCRL_B200_NO_VTAB", "1")
    if baked:
        monkeypatch.delenv("WFCRL_B200_NO_BAKED", raising=False)
    else:
        monkeypatch.setenv("WFCRL_B200_NO_BAKED", "1")


def _actions(rng, shape, continuous=True):
    import torch

    a = rng.uniform(-6, 6, shape) if continuous else rng.integers(0, 3, shape)
    return torch.as_tensor(a.astype(np.float32), device="cuda")


def _warm(fb, rng, steps=3, continuous=True):
    """A few random steps and a wind change, so that acc, num_moves, shaper_ref and ws_norm (!= ws) are non-trivial."""
    import torch

    for _ in range(steps):
        fb.step(_actions(rng, (fb.B, fb.T), continuous))
    ws = torch.as_tensor(np.clip(fb.get_state("ws") + rng.uniform(-1, 1, fb.B), 3, 28), device="cuda")
    fb.update_wind(ws, torch.as_tensor(fb.get_state("wd"), device="cuda"))


def _check_against_step(fb, act):
    """The reference loop: state_dict -> step(act[:, k]) -> load_state_dict, with an evaluation in the same state before each
    step (load_state_dict leaves the vortex table stale: both routes are covered).  Returns the number of flagged rows."""
    import torch

    K = act.shape[1]
    flagged = 0
    for k in range(K):
        ev = {key: v.clone() for key, v in fb.evaluate_actions(act).items()}
        sd = fb.state_dict()
        out = fb.step(act[:, k].contiguous())
        torch.cuda.synchronize()
        for key in OUTPUTS:
            assert torch.equal(ev[key][:, k], out[key]), (k, key)
        ref_amb = fb.get_state("ambiguous").astype(bool)
        assert np.array_equal(ev["ambiguous"][:, k].cpu().numpy(), ref_amb), k
        flagged += int(ref_amb.sum())
        fb.load_state_dict(sd)
    return flagged


@pytest.mark.parametrize("K", [1, 6])
@pytest.mark.parametrize("name", ["Ablaincourt_", "Turb32_Row5_", "HornsRev1_"])
@pytest.mark.parametrize("mode", list(MODES))
def test_equals_step(cuda_device, monkeypatch, mode, name, K):
    from wfcrl_b200.backend import FlorisBatch

    precision, strict, table, baked = MODES[mode]
    _env_vars(monkeypatch, table, baked)
    lx, ly = layout(name)
    T, B = len(lx), 64
    fb = FlorisBatch(lx, ly, B, precision=precision, kernel="fast", max_iter=1000, strict=strict, reward_shaper="step")
    ws, wd = sample_winds(B, seed=T + K, tie_every=5)
    fb.reset(ws, wd, host_trig=True)
    rng = np.random.default_rng(K)
    _warm(fb, rng)
    _check_against_step(fb, _actions(rng, (B, K, T)))
    fb.close()


# env semantics: (FlorisBatch keyword arguments, what the case needs)
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
    T, B, K = len(lx), 64, 5
    kw = SEMANTICS[case]
    continuous = kw.get("continuous_control", True)
    fb = FlorisBatch(lx, ly, B, precision=precision, kernel="fast", max_iter=1000, **kw)
    ws, wd = sample_winds(B, seed=len(case))
    fb.reset(ws, wd, host_trig=True)
    rng = np.random.default_rng(len(case))
    _warm(fb, rng, continuous=continuous)
    act = _actions(rng, (B, K, T), continuous)
    if case == "step_pct":
        assert np.all(fb.get_state("shaper_ref") != 0)
    if case == "constraint":  # the accumulator of half the envs is far over the limit: their actions are zeroed
        acc = fb.get_state("acc")
        acc[: B // 2] = 1e4
        fb.set_state("acc", acc)
        yaw0 = torch.as_tensor(fb.get_state("yaw"), device="cuda")
        ev = fb.evaluate_actions(act)
        torch.cuda.synchronize()
        moved = ev["yaw"].double() != yaw0[:, None, :]
        assert not bool(moved[: B // 2].any()) and bool(moved[B // 2:].any())
    if case == "multi_agent":  # per-agent staleness: acc_prev differs from acc
        acc_prev = fb.get_state("acc_prev")
        acc_prev[::2] = 1e4
        fb.set_state("acc_prev", acc_prev)
        assert not np.array_equal(fb.get_state("acc"), fb.get_state("acc_prev"))
    _check_against_step(fb, act)
    fb.close()


def test_strict_flagged_candidates_equal_the_resolve(cuda_device, monkeypatch):
    import torch

    from wfcrl_b200.backend import FlorisBatch

    _env_vars(monkeypatch, True)
    lx, ly = layout("Turb32_Row5_")
    T, B, K = len(lx), 512, 4
    rng = np.random.default_rng(3)
    ws, wd = sample_winds(B, seed=3)
    ws[: B // 2] = rng.uniform(3.0, 4.5, B // 2)  # over-sample the foot of the power curve
    fb = FlorisBatch(lx, ly, B, precision="f32", kernel="fast", max_iter=1000, reward_shaper="step")
    fb.reset(ws, wd, host_trig=True)
    for _ in range(2):
        fb.step(_actions(rng, (B, T)))
    act = _actions(rng, (B, K, T))
    amb = fb.evaluate_actions(act)["ambiguous"].clone()
    torch.cuda.synchronize()
    assert int(amb.sum()) > 0
    assert _check_against_step(fb, act) == int(amb.sum())
    fb.close()


@pytest.mark.parametrize("mode", ["f64_table", "f32_strict"])
def test_truncation_resets_nothing(cuda_device, monkeypatch, mode):
    import torch

    from wfcrl_b200.backend import FlorisBatch

    precision, strict, table, _ = MODES[mode]
    _env_vars(monkeypatch, table)
    lx, ly = layout("Turb6_Row2_")
    T, B, K, max_iter = len(lx), 128, 3, 8
    ws, wd = sample_winds(B, seed=4)
    twins = [FlorisBatch(lx, ly, B, precision=precision, kernel="fast", max_iter=max_iter, strict=strict,
                         reward_shaper="step") for _ in range(2)]
    rng = np.random.default_rng(4)
    acts = [_actions(rng, (B, T)) for _ in range(4)]
    for fb in twins:
        fb.reset(ws, wd, host_trig=True)
        fb.set_autoreset(True, seed=9)
        fb.step(acts[0])
        fb.set_state("num_iter", max_iter - 1)
    ev = twins[0].evaluate_actions(_actions(rng, (B, K, T)))
    torch.cuda.synchronize()
    assert bool(ev["truncated"].all())
    for fb in twins:  # a no-op unless something was marked for reset
        fb.autoreset_finish()
    torch.cuda.synchronize()
    for name in STATE:
        assert np.array_equal(twins[0].get_state(name), twins[1].get_state(name)), name
    for act in acts[1:]:
        outs = [{k: v.clone() for k, v in fb.step(act).items()} for fb in twins]
        for fb in twins:
            fb.autoreset_finish()
        torch.cuda.synchronize()
        for key in OUTPUTS:
            assert torch.equal(outs[0][key], outs[1][key]), key
        for name in STATE:
            assert np.array_equal(twins[0].get_state(name), twins[1].get_state(name)), name
    for fb in twins:
        fb.close()


@pytest.mark.parametrize("mode", ["f64_table", "f32_strict"])
def test_state_untouched(cuda_device, monkeypatch, mode):
    import torch

    from wfcrl_b200.backend import FlorisBatch

    precision, strict, table, _ = MODES[mode]
    _env_vars(monkeypatch, table)
    lx, ly = layout("Turb32_Row5_")
    T, B, K = len(lx), 512, 3
    rng = np.random.default_rng(8)
    ws, wd = sample_winds(B, seed=8)
    ws[: B // 2] = rng.uniform(3.0, 4.5, B // 2)  # a strict handle flags envs at the foot of the power curve
    kw = dict(precision=precision, kernel="fast", max_iter=20, strict=strict, reward_shaper="step")
    twins = [FlorisBatch(lx, ly, B, **kw) for _ in range(2)]
    for fb in twins:
        fb.reset(ws, wd, host_trig=True)
        fb.set_autoreset(True, seed=5)
    acts = [_actions(rng, (B, T)) for _ in range(4)]
    for fb in twins:
        fb.step(acts[0])
    torch.cuda.synchronize()
    if precision == "f32":
        assert twins[0].get_state("ambiguous").sum() > 0  # the previous step re-solved envs
    before = {name: twins[0].get_state(name).tobytes() for name in STATE}
    cand = _actions(rng, (B, K, T))
    twins[0].evaluate_actions(cand)
    torch.cuda.synchronize()
    for name in STATE:
        assert twins[0].get_state(name).tobytes() == before[name], name
    for act in acts[1:]:
        outs = [{k: v.clone() for k, v in fb.step(act).items()} for fb in twins]
        twins[0].evaluate_actions(cand)
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
    T, B, K = max(counts), 128, 4
    pool = FlorisBatch(*farms[-1], B, precision=precision, kernel="fast", max_iter=1000, reward_shaper="step")
    pool.set_mixed_layouts([f[0] for f in farms], [f[1] for f in farms])
    ids = np.arange(B) % 2
    pool.assign_layouts(None, ids)
    ws, wd = sample_winds(B, seed=2)
    pool.reset(ws, wd, host_trig=True)
    rng = np.random.default_rng(2)
    _warm(pool, rng)
    act = rng.uniform(-6, 6, (B, K, T)).astype(np.float32)
    for b in range(B):
        act[b, :, counts[ids[b]]:] = np.nan  # ignored
    act = torch.as_tensor(act, device="cuda")
    ev = pool.evaluate_actions(act)
    torch.cuda.synchronize()
    for lay, n in enumerate(counts):
        rows = torch.as_tensor(np.flatnonzero(ids == lay), device="cuda")
        for key in ("yaw", "wind_speed", "wind_direction", "power", "load"):
            assert not bool(ev[key][rows][:, :, n:].any()), key
    _check_against_step(pool, act)
    pool.close()


def test_launch_count_interleaving_and_refusals(cuda_device, monkeypatch):
    import torch

    from wfcrl_b200.backend import FlorisBatch
    from wfcrl_b200.vector_env import VecWindFarmEnv

    _env_vars(monkeypatch, True)
    lx, ly = layout("Turb32_Row5_")
    T, B = len(lx), 256
    rng = np.random.default_rng(7)
    act = _actions(rng, (B, 4, T))
    yaw = torch.as_tensor(rng.uniform(-40, 40, (B, 4, T)), device="cuda")
    ws, wd = sample_winds(B, seed=7)
    ws[: B // 2] = rng.uniform(3.0, 4.5, B // 2)  # a strict handle flags candidates: the shared fix list and yaw rows are used
    for precision, strict, launches in (("f64", True, 1), ("f32", True, 2), ("f32", False, 1)):
        kw = dict(precision=precision, kernel="fast", max_iter=1000, strict=strict)
        fb, ref = FlorisBatch(lx, ly, B, **kw), FlorisBatch(lx, ly, B, **kw)
        for h in (fb, ref):
            h.reset(ws, wd, host_trig=True)
        expect = {k: v.clone() for k, v in ref.evaluate_actions(act).items()}
        expect_yaw = {k: v.clone() for k, v in ref.evaluate_yaw(yaw).items()}
        torch.cuda.synchronize()
        if precision == "f32" and strict:
            assert int(expect["ambiguous"][:, 0].sum()) > 0 and int(expect_yaw["ambiguous"][:, 0].sum()) > 0
        # the two entry points share the scratch: interleaved with growing K, each result equals a fresh one
        for K in (1, 2, 3, 4):
            got = {k: v[:, :K].clone() for k, v in fb.evaluate_actions(act[:, :K].contiguous()).items()}
            got_yaw = {k: v.clone() for k, v in fb.evaluate_yaw(yaw[:, :K].contiguous()).items()}
            torch.cuda.synchronize()
            for key in got:
                assert torch.equal(got[key], expect[key][:, :K]), (precision, K, key)
            for key in got_yaw:
                assert torch.equal(got_yaw[key], expect_yaw[key][:, :K]), (precision, K, key)
        for K in (3, 1, 2):
            n0 = fb.launch_count()
            fb.evaluate_actions(act[:, :K].contiguous())
            assert fb.launch_count() - n0 == launches, (precision, strict, K)
        lib, h, st = fb.lib, fb.handle, fb._stream()
        p = C.c_void_p(act.data_ptr())
        out = C.byref(fb._out_struct)
        n0 = fb.launch_count()
        assert lib.wf_evaluate_actions(h, p, 0, out, None, st) == 1 and b"K" in lib.wf_last_error()
        assert lib.wf_evaluate_actions(h, p, -1, out, None, st) == 1
        assert lib.wf_evaluate_actions(h, None, 1, out, None, st) == 1 and b"NULL" in lib.wf_last_error()
        assert lib.wf_evaluate_actions(h, p, 1, None, None, st) == 1 and b"NULL" in lib.wf_last_error()
        assert lib.wf_evaluate_actions(h, p, 2**31 // B + 1, out, None, st) == 1 and b"2^31" in lib.wf_last_error()
        assert fb.launch_count() == n0
        with pytest.raises(ValueError):
            fb.evaluate_actions(torch.zeros(B, 0, T, dtype=torch.float32, device="cuda"))
        with pytest.raises(ValueError):
            fb.evaluate_actions(torch.zeros(B, 2, T + 1, dtype=torch.float32, device="cuda"))
        with pytest.raises(TypeError):
            fb.evaluate_actions(act.double())
        with pytest.raises(TypeError):
            fb.evaluate_actions(act.cpu())
        fb.close()
        ref.close()
    basic = FlorisBatch(lx, ly, B, precision="f64", kernel="basic", max_iter=1000)
    n0 = basic.launch_count()
    with pytest.raises(Exception, match="WF_KERNEL_FAST"):
        basic.evaluate_actions(act)
    assert basic.launch_count() == n0
    basic.close()
    env = VecWindFarmEnv("Turb6_Row2_", B, precision="f64")
    with pytest.raises(AssertionError):
        env.evaluate_actions(act)
    env.close()
    series = np.stack([np.full(20, 8.0), np.linspace(260, 280, 20)], 1)
    env = VecWindFarmEnv("Turb6_Row2_", B, precision="f64", wind_time_series=series)
    env.reset(seed=0)
    with pytest.raises(ValueError, match="time-series"):
        env.evaluate_actions(act)
    env.close()


@pytest.mark.parametrize("mode", ["f64_table", "f32_strict"])
def test_first_call_on_a_non_blocking_stream(cuda_device, monkeypatch, mode):
    import torch

    from wfcrl_b200.backend import FlorisBatch

    precision, strict, table, _ = MODES[mode]
    _env_vars(monkeypatch, table)
    lx, ly = layout("Turb32_Row5_")
    T, B, K = len(lx), 1024, 5
    rng = np.random.default_rng(12)
    ws, wd = sample_winds(B, seed=12)
    ws[: B // 2] = rng.uniform(3.0, 4.5, B // 2)  # flagged candidates on a strict handle
    twins = [FlorisBatch(lx, ly, B, precision=precision, kernel="fast", max_iter=1000, strict=strict) for _ in range(2)]
    for fb in twins:
        fb.reset(ws, wd, host_trig=True)
    act = _actions(rng, (B, K, T))
    ref = {k: v.clone() for k, v in twins[1].evaluate_actions(act).items()}
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        got = {k: v.clone() for k, v in twins[0].evaluate_actions(act).items()}
    torch.cuda.synchronize()
    if precision == "f32":
        assert int(ref["ambiguous"].sum()) > 0
    for key in ref:
        assert torch.equal(got[key], ref[key]), key
    for fb in twins:
        fb.close()


@pytest.mark.parametrize("copy_outputs", [False, True])
def test_vector_env_against_step(cuda_device, monkeypatch, copy_outputs):
    import torch

    from wfcrl_b200.vector_env import VecWindFarmEnv

    _env_vars(monkeypatch, True)
    B, K = 32, 4
    kw = dict(precision="f32", pad_turbines=True, copy_outputs=copy_outputs, max_num_steps=50)
    envs = [VecWindFarmEnv(["Turb6_Row2_", "Ablaincourt_"], B, **kw) for _ in range(2)]
    for env in envs:
        env.reset(seed=3)
    T = envs[0].num_turbines
    rng = np.random.default_rng(3)
    for k in range(K):
        cand = _actions(rng, (B, K, T))
        obs, reward, term, trunc, info = envs[0].evaluate_actions({"yaw": cand})
        obs = {key: v.clone() for key, v in obs.items()}
        reward, trunc, info = reward.clone(), trunc.clone(), {key: v.clone() for key, v in info.items()}
        assert obs["turbine_mask"].shape == (B, K, T) and not bool(term.any())
        ref = envs[1].step(cand[:, k])
        for key in ("yaw", "freewind_measurements", "wind_speed", "wind_direction", "turbine_mask"):
            assert torch.equal(obs[key][:, k], ref[0][key]), key
        assert torch.equal(reward[:, k], ref[1]) and torch.equal(trunc[:, k], ref[3])
        for key in ("power", "load"):
            assert torch.equal(info[key][:, k], ref[4][key]), key
        envs[0].step(cand[:, k])  # the twins stay in step
    views = envs[0].evaluate_actions(cand)
    shared = views[0]["yaw"].data_ptr() == envs[0].backend.evaluate_actions(cand)["yaw"].data_ptr()
    assert shared != copy_outputs
    for env in envs:
        env.close()


def test_multi_agent_split(cuda_device, monkeypatch):
    import torch

    from wfcrl_b200.vector_env import VecMAWindFarmEnv

    _env_vars(monkeypatch, True)
    B, K = 16, 3
    env = VecMAWindFarmEnv("Turb6_Row2_", B, precision="f64")
    env.reset(seed=1)
    T = env.num_turbines
    cand = _actions(np.random.default_rng(1), (B, K, T))
    joint = {key: v.clone() for key, v in env.backend.evaluate_actions(cand).items()}
    per_agent = {a: {"yaw": cand[:, :, i]} for a, i in env.agent_name_mapping.items()}
    for actions in (cand, per_agent):
        obs, reward, term, trunc, info = env.evaluate_actions(actions)
        for a, i in env.agent_name_mapping.items():
            assert torch.equal(obs[a]["yaw"], joint["yaw"][:, :, i])
            assert torch.equal(obs[a]["wind_speed"], joint["wind_speed"][:, :, i])
            assert torch.equal(reward[a], joint["reward"]) and torch.equal(trunc[a], joint["truncated"].bool())
            assert torch.equal(info[a]["power"], joint["power"][:, :, i])
            assert torch.equal(info[a]["load"], joint["load"][:, :, i])
    env.close()


@pytest.mark.parametrize("precision", ["f64", "f32"])
def test_greedy_lookahead_rollout(cuda_device, monkeypatch, precision):
    """Two episodes with auto-reset: the reward step returns for the greedy action is the predicted one, bit for bit, and
    no candidate was predicted to do better."""
    import torch

    from wfcrl_b200.planning import greedy_lookahead
    from wfcrl_b200.vector_env import VecWindFarmEnv

    _env_vars(monkeypatch, True)
    B, K, steps = 64, 6, 5
    env = VecWindFarmEnv("Turb32_Row5_", B, precision=precision, max_num_steps=steps, reward_shaper=None)
    env.reset(seed=11)
    rng = np.random.default_rng(11)
    truncations = 0
    for _ in range(2 * steps):
        cand = _actions(rng, (B, K, env.num_turbines))
        action, predicted, index = greedy_lookahead(env, cand)
        all_rewards = env.evaluate_actions(cand)[1].clone()
        assert torch.equal(all_rewards.gather(1, index[:, None])[:, 0], predicted)
        assert bool(((predicted[:, None] >= all_rewards) | all_rewards.isnan()).all())
        assert torch.equal(action, cand[torch.arange(B, device="cuda"), index])
        _obs, reward, _term, trunc, _info = env.step(action)
        assert torch.equal(reward, predicted)
        truncations += int(trunc.sum())
    assert truncations == 2 * B
    env.close()
