"""Post-processing passes: oracle vs the REAL reference wrappers (CPU; their outputs recorded,
tests/reference_record.py) and CUDA kernels vs oracle (GPU)."""
import numpy as np
import pytest

from oracle import postproc_oracle as po
from oracle.postproc_oracle import StandardizeEnv, discount_cumsum, episode_stats_env, frame_stack_env, gae_env
from reference_record import digest, recorded


class ScriptedEnv(object):
    """Minimal AbstractMAEnv stand-in that replays given observations / rewards."""

    def __init__(self, obs0, obs, rew, spaces_mod):
        self.obs0, self.obs_seq, self.rew_seq, self.t = obs0, obs, rew, 0
        A, D = obs0.shape

        class Ag(object):
            observation_space = spaces_mod.Box(low=-10, high=10, shape=(D,))
            action_space = spaces_mod.Box(low=-1, high=1, shape=(2,))
        self.agents = [Ag() for _ in range(A)]
        self.reward_mech = 'local'

    def seed(self, s=None):
        return [s]

    def reset(self):
        return [o.copy() for o in self.obs0]

    def step(self, a):
        o, r = self.obs_seq[self.t], self.rew_seq[self.t]
        self.t += 1
        return [x.copy() for x in o], list(r), False, {}


def test_oracles_equal_reference_wrappers():
    """ObservationBuffer and StandardizedEnv of the reference around a scripted env, against the oracle's
    frame stack and standardiser, bit for bit (reference side recorded)."""
    rs = np.random.RandomState(0)
    T, A, D, B = 40, 3, 5, 4
    obs0, obs, rew = rs.randn(A, D), rs.randn(T, A, D), rs.randn(T, A)

    def reference():
        from oracle.refshim import install
        install()
        import gym.spaces as spaces
        import madrl_environments as me
        me.ent = None  # noqa  (ObservationBuffer.agents has a typo'd name; not used here)
        w = me.ObservationBuffer.__new__(me.ObservationBuffer)
        w._unwrapped = ScriptedEnv(obs0, obs, rew, spaces)
        w._buffer_size = B
        w._buffer = [np.zeros((D, B)) for _ in range(A)]
        out = dict(buffer0=np.array(w.reset()), buffer=np.array([np.array(w.step(None)[0]) for _ in range(T)]))
        s = me.StandardizedEnv(ScriptedEnv(obs0, obs, rew, spaces), scale_reward=0.5, enable_obsnorm=True,
                               enable_rewnorm=True, obs_alpha=0.05, rew_alpha=0.02)
        out["std0"] = np.array(s.reset())
        steps = [s.step(None) for _ in range(T)]
        return dict(out, std_obs=np.array([np.array(x[0]) for x in steps]),
                    std_rew=np.array([np.array(x[1]) for x in steps]))
    ref = recorded("postproc_wrappers", reference)
    # ObservationBuffer
    o0, o = frame_stack_env(obs0, obs, np.zeros(T, bool), B)
    assert np.array_equal(ref["buffer0"], o0) and np.array_equal(ref["buffer"], o)
    # StandardizedEnv
    mine = StandardizeEnv(A, D, 0.5, True, True, 0.05, 0.02)
    assert np.array_equal(ref["std0"], mine.obs(obs0))
    for t in range(T):
        assert np.array_equal(ref["std_obs"][t], mine.obs(obs[t]))
        assert np.array_equal(ref["std_rew"][t], mine.rew(rew[t]))


def test_episode_stats_oracle_equals_reference_wrapper():
    """The episode statistics DiagnosticsWrapper logs, against the oracle's (reference side recorded)."""
    rs = np.random.RandomState(3)
    T, A, D = 60, 3, 2
    obs0, obs, rew = rs.randn(A, D), rs.randn(T, A, D), rs.randn(T, A)
    done = np.zeros(T, bool)
    done[[7, 30]] = True

    def reference():
        from oracle.refshim import install
        install()
        import gym.spaces as spaces
        import madrl_environments as me

        class Env(ScriptedEnv):
            def step(self, a):
                o, r, _, i = ScriptedEnv.step(self, a)
                return o, np.asarray(r), bool(done[self.t - 1]), i
        w = me.DiagnosticsWrapper(Env(obs0, obs, rew, spaces), discount=0.9, max_traj_len=12, log_interval=10 ** 9)
        w.reset()
        got = []
        for t in range(T):
            _, _, _, log = w.step(None)
            if 'global/episode_length' in log:
                got.append((t, [log['global/episode_reward_agent%d' % a] for a in range(A)],
                            log['global/episode_avg_reward'], log['global/episode_disc_return'],
                            log['global/episode_length']))
        return {k: np.array([g[j] for g in got]) for j, k in enumerate(("t", "agent", "avg", "disc", "length"))}
    ref = recorded("postproc_episode_stats", reference)
    got = list(zip(*(ref[k] for k in ("t", "agent", "avg", "disc", "length"))))
    mine = episode_stats_env(rew, done, 0.9, 12)
    assert len(got) == len(mine) >= 5
    for g, m in zip(got, mine):
        assert g[0] == m[0] and np.array_equal(g[1], m[1]) and g[2] == m[2] and g[3] == m[3] and g[4] == m[4]


def test_batch_statistics_oracle_equals_rllab_functions():
    """center_advantages / shift_advantages_to_positive / explained_variance_1d / discount_cumsum
    of the oracle against the reference's own functions (rllab/rllab/algos/util.py:7-12,
    rllab/rllab/misc/special.py:51-59,107-111), bit for bit (reference side recorded; arrays as digests)."""
    rs = np.random.RandomState(5)
    ns = (1, 2, 17, 4096)
    inputs = [(rs.randn(n) * 3 + 1, rs.randn(n)) for n in ns]
    const = np.full(9, 2.5)
    noise = rs.randn(9), rs.randn(9)

    def reference():
        from oracle.refshim import load_rllab_numeric
        util, special = load_rllab_numeric()
        out = {}
        for n, (adv, y) in zip(ns, inputs):
            out.update({"center%d" % n: digest(util.center_advantages(adv)),
                        "shift%d" % n: digest(util.shift_advantages_to_positive(adv)),
                        "ev%d" % n: special.explained_variance_1d(adv, y),
                        "cumsum%d" % n: digest(special.discount_cumsum(adv, 0.97))})
        return dict(out, ev_const=special.explained_variance_1d(const, const),
                    ev_noise=special.explained_variance_1d(noise[1], const))
    ref = recorded("postproc_batch_statistics", reference)
    for n, (adv, y) in zip(ns, inputs):
        assert np.array_equal(digest(po.center_advantages(adv)), ref["center%d" % n])
        assert np.array_equal(digest(po.shift_advantages_to_positive(adv)), ref["shift%d" % n])
        assert po.explained_variance_1d(adv, y) == ref["ev%d" % n]
        assert np.array_equal(digest(discount_cumsum(adv, 0.97)), ref["cumsum%d" % n])
    assert po.explained_variance_1d(const, const) == ref["ev_const"] == 1
    assert po.explained_variance_1d(noise[0], const) == ref["ev_noise"] == 0


def test_gae_oracle_matches_rllab_formulas():
    rs = np.random.RandomState(1)
    T, A = 30, 2
    rew, val = rs.randn(T, A), rs.randn(T, A)
    done = np.zeros(T, bool)
    done[[9, 19, 29]] = True
    adv, ret = gae_env(rew, val, done, 0.99, 0.95)
    for s, e in ((0, 10), (10, 20), (20, 30)):            # rllab: one call per complete path
        for a in range(A):
            b = np.append(val[s:e, a], 0)
            deltas = rew[s:e, a] + 0.99 * b[1:] - b[:-1]
            assert np.array_equal(adv[s:e, a], discount_cumsum(deltas, 0.99 * 0.95))
            assert np.array_equal(ret[s:e, a], discount_cumsum(rew[s:e, a], 0.99))
    assert ret[9, 0] == rew[9, 0]                          # a path's last step sees no future


def test_to_paths_splits_at_done():
    from madrl_b200.postproc import to_paths
    T, E, A = 6, 2, 2
    done = np.zeros((T, E), np.uint8)
    done[2, 0] = 1
    done[5, 1] = 1
    rew = np.arange(T * E * A, dtype=np.float32).reshape(T, E, A)
    paths = to_paths(np.zeros((T, E, A, 3)), np.zeros((T, E, A, 2)), rew, done, dict(x=np.ones((T, E))))
    lens = sorted((p['env'], p['agent'], len(p['rewards']), p['terminated']) for p in paths)
    assert lens == [(0, 0, 3, False), (0, 0, 3, True), (0, 1, 3, False), (0, 1, 3, True),
                    (1, 0, 6, True), (1, 1, 6, True)]
    assert all(p['env_infos']['x'].shape[0] == len(p['rewards']) for p in paths)


@pytest.mark.gpu
def test_cuda_postproc_matches_oracle():
    import torch
    from madrl_b200.postproc import EpisodeStats, FrameStack, Standardizer, gae
    rs = np.random.RandomState(2)
    T, E, A, D, B = 50, 7, 3, 11, 4
    obs0 = rs.randn(E, A, D).astype(np.float32)
    obs = rs.randn(T, E, A, D).astype(np.float32)
    rew = rs.randn(T, E, A).astype(np.float32)
    val = rs.randn(T, E, A).astype(np.float32)
    last = rs.randn(E, A).astype(np.float32)
    done = (rs.rand(T, E) < 0.1)
    dev = 'cuda'
    d_t = torch.as_tensor(done.astype(np.uint8), device=dev)
    # GAE
    for lv in (None, last):
        adv, ret = gae(torch.as_tensor(rew, device=dev), torch.as_tensor(val, device=dev), d_t, 0.99, 0.95,
                       None if lv is None else torch.as_tensor(lv, device=dev))
        for e in range(E):
            a_o, r_o = gae_env(rew[:, e], val[:, e], done[:, e], 0.99, 0.95, None if lv is None else lv[e])
            assert np.abs(adv[:, e].cpu().numpy() - a_o).max() < 1e-4
            assert np.abs(ret[:, e].cpu().numpy() - r_o).max() < 1e-4
    # frame stack (two consecutive rollouts exercise the carry)
    fs = FrameStack(E, A, D, B, dev)
    st0 = fs.reset(torch.as_tensor(obs0, device=dev)).cpu().numpy()
    o1 = fs.rollout(torch.as_tensor(obs[:20], device=dev), d_t[:20]).cpu().numpy()
    o2 = fs.rollout(torch.as_tensor(obs[20:], device=dev), d_t[20:]).cpu().numpy()
    for e in range(E):
        s0, so = frame_stack_env(obs0[e].astype(np.float64), obs[:, e].astype(np.float64), done[:, e], B)
        assert np.array_equal(st0[e], s0.astype(np.float32))
        assert np.array_equal(np.concatenate([o1, o2])[:, e], so.astype(np.float32))
    # standardizer
    sd = Standardizer(E, A, D, dev, scale_reward=0.5, enable_obsnorm=True, enable_rewnorm=True,
                      obs_alpha=0.05, rew_alpha=0.02)
    x0 = torch.as_tensor(obs0, device=dev).clone()
    sd.obs(x0)
    xo = torch.as_tensor(obs, device=dev).clone()
    xr = torch.as_tensor(rew, device=dev).clone()
    sd.obs(xo)
    sd.rew(xr)
    for e in range(E):
        m = StandardizeEnv(A, D, 0.5, True, True, 0.05, 0.02)
        assert np.abs(m.obs(obs0[e].astype(np.float64)) - x0[e].cpu().numpy()).max() < 1e-5
        for t in range(T):
            assert np.abs(m.obs(obs[t, e].astype(np.float64)) - xo[t, e].cpu().numpy()).max() < 1e-5
            assert np.abs(m.rew(rew[t, e].astype(np.float64)) - xr[t, e].cpu().numpy()).max() < 1e-5
        assert np.abs(m.obs_var - sd.obs_var[e].cpu().numpy()).max() < 1e-12
    # episode statistics (two calls exercise the carry)
    es = EpisodeStats(E, A, dev, discount=0.9, max_traj_len=12)
    r_t = torch.as_tensor(rew, device=dev)
    s1, s2 = es.rollout(r_t[:23], d_t[:23]), es.rollout(r_t[23:], d_t[23:])
    cat = {k: torch.cat([s1[k], s2[k]]).cpu().numpy() for k in s1}
    for e in range(E):
        recs = episode_stats_env(rew[:, e].astype(np.float64), done[:, e], 0.9, 12)
        assert [r[0] for r in recs] == list(np.nonzero(cat['end'][:, e])[0])
        for t, ep_r, avg, disc, length in recs:
            assert np.abs(cat['episode_reward'][t, e] - ep_r).max() < 1e-4
            assert abs(cat['episode_avg_reward'][t, e] - avg) < 1e-4 and abs(cat['episode_disc_return'][t, e] - disc) < 1e-4
            assert cat['episode_length'][t, e] == length


@pytest.mark.gpu
def test_cuda_batch_statistics_match_oracle():
    """madrl_center_advantages_f32 / madrl_moments_f32 against the oracle (float64 NumPy on the same
    float32 inputs); tolerance 1e-5 relative to the value scale, results deterministic."""
    import torch
    from madrl_b200.postproc import center_advantages, explained_variance, moments
    rs = np.random.RandomState(9)
    for shape in ((1,), (3,), (50, 7, 3), (256, 4096, 5)):
        adv = (rs.randn(*shape) * 3 + 1).astype(np.float32)
        ret = rs.randn(*shape).astype(np.float32)
        a_t, r_t = torch.as_tensor(adv, device='cuda'), torch.as_tensor(ret, device='cuda')
        flat = adv.ravel().astype(np.float64)
        for center, positive in ((True, False), (False, True), (True, True), (False, False)):
            want = flat
            if center:
                want = po.center_advantages(want)
            if positive:
                want = po.shift_advantages_to_positive(want)
            got = center_advantages(a_t, center=center, positive=positive)
            assert got.shape == a_t.shape and got.data_ptr() != a_t.data_ptr()
            tol = 1e-5 * max(1.0, np.abs(want).max())
            assert np.abs(got.cpu().numpy().ravel() - want).max() <= tol
            again = center_advantages(a_t, center=center, positive=positive)
            assert torch.equal(got, again)                                 # deterministic reduction
        assert torch.equal(a_t, torch.as_tensor(adv, device='cuda'))       # input untouched
        st = moments(a_t, r_t).cpu().numpy()
        r64 = ret.ravel().astype(np.float64)
        want_st = np.array([flat.mean(), r64.mean(), (r64 - flat).mean(), flat.var(), r64.var(),
                            (r64 - flat).var(), flat.min(), r64.min(), (r64 - flat).min()])
        assert np.allclose(st, want_st, rtol=1e-10, atol=1e-12)
        ev = explained_variance(a_t, r_t)
        assert abs(ev - po.explained_variance_1d(flat, r64)) < 1e-9
    const = torch.full((64,), 2.5, device='cuda')
    assert explained_variance(const, const) == 1
    assert explained_variance(torch.as_tensor(rs.randn(64).astype(np.float32), device='cuda'), const) == 0
    out = center_advantages(const.clone(), inplace=True)                  # zero variance: 0 / 1e-8
    assert torch.equal(out, torch.zeros_like(out))


@pytest.mark.gpu
def test_cuda_pack_paths_matches_host_to_paths():
    """Device-side path packing (csrc/postproc.cu paths_plan / paths_pack kernels, SURVEY 8f row 1:
    dec_rollout-shaped paths, rllab/rllab/sampler/ma_sampler.py:52-100) on a real Waterworld rollout
    with auto-reset, against the host `to_paths` triple loop."""
    import torch
    from madrl_b200 import BatchedMAWaterWorld
    from madrl_b200.postproc import pack_paths, to_paths
    E, T, mpl = 37, 50, 11
    eng = BatchedMAWaterWorld(E, 5, 5, n_coop=1, radius=0.04, seed=3, max_path_length=mpl)
    obs0 = eng.reset().clone()
    act = torch.randn(T, E, 5, 2, device="cuda") * 0.7
    obs, rew, done, info = eng.rollout(act, auto_reset=True)
    infos = dict(evcatches=info[..., 0].contiguous(), pocatches=info[..., 1].contiguous())
    pp = pack_paths(obs, act, rew, done, infos, obs_before=obs0)
    shifted = torch.cat([obs0.unsqueeze(0), obs[:-1]]).cpu()
    want = to_paths(shifted, act.cpu(), rew.cpu(), done.cpu(), {k: v.cpu() for k, v in infos.items()})
    got = pp.to_list()
    assert len(got) == len(want) == len(pp) and len(got) > E * 5 * (T // mpl)
    for g, w in zip(got, want):
        assert (g['env'], g['agent'], g['terminated']) == (w['env'], w['agent'], w['terminated'])
        for k in ('observations', 'actions', 'rewards'):
            assert np.array_equal(g[k], w[k]), k
        for k in infos:
            assert np.array_equal(g['env_infos'][k], w['env_infos'][k])
    one = pp.path(7)                       # zero-copy device views of one path
    assert one['observations'].is_cuda and one['observations'].shape == (int(pp.length[7]), eng.obs_dim)
    # a rollout without any done: one path per (env, agent) covering the whole rollout
    pp2 = pack_paths(obs, act, rew, torch.zeros_like(done), None)
    assert len(pp2) == E * 5 and int(pp2.length.min()) == T
    assert torch.equal(pp2.path(6)['observations'], obs[:, 1, 1])


@pytest.mark.gpu
def test_cuda_terminal_obs_side_tensor_and_standardizer_order():
    """engine.set_terminal_obs + Standardizer.obs(obs, done, terminal_obs) on the GPU: the side tensor
    holds the pre-reset observation of every done step, and the running estimate follows the reference
    order (terminal observation, then reset observation; madrl_environments/__init__.py:283-291)."""
    import torch
    from madrl_b200 import BatchedMAWaterWorld
    from madrl_b200.postproc import Standardizer
    E, T, mpl = 9, 23, 6
    mk = lambda: BatchedMAWaterWorld(E, 5, 5, seed=5, max_path_length=mpl)          # noqa: E731
    a, c = mk(), mk()
    a.reset(), c.reset()
    act = torch.randn(T, E, 5, 2, device="cuda") * 0.5
    term = torch.full((T, E, 5, a.obs_dim), -7.0, device="cuda")
    a.set_terminal_obs(term)
    obs, rew, done, _ = a.rollout(act, auto_reset=True)
    a.set_terminal_obs(None)
    assert int(done.sum()) == E * (T // mpl)
    for t in range(T):                                   # the same envs stepped without auto-reset
        o, _, d, _ = c.rollout(act[t:t + 1], auto_reset=False)
        hit = d[0].bool()
        assert torch.equal(term[t][hit], o[0][hit]) and bool((term[t][~hit] == -7.0).all())
        if hit.any():
            c.reset(mask=d[0])
    std = Standardizer(E, 5, a.obs_dim, "cuda", enable_obsnorm=True, obs_alpha=0.05)
    x, tm = obs.clone(), term.clone()
    std.obs(x, done, tm)
    obs_h, term_h, done_h = obs.cpu().numpy(), term.cpu().numpy(), done.cpu().numpy()
    for e in (0, 4, 8):
        mine = StandardizeEnv(5, a.obs_dim, 1.0, True, False, 0.05, 0.001)
        for t in range(T):
            if done_h[t, e]:
                assert np.abs(mine.obs(term_h[t, e].astype(np.float64)) - tm[t, e].cpu().numpy()).max() < 1e-4
            assert np.abs(mine.obs(obs_h[t, e].astype(np.float64)) - x[t, e].cpu().numpy()).max() < 1e-4, (t, e)
        assert np.abs(mine.obs_mean - std.obs_mean[e].cpu().numpy()).max() < 1e-9
