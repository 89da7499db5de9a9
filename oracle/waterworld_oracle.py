"""CPU oracle for the MAWaterWorld reset()/step() hot path (TEST INFRASTRUCTURE, float64 NumPy).

This is a restatement -- not a copy -- of the algorithm in the reference file
``madrl_environments/pursuit/waterworld.py`` (cited per function below, ``ww:LINE``).  State is
held as plain arrays instead of ``Archea`` objects.  It is pinned against the real reference
classes (imported through ``oracle/refshim.py``; their runs recorded in ``tests/golden/ref_ww_oracle_*.npz``) by
``tests/test_waterworld_oracle.py`` and by
the golden vectors in ``tests/golden`` produced by ``oracle/make_golden.py``; on identical
injected random streams the two agree bit for bit in float64.

Only ``tests/``, ``__graft_entry__.smoke()`` and ``bench.py``'s CPU-baseline legs may import it.
The product package ``madrl_b200`` never does.
"""
import numpy as np
import scipy.spatial.distance as ssd

from .philox import Stream


class WaterworldOracle(object):
    """One MAWaterWorld instance.  Constructor arguments mirror ww:77-81."""

    timestep_limit = 1000  # ww:124-126

    def __init__(self, n_pursuers, n_evaders, n_coop=2, n_poison=10, radius=0.015,
                 obstacle_radius=0.2, obstacle_loc=np.array([0.5, 0.5]), ev_speed=0.01,
                 poison_speed=0.01, n_sensors=30, sensor_range=0.2, action_scale=0.01,
                 poison_reward=-1., food_reward=1., encounter_reward=.05, control_penalty=-.5,
                 reward_mech='local', addid=True, speed_features=True, rng=None):
        self.Np, self.Ne, self.Npo, self.K = n_pursuers, n_evaders, n_poison, n_sensors
        self.n_coop = n_coop
        self.radius = radius
        self.obstacle_radius = obstacle_radius
        self.obstacle_loc = None if obstacle_loc is None else np.asarray(obstacle_loc, float)
        self.ev_speed, self.poison_speed = ev_speed, poison_speed
        self.sensor_range = sensor_range
        self.action_scale = action_scale
        self.poison_reward, self.food_reward = poison_reward, food_reward
        self.encounter_reward, self.control_penalty = encounter_reward, control_penalty
        self.reward_mech, self.addid, self.speed_features = reward_mech, addid, speed_features
        # radii, ww:108-118
        self.r_p, self.r_e, self.r_po = radius, radius * 2, radius * 3 / 4
        # sensor unit vectors, ww:29-31
        ang = np.linspace(0., 2. * np.pi, n_sensors + 1)[:-1]
        self.S = np.c_[np.cos(ang), np.sin(ang)]
        self.obs_dim = n_sensors * (7 if speed_features else 4) + 2 + (1 if addid else 0)  # ww:18-24
        self.np_random = rng if rng is not None else Stream(0, 0)
        self.t = 0
        self.obst = None
        self.px = self.pv = self.ex = self.ev = self.ox = self.ov = None

    # ------------------------------------------------------------------ state access (tests)
    def get_state(self):
        return dict(px=self.px.copy(), pv=self.pv.copy(), ex=self.ex.copy(), ev=self.ev.copy(),
                    ox=self.ox.copy(), ov=self.ov.copy(), obst=self.obst.copy(), t=self.t,
                    counter=getattr(self.np_random, 'counter', 0))

    def set_state(self, s):
        for k in ('px', 'pv', 'ex', 'ev', 'ox', 'ov', 'obst'):
            setattr(self, k, np.array(s[k], dtype=np.float64))
        self.t = int(s['t'])
        if 'counter' in s and hasattr(self.np_random, 'counter'):
            self.np_random.counter = int(s['counter'])

    def seed(self, seed=None, env_id=0):
        self.np_random = Stream(0 if seed is None else seed, env_id)
        return [seed]

    # ------------------------------------------------------------------ ww:139-142
    def _respawn(self, x, r):
        while ssd.cdist(x[None, :], self.obst) <= r * 2 + self.obstacle_radius:
            x = self.np_random.rand(2)
        return x

    # ------------------------------------------------------------------ ww:144-172
    def reset(self):
        rs = self.np_random
        self.t = 0
        if self.obstacle_loc is None:
            self.obst = rs.rand(1, 2)
        else:
            self.obst = self.obstacle_loc[None, :].copy()
        self.px = np.zeros((self.Np, 2)); self.pv = np.zeros((self.Np, 2))
        self.ex = np.zeros((self.Ne, 2)); self.ev = np.zeros((self.Ne, 2))
        self.ox = np.zeros((self.Npo, 2)); self.ov = np.zeros((self.Npo, 2))
        for i in range(self.Np):
            self.px[i] = self._respawn(rs.rand(2), self.r_p)
        for i in range(self.Ne):
            self.ex[i] = self._respawn(rs.rand(2), self.r_e)
            self.ev[i] = (rs.rand(2) - 0.5) * self.ev_speed
        for i in range(self.Npo):
            self.ox[i] = self._respawn(rs.rand(2), self.r_po)
            self.ov[i] = (rs.rand(2) - 0.5) * self.ev_speed  # ww:170 uses ev_speed, not poison_speed
        return self.step(np.zeros((self.Np, 2)))[0]

    # ------------------------------------------------------------------ ww:64-72
    def _sensed(self, i, objx, same=False):
        rel = objx - self.px[i][None, :]
        sv = self.S.dot(rel.T)
        bad = (sv < 0) | (sv > self.sensor_range) | (
            (rel ** 2).sum(axis=1)[None, :] - sv ** 2 > self.r_p ** 2)
        sv[bad] = np.inf
        if same:
            sv[:, i] = np.inf
        return sv

    # ------------------------------------------------------------------ ww:180-193
    @staticmethod
    def _caught(coll, n_coop):
        caught = np.where(coll.sum(axis=0) >= n_coop)[0]
        who = np.where(coll[:, caught] >= 1)[0]
        return caught, who

    # ------------------------------------------------------------------ ww:312-353
    def _features(self, sv_all, objv):
        """sv_all [Np,K,N] -> (dist [Np,K], speed [Np,K] or None, idx, mask)."""
        idx = np.argmin(sv_all, axis=2)                                        # first minimum
        d = np.take_along_axis(sv_all, idx[:, :, None], axis=2)[:, :, 0]      # ww:195-201
        mask = np.isfinite(d)
        dist = np.where(mask, d, 0.0)
        speed = None
        if objv is not None and self.speed_features:                           # ww:203-218
            speed = np.zeros((self.Np, self.K))
            for i in range(self.Np):
                rv = self.S.dot((objv - self.pv[i][None, :]).T)               # [K,N]
                speed[i] = np.where(mask[i], rv[np.arange(self.K), idx[i]], 0.0)
        return dist, speed

    # ------------------------------------------------------------------ ww:220-436
    def step(self, action):
        Np, Ne, Npo = self.Np, self.Ne, self.Npo
        act = np.asarray(action, dtype=np.float64).reshape((Np, 2)) * self.action_scale  # ww:221-224
        rewards = np.zeros(Np)
        # integrate pursuers, ww:229-231
        self.pv = self.pv + act
        self.px = self.px + self.pv
        # control penalty, ww:234-237
        if self.reward_mech == 'global':
            rewards += self.control_penalty * (act ** 2).sum()
        else:
            rewards += self.control_penalty * (act ** 2).sum(axis=1)
        # walls stop pursuers, ww:240-245
        clipped = np.clip(self.px, 0, 1)
        self.pv[self.px != clipped] = 0
        self.px = clipped
        # obstacle rebound (velocity only), ww:247-270
        hit = ssd.cdist(self.px, self.obst)[:, 0] <= self.r_p + self.obstacle_radius
        self.pv[hit] = -1 / 2 * self.pv[hit]
        hit = ssd.cdist(self.ex, self.obst)[:, 0] <= self.r_e + self.obstacle_radius
        self.ev[hit] = -1 / 2 * self.ev[hit]
        hit = ssd.cdist(self.ox, self.obst)[:, 0] <= self.r_po + self.obstacle_radius
        self.ov[hit] = -1 * self.ov[hit]
        # collisions, ww:278-293 (evader/poison positions are those left by the previous step)
        coll_ev = ssd.cdist(self.px, self.ex) <= self.r_p + self.r_e
        ev_caught, who_ev = self._caught(coll_ev, self.n_coop)
        coll_po = ssd.cdist(self.px, self.ox) <= self.r_p + self.r_po
        po_caught, who_po = self._caught(coll_po, 1)
        # sensing, ww:297-309
        sv_ob = np.array([self._sensed(i, self.obst) for i in range(Np)])
        sv_ev = np.array([self._sensed(i, self.ex) for i in range(Np)])
        sv_po = np.array([self._sensed(i, self.ox) for i in range(Np)])
        sv_pu = np.array([self._sensed(i, self.px, same=True) for i in range(Np)])
        f_ob, _ = self._features(sv_ob, None)
        f_ev, s_ev = self._features(sv_ev, self.ev)
        f_po, s_po = self._features(sv_po, self.ov)
        f_pu, s_pu = self._features(sv_pu, self.pv)
        # respawn caught objects, ww:358-374
        rs = self.np_random
        for j in ev_caught:
            self.ex[j] = self._respawn(rs.rand(2), self.r_e)
            self.ev[j] = (rs.rand(2) - 0.5) * self.ev_speed
        for j in po_caught:
            self.ox[j] = self._respawn(rs.rand(2), self.r_po)
            self.ov[j] = (rs.rand(2) - 0.5) * self.poison_speed
        # rewards, ww:376-385 (fancy-index += credits a pursuer at most once per category)
        ev_enc, who_enc = self._caught(coll_ev, 1)
        if self.reward_mech == 'global':
            rewards += (len(ev_caught) * self.food_reward + len(po_caught) * self.poison_reward +
                        len(ev_enc) * self.encounter_reward)
        else:
            rewards[who_ev] += self.food_reward
            rewards[who_po] += self.poison_reward
            rewards[who_enc] += self.encounter_reward
        # feature concat, ww:388-395 (feature-major, sensor-minor)
        if self.speed_features:
            feats = np.c_[f_ob, f_ev, s_ev, f_po, s_po, f_pu, s_pu]
        else:
            feats = np.c_[f_ob, f_ev, f_po, f_pu]
        # evaders / poison drift; bounce only if BOTH coordinates left [0,1], ww:397-409
        self.ex = self.ex + self.ev
        flip = np.all(self.ex != np.clip(self.ex, 0, 1), axis=1)
        self.ev[flip] = -1 * self.ev[flip]
        self.ox = self.ox + self.ov
        flip = np.all(self.ox != np.clip(self.ox, 0, 1), axis=1)
        self.ov[flip] = -1 * self.ov[flip]
        # obs assembly, ww:411-428
        obs = []
        for i in range(Np):
            tail = [float(coll_ev[i].sum() > 0), float(coll_po[i].sum() > 0)]
            if self.addid:
                tail.append(i + 1)
            obs.append(np.concatenate([feats[i], tail]))
        self.t += 1                                                            # ww:433
        done = self.t >= self.timestep_limit
        return obs, rewards, done, dict(evcatches=len(ev_caught), pocatches=len(po_caught))
