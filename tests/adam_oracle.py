"""CPU oracle of the Adam baseline (``b2e_step_adam``).  TEST INFRASTRUCTURE ONLY.

``AdamOracle`` is ``BatchedOptEnvOracle.step`` (MultiOptLRs.base_step, oracle/optenv_oracle.py) with the
agent's update ``w - g0 * lr(action)`` replaced by Keras 2.2 ``Adam.get_updates`` (amsgrad=False), restated
from the Keras source and not checked against Keras itself:

    g   = g0 / cnt                  the gradient of the MEAN minibatch loss (g0 is the batch SUM; cnt = 0: func)
    m   = b1 m + (1 - b1) g,        v = b2 v + (1 - b2) g^2        (m = v = 0 before step t = 1)
    a_t = lr sqrt(1 - b2^t) / (1 - b1^t)                           (fp64 of the fp32 constants, rounded to fp32)
    w   = w - a_t m / (sqrt(v) + eps)

Everything after the update (second evaluation, histories, reward, done, info) is the oracle's own step;
info's actions_mean / actions_std are taken over the per-parameter rate a_t / (sqrt(v) + eps).
"""
import numpy as np

from oracle import optenv_oracle as orc

KERAS_DEFAULTS = dict(beta_1=0.9, beta_2=0.999, epsilon=1e-7)
# per action version, the action whose learning rate is exactly 1 (utils_env.py:102-123)
_UNIT_ACTION = {0: 4.0, 1: 1000.0, 2: 0.0, 3: 999000.0}


def adam_alpha(lr, t, beta_1, beta_2):
    """a_t per env (lr [E], t [E]), as the device computes it."""
    b1, b2 = np.float64(np.float32(beta_1)), np.float64(np.float32(beta_2))
    lr = np.asarray(lr, np.float32).astype(np.float64)
    t = np.asarray(t, np.float64)
    return (lr * np.sqrt(1.0 - b2 ** t) / (1.0 - b1 ** t)).astype(np.float32).astype(np.float64)


class AdamOracle:
    """Adam in place of the actions of the MultiOptLRs envs of ``env`` (a ``BatchedOptEnvOracle``).
    ``lr``: float or [E]; m, v [E, P] float64 (natural order) are public, so that a test can load the
    device's moments before a step."""

    def __init__(self, env, lr=1e-3, beta_1=0.9, beta_2=0.999, epsilon=1e-7):
        assert env.cfg.env == 'optlrs'
        self.env = env
        self.lr = np.broadcast_to(np.asarray(lr, np.float32), (env.num_envs,)).copy()
        self.beta_1, self.beta_2, self.epsilon = beta_1, beta_2, epsilon
        self.m = np.zeros((env.num_envs, env.num_params))
        self.v = np.zeros_like(self.m)

    def update(self):
        """(m, v, rate) of this step from the current state; changes nothing."""
        env = self.env
        t = env.current_step + 1                                 # baseenvironment.py:37 counts this step
        g0, _ = env.evaluate()
        if env.spec.kind == 'func':
            g = g0
        else:
            cnt = env.current_batch()[1].astype(np.float64)
            g = g0 / cnt[:, None]
        b1, b2 = np.float64(np.float32(self.beta_1)), np.float64(np.float32(self.beta_2))
        eps = np.float64(np.float32(self.epsilon))
        first = (t == 1)[:, None]
        m = b1 * np.where(first, 0.0, self.m) + (1 - b1) * g
        v = b2 * np.where(first, 0.0, self.v) + (1 - b2) * g * g
        rate = adam_alpha(self.lr, t, self.beta_1, self.beta_2)[:, None] / (np.sqrt(v) + eps)
        return m, v, rate

    def step(self, advance=True):
        """One Adam env-step of every env -> (obs [E,P,obs_dim], reward [E], done [E], info)."""
        env = self.env
        m, v, rate = self.update()
        displacement = rate * m

        def first_evaluate():                 # multioptlrs.py:85 hands over the displacement ...
            del env.evaluate                  # (the second evaluation, :88, is the oracle's own)
            return displacement, None
        unit = np.full((env.num_envs, env.num_params), _UNIT_ACTION[env.cfg.action_version])
        assert np.all(orc.action_transform(unit, env.cfg.action_version) == 1.0)
        env.evaluate = first_evaluate         # ... and the unit learning rate applies it: w - displacement
        try:
            obs, reward, done, info = env.step(unit, advance)
        finally:
            env.__dict__.pop('evaluate', None)
        info = dict(info, actions_mean=rate.mean(axis=1), actions_std=rate.std(axis=1))
        self.m, self.v = m, v
        return obs, reward, done, info
