"""Host-side parts of the device PPO2 (custom_envs_b200.ppo2): stable-baselines' parameter names and layouts, the update
arithmetic, TF's Adam, the zip files and the argument checks.  No GPU needed."""
import io
import json
import math
import zipfile
from collections import OrderedDict

import numpy as np
import pytest
import torch

from custom_envs_b200.ppo2 import (PARAMETER_MAP, PPO2, MlpPolicy, frac_of, init_like_stable_baselines,
                                   load_sb_parameters, plain_hyperparameters, read_zip, sb_parameters, tf_adam,
                                   update_plan, write_zip)
from custom_envs_b200.vectorize.device_rollout import SharedMlpPolicy

SHAPES = {'model/pi_fc0/w:0': (15, 64), 'model/pi_fc0/b:0': (64,), 'model/vf_fc0/w:0': (15, 64),
          'model/vf_fc0/b:0': (64,), 'model/pi_fc1/w:0': (64, 64), 'model/pi_fc1/b:0': (64,),
          'model/vf_fc1/w:0': (64, 64), 'model/vf_fc1/b:0': (64,), 'model/vf/w:0': (64, 1), 'model/vf/b:0': (1,),
          'model/pi/w:0': (64, 1), 'model/pi/b:0': (1,), 'model/pi/logstd:0': (1, 1), 'model/q/w:0': (64, 1),
          'model/q/b:0': (1,)}


def random_model(seed, obs_dim=15):
    torch.manual_seed(seed)
    model = SharedMlpPolicy(obs_dim)
    with torch.no_grad():
        for p in model.parameters():
            p.uniform_(-1, 1)
    return model


def test_parameter_names_layouts_and_round_trip():
    model = random_model(0)
    params = sb_parameters(model)
    assert list(params) == [entry[0] for entry in PARAMETER_MAP] == list(SHAPES)
    assert {name: value.shape for name, value in params.items()} == SHAPES
    assert all(value.dtype == np.float32 for value in params.values())
    assert np.array_equal(params['model/pi_fc0/w:0'], model.pi[0].weight.detach().numpy().T)
    assert np.array_equal(params['model/vf_fc1/b:0'], model.vf[2].bias.detach().numpy())
    assert np.array_equal(params['model/vf/w:0'], model.vf[4].weight.detach().numpy().T)
    assert np.array_equal(params['model/pi/b:0'], model.pi[4].bias.detach().numpy())
    assert params['model/pi/logstd:0'][0, 0] == model.log_std.detach().numpy()
    assert not params['model/q/w:0'].any() and not params['model/q/b:0'].any()
    other = random_model(1)
    load_sb_parameters(other, params)
    for p, q in zip(model.parameters(), other.parameters()):
        assert torch.equal(p, q)


def test_parameter_loading_checks_names_and_shapes():
    model = random_model(2)
    params = sb_parameters(model)
    partial = OrderedDict((k, v) for k, v in params.items() if k != 'model/q/b:0')
    with pytest.raises(ValueError, match='missing'):
        load_sb_parameters(random_model(3), partial)
    target = random_model(3)
    load_sb_parameters(target, dict(partial, extra=np.zeros(3)), exact_match=False)
    assert torch.equal(target.pi[0].weight, model.pi[0].weight)
    bad = dict(params)
    bad['model/pi_fc1/w:0'] = np.zeros((64, 63), np.float32)
    with pytest.raises(ValueError, match='shape'):
        load_sb_parameters(random_model(4), bad)


def test_initialisation_follows_stable_baselines():
    model = SharedMlpPolicy(15)
    init_like_stable_baselines(model, torch.Generator().manual_seed(5))
    for tower, gain in ((model.pi, 0.01), (model.vf, 1.0)):
        lins = [m for m in tower if isinstance(m, torch.nn.Linear)]
        for i, lin in enumerate(lins):
            w = lin.weight.detach().double()
            g = gain if i == 2 else math.sqrt(2)
            small = w @ w.t() if w.shape[0] <= w.shape[1] else w.t() @ w
            assert torch.allclose(small, g * g * torch.eye(small.shape[0], dtype=torch.float64), atol=1e-5)
            assert not lin.bias.any()
    assert float(model.log_std.detach()) == 0.0
    again = SharedMlpPolicy(15)
    init_like_stable_baselines(again, torch.Generator().manual_seed(5))
    assert all(torch.equal(p, q) for p, q in zip(model.parameters(), again.parameters()))
    init_like_stable_baselines(again, torch.Generator().manual_seed(6))
    assert not torch.equal(model.pi[0].weight, again.pi[0].weight)


def test_update_count_and_schedule_argument():
    assert update_plan(10000, 8, 30, 4) == (240, 41)
    assert update_plan(239, 8, 30, 4) == (240, 0)
    n = 5
    assert [frac_of(u, n) for u in range(1, n + 1)] == [1.0, 0.8, 0.6, 1.0 - 3.0 / 5, 0.19999999999999996]
    with pytest.raises(AssertionError, match='nminibatches'):
        update_plan(10000, 3, 15, 4)


def tf_adam_np(param, grads, lr, b1=0.9, b2=0.999, eps=1e-5):
    """TF 1.x AdamOptimizer (adam.py _apply_dense / training_ops ApplyAdam) in float64."""
    m = np.zeros_like(param)
    v = np.zeros_like(param)
    out = []
    for t, g in enumerate(grads, start=1):
        lr_t = lr * math.sqrt(1 - b2 ** t) / (1 - b1 ** t)
        m = b1 * m + (1 - b1) * g
        v = b2 * v + (1 - b2) * g * g
        param = param - lr_t * m / (np.sqrt(v) + eps)
        out.append(param.copy())
    return out


@pytest.mark.parametrize('hooked', [True, False])
def test_adam_hook_is_tf_adam(hooked):
    """Gradients of the size of eps, where the epsilon placement matters: with the hook torch's Adam follows TF's
    formulas to 1e-6 over 100 steps; plain torch Adam with eps = 1e-5 does not."""
    rng = np.random.RandomState(0)
    start = rng.normal(size=50)
    grads = [rng.normal(size=50) * 3e-5 for _ in range(100)]
    want = tf_adam_np(start, grads, lr=2.5e-4)
    p = torch.nn.Parameter(torch.tensor(start))
    opt = tf_adam([p], lr=2.5e-4) if hooked else torch.optim.Adam([p], lr=2.5e-4, eps=1e-5)
    worst = 0.0
    for g, w in zip(grads, want):
        p.grad = torch.tensor(g)
        opt.step()
        worst = max(worst, float(np.max(np.abs(p.detach().numpy() - w) / np.abs(w))))
    if hooked:
        assert worst <= 1e-6, worst
    else:
        assert worst > 1e-5, worst


def test_zip_round_trip(tmp_path):
    params = sb_parameters(random_model(7))
    data = {'gamma': 0.95, 'n_steps': 16, 'learning_rate': 1e-3, 'seed': 3, 'n_envs': 45}
    write_zip(str(tmp_path / 'model'), data, params)
    assert (tmp_path / 'model.zip').is_file()                     # no extension: '.zip' added
    write_zip(str(tmp_path / 'model.pkl'), data, params)           # the reference's name is kept
    with zipfile.ZipFile(tmp_path / 'model.pkl') as file_:
        assert sorted(file_.namelist()) == ['data', 'parameter_list', 'parameters']
        assert json.loads(file_.read('parameter_list')) == list(params)
    for path in (str(tmp_path / 'model'), str(tmp_path / 'model.pkl')):
        got_data, got = read_zip(path)
        assert got_data == data and list(got) == list(params)
        assert all(np.array_equal(got[k], params[k]) and got[k].dtype == np.float32 for k in params)


def test_reads_a_zip_laid_out_by_stable_baselines(tmp_path):
    """The layout of stable-baselines 2.10's _save_to_file_zip: data with cloudpickled entries, the npz of the parameter
    OrderedDict, the JSON name list.  Only the parameters and the plain hyperparameters are taken."""
    params = sb_parameters(random_model(8))
    data = {'gamma': 0.9, 'n_steps': 32, 'ent_coef': 0.0, 'learning_rate': 2.5e-4, 'lam': 0.9, 'nminibatches': 1,
            'noptepochs': 4, 'cliprange': 0.2, 'cliprange_vf': None, 'verbose': 1, 'seed': None, 'policy_kwargs': {},
            'n_envs': 15, 'n_cpu_tf_sess': None, '_vectorize_action': False,
            'policy': {':type:': "<class 'abc.ABCMeta'>", ':serialized:': 'gANjc3RhYmxlX2Jhc2VsaW5lcw=='},
            'observation_space': {':type:': "<class 'gym.spaces.box.Box'>", ':serialized:': 'gASVAAAA',
                                  'shape': [15], 'dtype': 'float32'},
            'action_space': {':type:': "<class 'gym.spaces.box.Box'>", ':serialized:': 'gASVAAAA'}}
    raw = io.BytesIO()
    np.savez(raw, **params)
    with zipfile.ZipFile(tmp_path / 'sb.zip', 'w') as file_:
        file_.writestr('data', json.dumps(data, indent=4))
        file_.writestr('parameters', raw.getvalue())
        file_.writestr('parameter_list', json.dumps(list(params.keys()), indent=4))
    got_data, got = read_zip(str(tmp_path / 'sb.zip'))
    assert list(got) == list(params)
    target = random_model(9)
    load_sb_parameters(target, got)
    assert sb_parameters(target).keys() == params.keys()
    assert all(np.array_equal(a, b) for a, b in zip(sb_parameters(target).values(), params.values()))
    assert plain_hyperparameters(got_data) == {'gamma': 0.9, 'n_steps': 32, 'ent_coef': 0.0, 'learning_rate': 2.5e-4,
                                               'lam': 0.9, 'nminibatches': 1, 'noptepochs': 4, 'cliprange': 0.2,
                                               'cliprange_vf': None, 'verbose': 1, 'seed': None, 'policy_kwargs': {}}
    (tmp_path / 'legacy.pkl').write_bytes(b'\x80\x03cstable_baselines')
    with pytest.raises(ValueError, match='not a zip'):
        read_zip(str(tmp_path / 'legacy.pkl'))


def test_rejections():
    for policy in ('CnnPolicy', 'MlpLstmPolicy', object):
        with pytest.raises(ValueError, match='MlpPolicy only'):
            PPO2(policy, None)
    for kwargs in (dict(net_arch=[128, 128]), dict(act_fun=torch.relu), dict(net_arch=[dict(pi=[64], vf=[64])])):
        with pytest.raises(ValueError, match='policy_kwargs item %r' % next(iter(kwargs))):
            PPO2(MlpPolicy, None, policy_kwargs=kwargs)
    with pytest.raises(ValueError, match='needs an env'):
        PPO2('MlpPolicy', None, policy_kwargs=dict(net_arch=[dict(pi=[64, 64], vf=[64, 64])]))
    model = PPO2(MlpPolicy, None, _init_setup_model=False, tensorboard_log='/nonexistent', n_cpu_tf_sess=4)
    with pytest.raises(ValueError, match='needs an env'):
        model.learn(1000)
    with pytest.raises(ValueError, match='BatchedOptEnv'):
        model.set_env(object())
