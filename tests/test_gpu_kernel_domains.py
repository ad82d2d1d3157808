"""Oracle parity of every eval kernel of the large-problem step across the shapes its dispatch accepts.

``configure()`` (csrc/b200env.cu) and the ``b2e_*_supported`` predicates (b200tc.cu, b200thin.cu) pick the
eval kernel from the problem's shape.  The BASELINE shapes 784-64-10 and 784-10 reach one instantiation
each; the table below reaches the others, at the tile edges where they differ: generic class counts of the
tcgen05 kernel (one to three 32-feature units more than a multiple of the backward tile, fewer units per
env than forward ring stages), the FFMA eval kernel at run-time layer widths, tile lengths and minibatch
sizes, the fused kernel's step mode just below the eval-kernel split, ragged feature chunks of the
streamed softmax kernel, and both resident-minibatch kernels up to their shared-memory limits.

Per case: the launched kernel is the one named (torch.profiler), b2e_eval matches the float64 oracle, and
seven steps from identical states match it (the bars of test_gpu_parity.py).  One shape per kernel also
runs 2 x SMs + 4 envs, so that envs at CTA and round boundaries of the persistent grids are checked.
"""
import os
import re
import sys

import numpy as np
import pytest
import torch

from oracle import optenv_oracle as orc

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))       # the helpers of test_gpu_parity.py
from test_gpu_parity import (_mods, eval_parity, make_data, product_spec, reset_pipeline_parity,  # noqa: E402
                             sampled_env_parity, step_parity)

pytestmark = pytest.mark.gpu

TC = {'B2E_TC_CHECK': '1'}        # a stalled tcgen05 pipeline comes back as an error instead of a hang
TC2_C = r'tc2_eval_kernel<(false|true), 0>'
TC2_10 = r'tc2_eval_kernel<(false|true), 10>'
FFMA = r'(?<!\w)eval_kernel<(false|true), 0, 0>'
FFMA_C = r'(?<!\w)eval_kernel<(false|true), 64, 112>'
FUSED = r'optenv_kernel<5, true>'
THIN_C = r'thin_eval_kernel<(false|true), 0>'
THIN_10 = r'thin_eval_kernel<(false|true), 10>'
THIN2 = r'thin2_eval_kernel<(false|true)>'
THIN3 = r'thin3_eval_kernel<(false|true)>'


def S(kind, d, hidden, c):
    return orc.ProblemSpec(kind, d, hidden, c)


# (id, spec, batch size, env overrides, launched kernel, also at 2 x SMs + 4 envs)
CASES = [
    ('tc2_784x64x3', S('softmax', 784, (64,), 3), 32, TC, TC2_C, True),
    ('tc2_784x64x16', S('softmax', 784, (64,), 16), 32, TC, TC2_C, False),        # CMAX classes
    ('tc2_100x64x7', S('softmax', 100, (64,), 7), 32, TC, TC2_C, False),          # 4 units, the last one partial; one backward tile
    ('tc2_132x64x11', S('softmax', 132, (64,), 11), 32, TC, TC2_C, False),        # two backward tiles, the last 4 features wide
    ('tc2_64x64x2', S('softmax', 64, (64,), 2), 32, TC, TC2_C, False),            # fewer units than forward ring stages
    ('tc2_260x64x10', S('softmax', 260, (64,), 10), 32, TC, TC2_10, True),        # 9 units, partial last unit and tile
    ('tc2_1000x64x10', S('softmax', 1000, (64,), 10), 32, TC, TC2_10, False),
    ('ffma_49x128x10', S('softmax', 49, (128,), 10), 32, {}, FFMA, True),          # load_data('mnist') features
    ('ffma_49x256x10', S('softmax', 49, (256,), 10), 32, {}, FFMA, False),
    ('ffma_784x32x10', S('softmax', 784, (32,), 10), 32, {}, FFMA, False),
    ('ffma_784x128x10', S('softmax', 784, (128,), 10), 32, {}, FFMA, False),
    ('ffma_784x64x10_b16', S('softmax', 784, (64,), 10), 16, {}, FFMA, False),
    ('ffma_784x64x10_b1', S('softmax', 784, (64,), 10), 1, {}, FFMA, False),
    # N1 = 64, 112-row tiles and B = 32 without the softmax bulk-copy form: linear regression with 64 outputs
    ('ffma64_linreg_784x64', S('linreg', 784, (), 64), 32, {}, FFMA_C, True),
    ('fused_60x64x10', S('softmax', 60, (64,), 10), 32, {}, FUSED, True),         # register-tiled, below the eval-kernel split
    ('fused_124x32x10', S('softmax', 124, (32,), 10), 32, {}, FUSED, False),
    ('thin_524x16', S('softmax', 524, (), 16), 32, {}, THIN_C, True),             # no chunk divides D: ragged last chunk
    ('thin_1536x3', S('softmax', 1536, (), 3), 32, {}, THIN_C, False),
    ('thin_1100x10', S('softmax', 1100, (), 10), 32, {}, THIN_10, True),          # wider than the resident kernels
    ('thin_784x10_thin2off', S('softmax', 784, (), 10), 32, {'B2E_THIN2': '0'}, THIN_10, False),
    ('thin2_860x10', S('softmax', 860, (), 10), 32, {}, THIN2, True),             # D % 8 != 0, widest that fits two CTAs per SM
    ('thin2_500x10_b20', S('softmax', 500, (), 10), 20, {}, THIN2, False),
    ('thin3_416x10', S('softmax', 416, (), 10), 32, {}, THIN3, True),             # near the P >= 4096 floor
    ('thin3_848x10', S('softmax', 848, (), 10), 32, {}, THIN3, False),            # widest that fits three CTAs per SM
]
# Cap of the well-conditioned observation entries (test_gpu_parity.check_obs: 20 RTOL) where rounding exceeds
# it.  3 classes under learning rates up to 0.1: the softmax saturates, and d loss / d logit_y = p_y - 1
# carries the fp32 rounding of p_y (6e-8 absolute) into gradients whose other terms are small.  Worst measured
# (B200 at 1000 W, 2 x 148 + 4 envs, B2E_TEST_STATS): 27 RTOL on one entry of 6.8 M with the tcgen05 kernel,
# below 20 with the FFMA kernel (B2E_TC=0) on the same shape; every other case of the table below 16.
OBS_CAP = {'tc2_784x64x3': 40}
IDS = [c[0] for c in CASES]
BY_ID = {c[0]: c for c in CASES}
NUM_ENVS = 3


def num_rows_of(batch):
    """Two full minibatches and a ragged third: not a multiple of the batch size (except B = 1)."""
    return 2 * batch + 5


def case_data(spec, num_rows):
    """make_data, except for linear regression: features scaled by 1/sqrt(D), so that the learning rates of
    the action range (up to 0.1) keep the 784-feature problem stable and far from the divergence rule."""
    if spec.kind != 'linreg':
        return make_data(spec, num_rows)
    rng = np.random.RandomState(5)
    feats = (rng.uniform(size=(num_rows, spec.num_features)) / np.sqrt(spec.num_features)).astype(np.float32)
    true_w = rng.normal(size=(spec.num_features, spec.num_outputs))
    targs = (feats @ true_w + 0.1 * rng.normal(size=(num_rows, spec.num_outputs))).astype(np.float32)
    return feats, targs


def setup_case(case_id, monkeypatch):
    _, spec, batch, env_vars, pattern, _ = BY_ID[case_id]
    for key in ('B2E_TC', 'B2E_THIN2', 'B2E_FORCE_GENERIC', 'B2E_RESET_PIPELINE'):
        monkeypatch.delenv(key, raising=False)
    for key, value in env_vars.items():
        monkeypatch.setenv(key, value)
    return spec, batch, pattern


def launched_kernels(env):
    """Names of the kernels one reset and one step launch."""
    from torch.profiler import ProfilerActivity, profile
    actions = torch.rand(env.num_rows, device=env.device, generator=torch.Generator(device=env.device).manual_seed(0))
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        env.reset()
        env.step(actions)
        torch.cuda.synchronize(env.device)
    return sorted({e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA})


@pytest.mark.parametrize('case_id', IDS)
def test_dispatch_launches_the_named_kernel(case_id, monkeypatch):
    """The shape reaches the kernel the table names, in both evaluation passes of the step."""
    BatchedOptEnv, _ = _mods()
    spec, batch, pattern = setup_case(case_id, monkeypatch)
    num_rows = num_rows_of(batch)
    feats, targs = case_data(spec, num_rows)
    env = BatchedOptEnv(product_spec(spec), feats, targs, NUM_ENVS, batch_size=batch, max_batches=4, init_seed=1)
    names = launched_kernels(env)
    env.close()
    assert names, 'the profiler recorded no kernel'
    for second in ('false', 'true'):
        want = pattern.replace('(false|true)', second)
        assert any(re.search(want, n) for n in names), (case_id, want, names)


@pytest.mark.parametrize('case_id', IDS)
def test_eval_matches_oracle(case_id, monkeypatch):
    """b2e_eval (loss and batch-sum gradient, the last env on a ragged minibatch) against the float64 oracle."""
    spec, batch, _ = setup_case(case_id, monkeypatch)
    num_rows = num_rows_of(batch)
    eval_parity((spec, num_rows, batch, NUM_ENVS), case_id, data=case_data(spec, num_rows))


@pytest.mark.parametrize('case_id', IDS)
def test_step_parity_from_identical_states(case_id, monkeypatch):
    """Seven steps with host-supplied minibatches (one ragged per step) against the oracle."""
    spec, batch, _ = setup_case(case_id, monkeypatch)
    num_rows = num_rows_of(batch)
    step_parity((spec, num_rows, batch, NUM_ENVS), (case_id, 'lexicographic'), data=case_data(spec, num_rows),
                obs_cap=OBS_CAP.get(case_id, 20))


@pytest.mark.parametrize('case_id', [c[0] for c in CASES if c[5]])
def test_more_envs_than_resident_ctas(case_id, monkeypatch):
    """2 x SMs + 4 envs on the on-device minibatch stream with auto-reset: the oracle follows the envs at the
    CTA and round boundaries of a one-CTA-per-SM grid (0, 1, SMs - 1, SMs, SMs + 1, the last four)."""
    spec, batch, _ = setup_case(case_id, monkeypatch)
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    num_envs = 2 * sms + 4
    sample = {0, 1, sms - 1, sms, sms + 1} | set(range(num_envs - 4, num_envs))
    num_rows = num_rows_of(batch)
    data = case_data(spec, num_rows) if spec.kind == 'linreg' else None
    ragged = sampled_env_parity(spec, num_rows, num_envs, case_id, sample=sample, batch=batch, data=data,
                                obs_cap=OBS_CAP.get(case_id, 20))
    assert ragged > 0, case_id


def test_reset_pipeline_of_the_generic_class_tensor_core_path(monkeypatch):
    """test_reset_pipeline_of_the_tensor_core_path with 7 classes and 100 features: the reset work list runs
    tc2_eval_kernel<., 0> on four forward units, the last one partial."""
    monkeypatch.setenv('B2E_TC_CHECK', '1')
    reset_pipeline_parity(orc.ProblemSpec('softmax', 100, (64,), 7), monkeypatch)
