"""Host side of data-parallel PPO: shard offsets, per-rank permutation keys, the rank-table check every rank runs on the
gathered table, and a plain-C client of the new entry points.  None of these needs a GPU."""
import os

import pytest

from custom_envs_b200 import _lib
from custom_envs_b200.sharding import shard_bases, shard_range
from custom_envs_b200.vectorize.device_policy import _check_rank_table, epoch_key, rank_epoch_key


def test_shard_bases_follow_the_global_env_and_row_index():
    P = 50890
    for E, world in [(4096, 8), (5, 2), (7, 3), (3, 4)]:
        rows = 0
        for r in range(world):
            first, count = shard_range(E, world, r)
            assert shard_bases(E, world, r, P) == (first, first * P)
            assert first * P == rows
            rows += count * P
        assert rows == E * P


def test_rank_keys():
    """Rank 0 uses the single-GPU epoch key (a one-rank update is the single-GPU one); other ranks get distinct keys."""
    keys = set()
    for seed in (0, 7, 2 ** 62 - 1, 2 ** 64 - 1):
        for epoch in range(4):
            assert rank_epoch_key(seed, epoch, 0) == epoch_key(seed, epoch)
            for rank in range(8):
                k = rank_epoch_key(seed, epoch, rank)
                assert 0 <= k < 2 ** 64
                keys.add(k)
    assert len(keys) == 4 * 4 * 8
    # pinned: splitmix64 finaliser of epoch_key + rank * 0x9E3779B97F4A7C15
    z = (epoch_key(3, 1) + 2 * 0x9E3779B97F4A7C15) % 2 ** 64
    z = ((z ^ (z >> 30)) * 0xBF58476D1CE4E5B9) % 2 ** 64
    z = ((z ^ (z >> 27)) * 0x94D049BB133111EB) % 2 ** 64
    assert rank_epoch_key(3, 1, 2) == z ^ (z >> 31)


def test_rank_table_check():
    """[T, buffer width, obs_width, obs_dim, T * rows, n_epochs, n_minibatches, seed] of every rank."""
    ok = [2, 16, 16, 15, 2000, 4, 4, 9], [2, 16, 16, 15, 3000, 4, 4, 123]
    assert _check_rank_table([list(r) for r in ok], 4) == (9, 1250)
    assert _check_rank_table([ok[0][:7] + [-1]], 4) == (2 ** 64 - 1, 500)
    with pytest.raises(ValueError, match=r'disagree on T \(n_steps\): \[2, 3\]'):
        _check_rank_table([ok[0], [3] + ok[1][1:]], 4)
    with pytest.raises(ValueError, match='disagree on the observation width'):
        _check_rank_table([ok[0], ok[1][:2] + [32, 30] + ok[1][4:]], 4)
    with pytest.raises(ValueError, match='disagree on n_epochs'):
        _check_rank_table([ok[0], ok[1][:5] + [3] + ok[1][6:]], 4)
    with pytest.raises(ValueError, match=r'rank\(s\) \[1\] are not'):
        _check_rank_table([ok[0], [2, 32] + ok[1][2:]], 4)
    with pytest.raises(ValueError, match=r'T \* rows = \[3004\] of rank\(s\) \[1\]'):
        _check_rank_table([ok[0][:4] + [2000, 4, 8, 9], ok[1][:4] + [3004, 4, 8, 9]], 8)
    with pytest.raises(ValueError, match='n_minibatches = 0'):
        _check_rank_table([ok[0][:6] + [0, 9]], 0)


def test_a_c_client_reaches_the_data_parallel_entry_points(tmp_path):
    import shutil
    import subprocess
    if shutil.which('gcc') is None:
        pytest.skip('no C compiler')
    if not os.path.exists(_lib.LIB_PATH):
        pytest.skip('libb200env.so is not built')
    here = os.path.dirname(os.path.abspath(__file__))
    exe = str(tmp_path / 'c_abi_dist_smoke')
    subprocess.run(['gcc', '-std=c99', '-pedantic', '-Wall', '-Werror', '-I', os.path.join(here, '..', 'include'),
                    os.path.join(here, 'c_abi_dist_smoke.c'), '-o', exe, '-ldl'], check=True)
    out = subprocess.run([exe, _lib.LIB_PATH], capture_output=True, text=True)
    assert out.returncode == 0 and 'c dist abi ok' in out.stdout, (out.returncode, out.stderr)
