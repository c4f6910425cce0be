"""Pins the oracle port (oracle/port.py) against golden vectors recorded from
the UNMODIFIED reference (tests/golden/*.npz, made by oracle/make_golden.py).
Everything here runs on the CPU."""

import numpy as np
import pytest
import torch

from oracle import port, scenarios, synth_env


@pytest.fixture
def one_blas_thread():
    """The BLAS splits a matrix product's sums over its threads, so the last bits of the torch
    CPU arithmetic depend on how many threads the host gives it; with one thread the oracle
    reproduces the golden run bit for bit whatever the host's core count."""
    saved = torch.get_num_threads()
    torch.set_num_threads(1)
    yield
    torch.set_num_threads(saved)


def test_lambda_returns_kats(golden):
    g = golden('units')
    for tag in 'abc':
        args = [g[f'lam_{tag}/{k}'] for k in
                ('values', 'next_values', 'rewards', 'resets', 'terminations')]
        out = port.lambda_returns(*args, 0.99, 0.97)
        np.testing.assert_array_equal(out, g[f'lam_{tag}/returns'])
    # SURVEY.md 8(c) KAT1
    kat1 = np.array([1.9285942, -0.368923, 0.45567083, -0.18323392,
                     -1.2782894, 0.6536186, 1.3038608, -0.4118274], np.float32)
    np.testing.assert_allclose(g['kat1/returns'].ravel(), kat1, rtol=1e-6)


@pytest.mark.parametrize('tag', 'abc')
def test_segment_index_stream(golden, tag):
    g = golden('units')
    size, workers, iters, bs, seed = g[f'segidx_{tag}/cfg']
    seg = port.SegmentStore(size=size, batch_iterations=iters, batch_size=bs)
    seg.initialize(seed)
    for t in range(size):
        seg.store(ids=np.arange(workers) + t * workers)
    batches = [b['ids'].astype(np.int64) for b in seg.batches('ids')]
    np.testing.assert_array_equal(np.concatenate(batches), g[f'segidx_{tag}/indices'])
    np.testing.assert_array_equal([len(b) for b in batches], g[f'segidx_{tag}/lengths'])


def test_advantage_normalisation(golden):
    g = golden('units')
    seg = port.SegmentStore(size=32, batch_iterations=1, batch_size=None)
    seg.initialize(0)
    for t in range(32):
        seg.store(rewards=g['adv/rewards'][t], resets=g['adv/resets'][t],
                  terminations=np.zeros(16))
    seg.compute_returns(g['adv/values'], g['adv/next_values'])
    full = seg.flat('advantages', 'returns')
    np.testing.assert_array_equal(full['returns'], g['adv/returns'])
    np.testing.assert_array_equal(full['advantages'], g['adv/advantages'])


def test_ring_buffer_stream(golden):
    g = golden('units')
    buf = port.RingStore(size=40, batch_iterations=3, batch_size=8,
                         steps_before_batches=0, steps_between_batches=1)
    buf.initialize(9)
    for t in range(14):
        buf.store(ids=np.arange(4) + 4 * t, terminations=np.arange(4) == t % 4)
    got = list(buf.batches('ids', 'discounts', steps=100))
    np.testing.assert_array_equal(np.stack([b['ids'] for b in got]), g['bufidx/ids'])
    np.testing.assert_array_equal(np.stack([b['discounts'] for b in got]),
                                  g['bufidx/discounts'])
    assert buf.last_steps == 100


def test_running_moments(golden):
    g = golden('units')
    ms = port.RunningMoments(5)
    snaps = []
    for i, b in enumerate(g['meanstd/batches']):
        ms.record(b)
        if i % 2 == 1:
            ms.update()
            snaps.append(np.stack([ms.t_mean.numpy(), ms.t_std.numpy()]))
    np.testing.assert_array_equal(np.stack(snaps), g['meanstd/snapshots'])


def test_vector_env_matches_reference_sequential(golden):
    g = golden('units')
    env = port.VectorEnv(7, 3, 5, 6)
    env.initialize(21)
    obs = [env.start()]
    for t, a in enumerate(g['env/actions']):
        o, infos = env.step(a)
        obs.append(o)
        np.testing.assert_array_equal(infos['observations'], g['env/next_observations'][t])
        np.testing.assert_array_equal(infos['rewards'], g['env/rewards'][t])
        np.testing.assert_array_equal(infos['resets'], g['env/resets'][t])
        np.testing.assert_array_equal(infos['terminations'], g['env/terminations'][t])
    np.testing.assert_array_equal(np.array(obs), g['env/observations'])
    assert g['env/terminations'].sum() > 0 and g['env/resets'].sum() > g['env/terminations'].sum()


def test_vectorised_env_helpers_match_scalar():
    seeds = np.arange(5) + 21
    eps = np.array([0, 3, 1, 7, 2])
    vec = synth_env.reset_state_vec(seeds, eps, 9)
    for i in range(5):
        np.testing.assert_array_equal(vec[i], synth_env.reset_state(int(seeds[i]), int(eps[i]), 9))
    assert vec.min() >= -1 and vec.max() < 1


@pytest.mark.parametrize('name', list(scenarios.SCENARIOS))
def test_oracle_reproduces_reference_scenario(golden, name, one_blas_thread):
    g = golden(name)
    cfg = scenarios.SCENARIOS[name]
    rec = scenarios.InfoRecorder()
    agent, env = port.build(cfg, log=rec)
    w0 = scenarios.state_arrays(agent.state_dict(), 'w0/')
    out = scenarios.drive(agent, env, cfg['vector_steps'])
    out.update(rec.arrays())
    # trajectories: bit-exact (same torch/numpy calls in the same order)
    for k in ('start_observations', 'actions', 'observations', 'next_observations',
              'rewards', 'resets', 'terminations'):
        np.testing.assert_array_equal(out[k], g[k], err_msg=k)
    assert list(out['info_keys']) == list(g['info_keys'])
    np.testing.assert_allclose(out['info_mean'], g['info_mean'], rtol=1e-6, atol=1e-7)
    np.testing.assert_allclose(out['info_abs'], g['info_abs'], rtol=1e-6, atol=1e-7)
    w = scenarios.state_arrays(agent.state_dict(), 'w/')
    w.update(w0)
    checked = 0
    for k, v in w.items():
        if k in g:
            np.testing.assert_allclose(v, g[k], rtol=1e-6, atol=1e-7, err_msg=k)
            checked += 1
        elif 'digest_' + k in g:
            f = v.astype(np.float64).ravel()
            d = np.concatenate([[f.sum(), np.abs(f).sum()], f[:8], np.zeros(max(0, 8 - f.size))])
            np.testing.assert_allclose(d, g['digest_' + k], rtol=1e-6, atol=1e-6, err_msg=k)
            checked += 1
    # every tensor of the reference state_dict exists in the oracle's
    ref_keys = {k.replace('digest_', '') for k in g
                if k.startswith(('w/', 'w0/', 'digest_w/', 'digest_w0/'))}
    assert ref_keys == set(w)
    assert checked == len(ref_keys)


@pytest.mark.skipif(not __import__('os').environ.get('TONIC_B200_SLOW_TESTS'),
                    reason='takes ~1-2 CPU minutes: set TONIC_B200_SLOW_TESTS=1')
def test_oracle_reproduces_reference_at_the_benched_shape(golden):
    """Oracle port vs the unmodified reference at BASELINE configs[1]'s shape (digests)."""
    from oracle import bench_shape
    g = golden('ppo_bench')
    cfg = bench_shape.CFG
    rec = scenarios.InfoRecorder()
    agent, env = port.build(cfg, log=rec)
    out = bench_shape.drive(agent, env, cfg)
    for k in ('observation_digest', 'reward_digest', 'reset_count', 'termination_count'):
        np.testing.assert_array_equal(out[k], g[k], err_msg=k)
    np.testing.assert_allclose(out['action_sample'], g['action_sample'], rtol=1e-6, atol=1e-6)
    assert list(rec.keys) == list(g['info_keys'])
    np.testing.assert_allclose(rec.means, g['info_mean'], rtol=1e-5, atol=1e-6)
    w = bench_shape.weight_digests(agent.state_dict(), 'digest_w/')
    for k, v in w.items():
        np.testing.assert_allclose(v, g[k], rtol=1e-4, atol=1e-5, err_msg=k)


def test_benched_shape_fixture_is_the_benchmark_configuration(golden):
    from oracle import bench_shape
    g = golden('ppo_bench')
    cfg = bench_shape.CFG
    assert (cfg['workers'], cfg['segment']['size'], cfg['segment']['batch_size'],
            cfg['segment']['batch_iterations'], cfg['hidden']) == (4096, 128, 16384, 10, (256, 256))
    assert g['action_digest'].shape == (128, 2) and g['action_sample'].shape == (128, 32, 6)
    keys = list(g['info_keys'])
    assert keys.count('critic/loss') == 320
    a = bench_shape.driving_actions(3, 4096, 6)
    assert a.dtype == np.float32 and a.min() >= -1.25 and a.max() < 1.25 and (np.abs(a) > 1).any()


def test_parallel_worker_grid_equals_sequential():
    """The forked P x M grid (distributed.py:69-155) returns what one sequential group of
    P * M environments returns: same seeds (seed + j), group-major order."""
    seq = port.VectorEnv(5, 2, 6, 7)
    par = port.ParallelVectorEnv(5, 2, 3, 2, 7)
    seq.initialize(11)
    par.initialize(11)
    try:
        np.testing.assert_array_equal(seq.start(), par.start())
        rs = np.random.RandomState(0)
        for _ in range(20):
            a = rs.normal(size=(6, 2)).astype(np.float32)
            o1, i1 = seq.step(a)
            o2, i2 = par.step(a)
            np.testing.assert_array_equal(o1, o2)
            for k in i1:
                np.testing.assert_array_equal(i1[k], i2[k], err_msg=k)
    finally:
        par.close()
