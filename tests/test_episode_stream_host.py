"""CPU: the device episode stream's C-ABI surface, argument validation (checked before anything is launched), the
scripted-agent count and the exact probabilities the GPU distribution tests compare against."""
import ctypes as C
import math
import os
import subprocess
import tempfile

import numpy as np
import pytest

from episode_stream_util import expected_duplicate_pairs, k_of_u, k_probabilities, node_inclusion
from melissa_b200 import _lib, reset_chain
from melissa_b200.batched_env import EpisodeStream, scripted_count

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FAKE = 0x1000          # a non-NULL address: every call below fails validation before it could be dereferenced


def test_sampler_struct_matches_the_header_and_version():
    prog = ('#include <stdio.h>\n#include <stddef.h>\n#include "melissa_b200.h"\nint main(){'
            'printf("%zu %zu %zu\\n", sizeof(MlsEpisodeSampler), offsetof(MlsEpisodeSampler, pool_size), '
            'offsetof(MlsEpisodeSampler, slot_offset)); return 0;}')
    with tempfile.TemporaryDirectory() as d:
        c = os.path.join(d, "t.c")
        open(c, "w").write(prog)
        subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), c, "-o", os.path.join(d, "t")])
        size, off_pool, off_slot = map(int, subprocess.check_output([os.path.join(d, "t")], text=True).split())
    assert size == C.sizeof(_lib.MlsEpisodeSampler) == 24
    assert off_pool == _lib.MlsEpisodeSampler.pool_size.offset and off_slot == _lib.MlsEpisodeSampler.slot_offset.offset
    L = _lib.lib()
    assert L.mls_version() >= 214
    for name in ("mls_env_reset_sampled", "mls_env_step_sampled", "mls_episode_sample"):
        assert hasattr(L, name)


def _sample(smp, n_nodes=20, n=4, arrays=True):
    p = FAKE if arrays else None
    return _lib.lib().mls_episode_sample(C.byref(smp) if smp is not None else None, n_nodes, p, p, n, p, p, p, p, None)


def test_episode_sample_validates_its_arguments():
    ok = _lib.MlsEpisodeSampler(1, 8, 0, 1, 0)
    assert _sample(ok, n=0) == 0                                         # nothing to draw: no launch
    bad = [(None, {}), (_lib.MlsEpisodeSampler(1, 0, 0, 1, 0), {}), (_lib.MlsEpisodeSampler(1, -3, 0, 1, 0), {}),
           (_lib.MlsEpisodeSampler(1, 8, 21, 1, 0), {}), (_lib.MlsEpisodeSampler(1, 8, -1, 1, 0), {}),
           (ok, dict(n_nodes=0)), (ok, dict(n_nodes=257)), (ok, dict(n=-1)), (ok, dict(arrays=False))]
    for smp, kw in bad:
        assert _sample(smp, **kw) == -1, (smp, kw)                      # MLS_ERR_INVALID
        assert _lib.lib().mls_last_error()
    with pytest.raises(ValueError, match="n_scripted"):
        _lib.check(_sample(_lib.MlsEpisodeSampler(1, 8, 21, 1, 0)))
    with pytest.raises(ValueError, match="arrays missing"):
        _lib.check(_sample(ok, arrays=False))


def test_sampled_round_calls_validate_the_sampler():
    L = _lib.lib()
    desc = _lib.MlsEnvDesc(4, 20, 0, 0, 0, 0, 0, 0)
    state = _lib.MlsEnvState(FAKE, FAKE, None, FAKE, FAKE, None, None, FAKE, FAKE, 8, 0)
    inp = _lib.MlsRoundInputs(FAKE, None, None, None, 9)
    out = _lib.MlsRoundOutputs()
    for smp, msg in ((_lib.MlsEpisodeSampler(1, 9, 0, 1, 0), "pool_size"),        # more graphs than the topology pool
                     (_lib.MlsEpisodeSampler(1, 0, 0, 1, 0), "pool_size"),
                     (_lib.MlsEpisodeSampler(1, 8, 21, 1, 0), "n_scripted")):
        with pytest.raises(ValueError, match=msg):
            _lib.check(L.mls_env_step_sampled(C.byref(desc), C.byref(state), C.byref(inp), C.byref(out), C.byref(smp), None))
        with pytest.raises(ValueError, match=msg):
            _lib.check(L.mls_env_reset_sampled(C.byref(desc), C.byref(state), None, 4, C.byref(smp), None, None, None))
    smp = _lib.MlsEpisodeSampler(1, 8, 0, 1, 0)
    with pytest.raises(ValueError, match="sampler is NULL"):
        _lib.check(L.mls_env_step_sampled(C.byref(desc), C.byref(state), C.byref(inp), C.byref(out), None, None))
    with pytest.raises(ValueError, match="more resets than episodes"):
        _lib.check(L.mls_env_reset_sampled(C.byref(desc), C.byref(state), None, 5, C.byref(smp), None, None, None))
    with pytest.raises(ValueError, match="n < 0"):
        _lib.check(L.mls_env_reset_sampled(C.byref(desc), C.byref(state), None, -1, C.byref(smp), None, None, None))
    with pytest.raises(ValueError, match="actions missing"):
        _lib.check(L.mls_env_step_sampled(C.byref(desc), C.byref(state), None, C.byref(out), C.byref(smp), None))


def test_episode_stream_arguments_and_scripted_rounding():
    for r in (-0.1, 1.5):
        with pytest.raises(ValueError, match="must be in"):
            EpisodeStream(20, 8, 1, scripted_agents_ratio=r)
    with pytest.raises(ValueError):
        EpisodeStream(20, 0, 1)
    with pytest.raises(ValueError):
        EpisodeStream(0, 8, 1)
    with pytest.raises(ValueError):
        EpisodeStream(20, 8, 1, slot_offset=-1)
    # Python's round: half to even, on the fp64 product
    assert [scripted_count(r, n) for r, n in ((0.25, 10), (0.75, 10), (0.5, 5), (0.5, 1), (0.3, 5), (1.0, 50))] == \
        [2, 8, 2, 0, 2, 50]
    for ratio in np.linspace(0.0, 1.0, 41):
        for n in (1, 5, 20, 50, 200):
            assert scripted_count(float(ratio), n) == round(float(ratio) * n)
    # the host reset chain draws round(ratio * N) scripted agents and then drops the source when ratio < 1
    gi, src, inter, scr, _ = reset_chain.episode_pool(9, 64, 20, 8, scripted_agents_ratio=0.25)
    assert set(scr.sum(1).tolist()) <= {scripted_count(0.25, 20), scripted_count(0.25, 20) - 1}
    s = EpisodeStream(50, 16, 2 ** 64 + 5, scripted_agents_ratio=0.4, slot_offset=7)
    assert (s.sampler.seed, s.sampler.pool_size, s.sampler.n_scripted, s.sampler.drop_source_from_scripted,
            s.sampler.slot_offset) == (5, 16, 20, 1, 7)
    assert EpisodeStream(50, 16, 1, scripted_agents_ratio=1.0).sampler.drop_source_from_scripted == 0


def test_rank_slot_offsets_are_disjoint():
    from melissa_b200.sharding import rank_slot_offset
    B = 32768
    ranges = [range(rank_slot_offset(k, B), rank_slot_offset(k, B) + B) for k in range(8)]
    assert ranges[0].start == 0 and all(a.stop == b.start for a, b in zip(ranges, ranges[1:]))


@pytest.mark.parametrize("N", [1, 20, 50, 200])
def test_k_probabilities_are_the_exact_interval_shares(N):
    p = k_probabilities(N)
    assert abs(p.sum() - 1.0) < 1e-12
    lo = int(0.1 * N)
    assert p[:lo].sum() == 0.0 and p[lo] > 0
    # the bisection edges are where k changes on the 2^53 grid
    top = 1 << 53
    acc = 0
    for m in range(N + 1):
        if p[m] == 0.0:
            continue
        start = acc
        acc += round(p[m] * top)
        assert k_of_u(start, N) == m and k_of_u(acc - 1, N) == m
        if start > 0:
            assert k_of_u(start - 1, N) < m
    assert acc == top
    # the inner values take 1 / (0.9 N) of the mass each, up to the grid
    inner = p[lo + 1:N - 1]
    if len(inner):
        assert np.allclose(inner, 1.0 / (0.9 * N), rtol=1e-6)
    # same law as numpy's uniform(0.1, 1.0) followed by int(density * N)
    rs = np.random.RandomState(3)
    ks = (rs.uniform(0.1, 1.0, 200000) * N).astype(int)
    counts = np.bincount(ks, minlength=N + 1)
    nz = p > 0
    assert np.abs(counts[nz] / 200000 - p[nz]).max() < 6 * math.sqrt(0.25 / 200000)


def test_inclusion_and_duplicate_helpers():
    p1, p2 = node_inclusion(np.array([0, 1, 10, 20]), 20)
    assert np.allclose(p1, [0, 0.05, 0.5, 1.0]) and np.allclose(p2, [0, 0, 90 / 380, 1.0])
    # a brute-force count on a tiny space: N = 1, G = 2 -> tuples (g, source 0, k = 0 or 1)
    pk = k_probabilities(1)
    want = 10 * 9 / 2 * sum(pk[m] ** 2 for m in range(2)) / 2
    assert math.isclose(expected_duplicate_pairs(10, 1, 2), want)
