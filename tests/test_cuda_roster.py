"""The standard rollout kernel with the bench game compiled in (a roster: extermination, agent + 2 terminators): it is
the kernel a bench-shaped rollout launches, and in every lane layout and occupancy it is compiled for it computes what the
kernel that reads the game from the parameters computes (ZS_NO_ROSTER) — observations, reward bits, flags, final state and
episode statistics — and what the oracle computes."""
import re

import numpy as np
import pytest
import torch

from libzombsole_b200 import abi
from test_cuda_properties import engine, state_snapshot, assert_same_state

pytestmark = pytest.mark.gpu

# (lanes per env, CTAs per SM): every roster kernel zs_create can pick
INSTANTIATIONS = [("16", "4"), ("16", "6"), ("16", "7"), ("32", "4"), ("32", "7")]


def _rollout(monkeypatch, lanes, occ, K, roster, N=1024, seed=31, mes=30, name="c1_bridge_ext", kernels=None):
    """A fused K-step rollout of the bench game (on the bridge map unless `name` says otherwise) from a fresh world, on an
    action tape; short episodes (mes) so that every launch meets world inits.  occ=None leaves the occupancy to
    zs_create; a list as `kernels` receives the names of the step kernels the rollout launched."""
    monkeypatch.setenv("ZS_LANES_PER_ENV", lanes)
    if occ is None:
        monkeypatch.delenv("ZS_OCC", raising=False)
    else:
        monkeypatch.setenv("ZS_OCC", occ)
    if roster:
        monkeypatch.delenv("ZS_NO_ROSTER", raising=False)
    else:
        monkeypatch.setenv("ZS_NO_ROSTER", "1")
    eng, cfg, m = engine(name, N, seed=seed, mes=mes)
    assert eng.lanes_per_env() == int(lanes)
    obs = eng.new_obs(3)
    rew, term, trunc = eng.new_outputs(K)
    acts = torch.zeros((K, N, eng.A), dtype=torch.int32, device=eng.device)
    for s in range(K):
        eng.fill_synthetic_actions(s, acts[s])
    run = lambda: eng.rollout(K, 0, acts, abi.ACTIONS_DISCRETE, obs, rew, term, trunc)  # noqa: E731
    if kernels is None:
        run()
    else:
        kernels += _kernels_launched(run)
    out = dict(obs=obs.cpu().numpy(), rew=rew.cpu().numpy().view(np.uint64), term=term.cpu().numpy(),
               trunc=trunc.cpu().numpy(), stats=eng.episode_stats().cpu().numpy(), state=state_snapshot(eng), M=eng.M)
    eng.close()
    return out, cfg, m


def _kernels_launched(fn):
    from torch.profiler import profile, ProfilerActivity
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return [e.name for e in prof.events() if "zs_sim_kernel" in e.name]


@pytest.mark.parametrize("roster", [True, False])
def test_bench_rollout_launches_the_roster_kernel(monkeypatch, roster):
    """bench.py's workload (4,096 envs, K=20 on an action tape) runs zs_sim_kernel<MODE_STEP, 16, G, 1, OCC, ROS> with the
    bench roster compiled in; ZS_NO_ROSTER gives ROS = 0."""
    if not roster:
        monkeypatch.setenv("ZS_NO_ROSTER", "1")
    N, K = 4096, 20
    eng, cfg, m = engine("c1_bridge_ext", N, seed=5)
    obs = eng.new_obs()
    rew, term, trunc = eng.new_outputs(K)
    acts = torch.zeros((K, N, eng.A), dtype=torch.int32, device=eng.device)
    names = _kernels_launched(lambda: eng.rollout(K, 0, acts, abi.ACTIONS_DISCRETE, obs, rew, term, trunc))
    eng.close()
    ros = 1 + abi.RULES["extermination"] + 4 * 3 if roster else 0
    pat = re.compile(r"zs_sim_kernel<0, 16, (16|32), 1, \d+, %d>" % ros)
    assert names and all(pat.search(n) for n in names), names


@pytest.mark.parametrize("K", [1, 7, 64])
@pytest.mark.parametrize("lanes,occ", INSTANTIATIONS)
def test_roster_kernel_equals_generic_kernel(monkeypatch, lanes, occ, K):
    a, _, _ = _rollout(monkeypatch, lanes, occ, K, roster=True)
    b, _, _ = _rollout(monkeypatch, lanes, occ, K, roster=False)
    for k in ("obs", "rew", "term", "trunc", "stats"):
        assert np.array_equal(a[k], b[k]), k
    assert_same_state(a["state"], b["state"], a["M"])


@pytest.mark.parametrize("lanes,occ", INSTANTIATIONS)
def test_roster_kernel_matches_oracle(monkeypatch, lanes, occ):
    from oracle import oracle as orc
    K, N = 64, 1024
    a, cfg, m = _rollout(monkeypatch, lanes, occ, K, roster=True, N=N)
    ref = orc.OracleEnv(cfg, m)
    o, r, te, tr = ref.rollout_synthetic(K, 0)
    assert np.array_equal(a["obs"][(K - 1) % 3].reshape(N, -1), o)
    assert np.array_equal(a["rew"].reshape(K, N, 1), r.view(np.uint64))
    assert np.array_equal(a["term"], te) and np.array_equal(a["trunc"], tr)
    assert np.array_equal(a["stats"], ref.stats())


# the bench game on the maps at the edges of the accepted geometry (tests/maps): 143 cells (3 mod 4, no TMA template), one
# row of 81 cells, and 2,047 x 32 = 65,504 cells (moves, hits and distances at cell indices past 32,767)
EDGE_MAPS = [("bench_odd_cells", 1024), ("bench_strip_row", 1024), ("bench_wide_max", 64)]


@pytest.mark.parametrize("lanes", ["16", "32"])
@pytest.mark.parametrize("name,N", EDGE_MAPS)
def test_roster_kernel_on_edge_maps(monkeypatch, name, N, lanes):
    """The roster kernel launches on these maps in both lane layouts, and computes what the kernel that reads the game from
    the parameters computes and what the oracle computes."""
    from oracle import oracle as orc
    K = 64
    names = []
    a, cfg, m = _rollout(monkeypatch, lanes, None, K, roster=True, N=N, name=name, kernels=names)
    ros = 1 + abi.RULES["extermination"] + 4 * 3
    pat = re.compile(r"zs_sim_kernel<0, 16, %s, 1, \d+, %d>" % (lanes, ros))
    assert names and all(pat.search(n) for n in names), names
    b, _, _ = _rollout(monkeypatch, lanes, None, K, roster=False, N=N, name=name)
    for k in ("obs", "rew", "term", "trunc", "stats"):
        assert np.array_equal(a[k], b[k]), k
    assert_same_state(a["state"], b["state"], a["M"])
    ref = orc.OracleEnv(cfg, m)
    o, r, te, tr = ref.rollout_synthetic(K, 0)
    assert np.array_equal(a["obs"][(K - 1) % 3].reshape(N, -1), o)
    assert np.array_equal(a["rew"].reshape(K, N, 1), r.view(np.uint64))
    assert np.array_equal(a["term"], te) and np.array_equal(a["trunc"], tr)
    assert np.array_equal(a["stats"], ref.stats())
    assert a["stats"][0] > 0  # episodes ended and worlds were re-initialised inside the rollout
