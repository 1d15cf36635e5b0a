"""MAAC-R reward across the magnitudes of the PMI network's weights and inputs, on both PMI kernels (path 1: fp32 CUDA
cores; path 2: tcgen05 tensor cores with split fp16 operands), against the CPU oracle, which runs the BatchNorms unfolded
in fp32 and so shares nothing with fold_pmi or the per-unit rebalancing of uavsim_set_pmi_weights.

The networks are edited copies of a PMINetwork state dict: exactly rescaled BatchNorms (ReLU is positively homogeneous,
so the fp32 function is bit-identical while every magnitude the kernels see moves by 2^k), degenerate BatchNorm units,
folded fc1 weights near 10^3, and networks trained on observations of a rollout.  Inputs go far outside the map and into
the origin corner, and the pair counts of an environment group hit the tensor kernel's tile boundaries.  Every run that
the tensor path serves exactly must report pmi_rows_out_of_range = 0; one run beyond its range must count its rows."""
import numpy as np
import pytest
import torch

from gpu_util import max_scaled_err, oracle_params_from_config, oracle_pmi_from_module

pytestmark = pytest.mark.gpu
TOL_TC = 2e-6        # as test_gpu_pmi_tensor.py: fp32-class products on both paths
HIDDEN = [64, 128]   # the constructor default and the shipped configs
PATHS = [1, 2]
BRANCH_BN = ("bn_comm", "bn_obs", "bn_boundary_state")


def _cfg(n, m, **kw):
    from marl_uavs_targets_tracking_b200 import default_config
    return default_config("MAAC-R", n, m, **kw)


def _net(hidden, seed=1, sd=None):
    """A PMINetwork in eval mode: perturbed BatchNorm statistics (as test_gpu_pmi_tensor.py), or the given state dict."""
    from marl_uavs_targets_tracking_b200 import PMINetwork
    torch.manual_seed(seed)
    net = PMINetwork(hidden_dim=hidden)
    if sd is None:
        for bn in BRANCH_BN + ("bn1",):
            getattr(net, bn).running_mean.normal_(0, 0.3)
            getattr(net, bn).running_var.uniform_(0.5, 1.5)
    else:
        net.load_state_dict(sd)
    return net.eval()


def _edited(net, edit):
    """A new network whose state dict is `net`'s after edit(sd) (sd: name -> float64 tensor copy, edited in place)."""
    sd = {k: v.detach().cpu().clone() for k, v in net.state_dict().items()}
    work = {k: v.double() for k, v in sd.items() if v.is_floating_point()}
    edit(work)
    for k, v in work.items():
        sd[k] = v.to(sd[k].dtype)
    return _net(net.hidden_dim, sd=sd)


def _rescaled(net, k):
    """Branch BatchNorms' weight and bias times 2^k, fc1.weight times 2^-k: the same fp32 function."""
    def edit(sd):
        for bn in BRANCH_BN:
            sd[bn + ".weight"] *= 2.0 ** k
            sd[bn + ".bias"] *= 2.0 ** k
        sd["fc1.weight"] *= 2.0 ** -k
    return _edited(net, edit)


def _run(oracle, pmi, path, n=10, m=10, E=48, T=6, cfg=None, state=None, seed=21, act_seed=5):
    """Steps E environments T times on PMI path `path` and replays them in the oracle.  Returns the worst scaled reward
    error, the per-step GPU and oracle rewards and the out-of-range row count of the run."""
    from marl_uavs_targets_tracking_b200 import BatchedEnvironment
    cfg = cfg or _cfg(n, m)
    e = cfg["environment"]
    env = BatchedEnvironment(n, m, e["x_max"], e["y_max"], e["na"], n_envs=E, device="cuda:0", seed=seed)
    env.set_pmi_path(path)
    if state is None:
        env.reset(cfg)
    else:
        env.set_state(cfg, *state)
    P = oracle_params_from_config(cfg, n, m)
    opmi = oracle_pmi_from_module(pmi)
    st = {k: np.ascontiguousarray(v.cpu().numpy()) for k, v in env.get_state().items()}
    worst, got, ref = 0.0, [], []
    for t in range(T):
        a = env.random_actions(act_seed, t).cpu().numpy().copy()
        r = oracle.step_batch(P, 2, float(cfg["cooperative"]), opmi, st, a, nthreads=8)
        _, rew4, _ = env.step_device(cfg, pmi)
        g = rew4[0].double().cpu().numpy()
        assert np.isfinite(g).all(), (path, t)
        worst = max(worst, max_scaled_err(g, r["rew4"][0]))
        got.append(g)
        ref.append(r["rew4"][0])
    oor = env.episode_stats().get("pmi_rows_out_of_range")
    env.close()
    return {"worst": worst, "got": got, "ref": ref, "oor": oor}


def _check(res, what):
    print(what, "worst %.2e" % res["worst"], "out-of-range rows", res["oor"])
    assert res["worst"] <= TOL_TC, (what, res["worst"])
    assert res["oor"] == 0, (what, res["oor"])


# ---------------------------------------------------------------------------------------------------- A. exact rescaling
@pytest.mark.parametrize("path", PATHS)
@pytest.mark.parametrize("hidden", HIDDEN)
def test_exact_rescaling_of_branch_batchnorms(oracle, hidden, path):
    """2^k on the branch BatchNorms and 2^-k on fc1 for k in -16..16: the oracle's rewards are bit-identical across k
    (this checks the construction), both kernels stay within tolerance at every k, and both are bit-identical across k
    (the CUDA-core kernel by fp32 exactness, the tensor kernel because the upload rebalances every unit by a power of two
    chosen from quantities that scale with it)."""
    base = _net(hidden, seed=3)
    runs = {k: _run(oracle, _rescaled(base, k), path) for k in (-16, -12, -8, -4, 0, 4, 8, 12, 16)}
    print({k: "%.1e" % r["worst"] for k, r in runs.items()})
    for k, r in runs.items():
        for t in range(len(r["ref"])):
            assert np.array_equal(r["ref"][t], runs[0]["ref"][t]), ("oracle not invariant", k, t)
    for k, r in runs.items():
        _check(r, "k=%d" % k)
    for k, r in runs.items():
        for t in range(len(r["got"])):
            assert np.array_equal(r["got"][t], runs[0]["got"][t]), ("kernel not invariant", k, t)


# ------------------------------------------------------------------------------------------------ B. degenerate BatchNorm
def _degenerate(sd, hidden):
    """In every BatchNorm: running_var = 0, weight = 0, negative weight, and a running_mean that keeps the unit at zero
    after the ReLU, on disjoint groups of units."""
    g = hidden // 8
    for bn in BRANCH_BN + ("bn1",):
        w, rm, rv = sd[bn + ".weight"], sd[bn + ".running_mean"], sd[bn + ".running_var"]
        rv[0:g] = 0.0
        w[g:2 * g] = 0.0
        w[2 * g:3 * g] = -(w[2 * g:3 * g].abs() + 0.5)
        w[3 * g:4 * g] = w[3 * g:4 * g].abs() + 0.1
        rm[3 * g:4 * g] = 1e4


@pytest.mark.parametrize("path", PATHS)
@pytest.mark.parametrize("hidden", HIDDEN)
def test_degenerate_batchnorm_units(oracle, hidden, path):
    base = _net(hidden, seed=5)
    _check(_run(oracle, _edited(base, lambda sd: _degenerate(sd, hidden)), path), "degenerate units")

    def dead_branch(sd):  # the observation branch is zero after the ReLU for every input
        sd["bn_obs.weight"].zero_()
        sd["bn_obs.bias"].fill_(-1.0)
    _check(_run(oracle, _edited(base, dead_branch), path), "dead observation branch")


# ----------------------------------------------------------------------------------------------------- C. large folded fc1
def _large_fc1(sd, target=1e3):
    """bn1.running_var = 0 on every 9th unit, fc1 rows of those units scaled so that the largest folded weight is about
    `target`, fc2 weights of the units scaled down by the same factor (the logits stay of order one)."""
    units = torch.arange(0, sd["bn1.weight"].numel(), 9)
    sd["bn1.running_var"][units] = 0.0
    s1 = sd["bn1.weight"] / torch.sqrt(sd["bn1.running_var"] + 1e-5)
    for u in units.tolist():
        folded = (sd["fc1.weight"][u] * s1[u]).abs().max()
        c = float(target / folded)
        sd["fc1.weight"][u] *= c
        sd["fc2.weight"][0, u] /= c * float(s1[u].abs())


@pytest.mark.parametrize("path", PATHS)
@pytest.mark.parametrize("hidden", HIDDEN)
def test_large_folded_fc1_weights(oracle, hidden, path):
    from marl_uavs_targets_tracking_b200.pmi import fold_pmi
    net = _edited(_net(hidden, seed=6), _large_fc1)
    assert 900 < np.abs(fold_pmi(net)["w1"]).max() < 1100
    _check(_run(oracle, net, path), "folded |w1| ~ 1e3")


def test_weights_beyond_fp16_range_use_the_cuda_core_kernel(oracle):
    """Folded fc1 weights of ~1e7 cannot be held by the fp16 operands of the tensor path even after rebalancing: the
    automatic choice takes the CUDA-core kernel (exact), asking for the tensor path fails, and a swarm only the tensor
    path can hold (n = 128) refuses the weights at upload."""
    from marl_uavs_targets_tracking_b200 import BatchedEnvironment, UavSimError
    net = _edited(_net(128, seed=7), lambda sd: _large_fc1(sd, target=1e7))
    _check(_run(oracle, net, 0), "automatic, folded |w1| ~ 1e7")
    for n, path in ((10, 2), (128, 0)):
        cfg = _cfg(n, 5)
        env = BatchedEnvironment(n, 5, 2000, 2000, 12, n_envs=2, device="cuda:0", seed=21)
        env.set_pmi_path(path)
        env.reset(cfg)
        with pytest.raises(UavSimError):
            env.step_device(cfg, net)
        env.close()


# ---------------------------------------------------------------------------------------------------- D. trained networks
def _rollout_obs(n, m, E, T, seed):
    from marl_uavs_targets_tracking_b200 import BatchedEnvironment
    cfg = _cfg(n, m)
    env = BatchedEnvironment(n, m, 2000, 2000, 12, n_envs=E, device="cuda:0", seed=seed)
    env.reset(cfg)
    obs = []
    for t in range(T):
        env.random_actions(seed, t)
        o, _, _ = env.step_device(cfg, None)
        obs.append(o.clone())
    env.close()
    return torch.stack(obs).reshape(-1, 12)   # [(t, env) x n_uav, 12]: one "timestep" per environment-step


@pytest.mark.parametrize("hidden", HIDDEN)
def test_trained_networks(oracle, hidden):
    """The regime MAAC-R runs in: PMINetwork.train_pmi on observations of a seeded rollout (on the device), then both
    paths with the trained network (after 1 and after 36 rounds)."""
    from marl_uavs_targets_tracking_b200 import PMINetwork
    n = m = 10
    data = _rollout_obs(n, m, 32, 30, seed=11)
    torch.manual_seed(hidden)
    net = PMINetwork(hidden_dim=hidden).to("cuda:0")
    cfg = _cfg(n, m)
    done = 0
    for rounds in (1, 36):
        while done < rounds:
            net.train_pmi(cfg, data, n)
            done += 1
        net.eval()
        for path in PATHS:
            _check(_run(oracle, net, path, E=64, T=8), "trained %d rounds, path %d" % (rounds, path))


# -------------------------------------------------------------------------------------------------------- E. input range
def _far_state(n, m, E, centres, rng, spread=60.0):
    """UAVs in clusters (UAV i in cluster i % len(centres)) within `spread` m of the centres; targets on the map."""
    c = np.asarray(centres, np.float64)[np.arange(n) % len(centres)]
    ux = c[None, :, 0] + rng.uniform(0, spread, (E, n))
    uy = c[None, :, 1] + rng.uniform(0, spread, (E, n))
    uh = rng.uniform(-np.pi, np.pi, (E, n))
    ua = np.zeros((E, n), np.int32)
    tx, ty = rng.uniform(0, 2000, (E, m)), rng.uniform(0, 2000, (E, m))
    th = rng.uniform(-np.pi, np.pi, (E, m))
    return ux, uy, uh, ua, tx, ty, th


@pytest.mark.parametrize("path", PATHS)
@pytest.mark.parametrize("hidden", HIDDEN)
def test_uavs_far_outside_the_map_and_in_the_origin_corner(oracle, hidden, path):
    """obs[9:11] = position / dc reaches 40 at 2e4 m: pair inputs up to 1 600, inside the tensor path's range."""
    n, m, E = 12, 6, 32
    rng = np.random.default_rng(4)
    st = _far_state(n, m, E, [(1e4, 1.2e4), (2e4, 1.5e4), (1.5e4, 2e4), (0.0, 0.0)], rng)
    _check(_run(oracle, _net(hidden, seed=8), path, n=n, m=m, E=E, T=6, state=st), "far clusters")


def test_inputs_beyond_the_tensor_range_are_counted(oracle):
    """A cluster at 2e5 m (obs[9:11] ~ 400, pair inputs ~ 1.6e5) is beyond any input range the fp16 activations of the
    tensor path hold: every pair row of that cluster is counted (and only those), the CUDA-core kernel still matches
    the oracle and counts nothing."""
    n, m, E, T = 8, 4, 5, 3
    rng = np.random.default_rng(5)
    # UAVs 0, 2, 4, 6 in the far cluster, 1 and 5 near the map centre, 3 and 7 alone
    st = _far_state(n, m, E, [(2e5, 2e5), (1000.0, 1000.0), (2e5, 2e5), (5000.0, 500.0)], rng, spread=40.0)
    st[0][:, 7] += 3000.0
    net = _net(128, seed=9)
    far = _run(oracle, net, 2, n=n, m=m, E=E, T=T, state=st)
    print("far cluster, tensor path: out-of-range rows", far["oor"], "worst %.2e" % far["worst"])
    assert far["oor"] == E * T * 4 * 3
    _check(_run(oracle, net, 1, n=n, m=m, E=E, T=T, state=st), "far cluster, CUDA-core path")


# -------------------------------------------------------------------------------------- F. pair-count boundaries (path 2)
LAYOUTS = {0: [], 2: [2], 126: [9, 7, 4], 128: [9, 8], 130: [11, 4, 3, 2], 254: [16, 4, 2], 256: [16, 4, 2, 2],
           258: [16, 4, 3], 16256: [128]}


def _layout_state(clusters, n, m, E, rng, x_max):
    """Clusters of the given sizes on a 10 m grid (diameter <= 150 m: still within dp = 200 m after a 20 m move of
    each UAV), cluster centres 1 km apart, every other UAV alone on a 600 m grid."""
    ux, uy = np.empty(n), np.empty(n)
    i = 0
    for c, k in enumerate(clusters):
        for j in range(k):
            ux[i] = 500.0 + 1000.0 * c + 10.0 * (j % 11)
            uy[i] = 500.0 + 10.0 * (j // 11)
            i += 1
    for j in range(n - i):
        ux[i + j] = 300.0 + 600.0 * (j % 15)
        uy[i + j] = 1500.0 + 600.0 * (j // 15)
    rep = lambda a: np.repeat(a[None], E, 0)  # noqa: E731
    uh = rng.uniform(-np.pi, np.pi, (E, n))
    tx, ty = rng.uniform(0, x_max, (E, m)), rng.uniform(0, x_max, (E, m))
    return rep(ux), rep(uy), uh, np.zeros((E, n), np.int32), tx, ty, rng.uniform(-np.pi, np.pi, (E, m))


@pytest.mark.parametrize("E", [1, 3])
@pytest.mark.parametrize("pairs", sorted(LAYOUTS))
def test_pair_counts_at_tile_boundaries(oracle, pairs, E):
    """n = 128: ordered neighbour-pair totals of one environment around the tensor kernel's 128-row tiles and 2-tile
    sets (0 .. 258) and the most a group holds (16 256)."""
    n, m, x_max = 128, 5, 10000.0
    assert sum(k * (k - 1) for k in LAYOUTS[pairs]) == pairs
    cfg = _cfg(n, m, environment__x_max=x_max, environment__y_max=x_max)
    st = _layout_state(LAYOUTS[pairs], n, m, E, np.random.default_rng(pairs), x_max)
    # the layout keeps its pair count through the first step (the 20 m moves change no neighbour relation)
    d = np.hypot(st[0][0][:, None] - st[0][0][None], st[1][0][:, None] - st[1][0][None])
    assert int(((d <= 150.0) & (d > 0)).sum()) == pairs and int(((d > 150.0) & (d <= 240.0)).sum()) == 0
    _check(_run(oracle, _net(128, seed=10), 2, n=n, m=m, E=E, T=1, cfg=cfg, state=st), "n=128 pairs=%d E=%d" % (pairs, E))


@pytest.mark.parametrize("E", [1, 2, 147, 148, 149, 1001])
def test_only_the_last_environment_has_neighbours(oracle, E):
    n, m = 10, 10
    rng = np.random.default_rng(E)
    alone = [(200.0 + 400.0 * (i % 5), 300.0 + 800.0 * (i // 5)) for i in range(n)]
    st = list(_far_state(n, m, E, alone, rng, spread=10.0))
    st[0][-1, :4] = 1000.0 + 30.0 * np.arange(4)
    st[1][-1, :4] = 1900.0
    _check(_run(oracle, _net(64, seed=12), 2, n=n, m=m, E=E, T=1, state=st), "neighbours in env %d only" % (E - 1))


@pytest.mark.parametrize("E", [1, 2, 147, 148, 149, 1001, 16385])
def test_partial_last_groups(oracle, E):
    _check(_run(oracle, _net(128, seed=13), 2, E=E, T=3), "E=%d" % E)
