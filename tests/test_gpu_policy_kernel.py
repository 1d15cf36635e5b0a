"""The fused policy kernel (csrc/policy.cuh) against an fp64 reference of the same operation: softmax(fc2(relu(fc1(x))))
on the fp32 weights cast to float64, and the inverse-CDF draw of the row's Philox uniform (tests/philox_ref.py, the
kernel's full key (row_lo, row_hi, counter_lo, counter_hi; seed)) on the fp64 cumulative probabilities.  Both kernel
forms are checked: the plain one through `uavsim_policy_sample`, the PDL one through `uavsim_run_policy`.

The probability tolerance is a rounding-error bound, not a tuned constant.  With u = 2^-24 and g(n) = n u / (1 - n u):
  hidden unit  e_j     = g(13) (|b1_j| + sum_k |w1_jk x_k|)                 12 fmas onto the bias
  logit        delta_a = g(ceil(H/2) + 2) (sum_j |w2_aj| h_j + |b2_a|)      two fma chains of ceil(H/2) units, their sum,
                         + sum_j |w2_aj| e_j (1 + u)                         the bias; plus the hidden errors carried
  probability  |p - p64| <= 2 (p64 (2 Delta + (A + 4) 2^-23) + 2^-126),  Delta = max_a delta_a
(a softmax ratio moves by at most exp(2 Delta); expf, the sum, the reciprocal and the product add A + 4 roundings; 2^-126
covers results below the normal range).  The factor 2 is the only slack.  A dropped, mis-paired or duplicated hidden unit, a
missing bias or a wrong fc2 row moves a logit by a whole w2 h term, far outside the bound.

A drawn action must be consistent with the fp64 rule: cdf64[a-1] - tau <= u53 <= cdf64[a] + tau, tau = the row's summed
probability bound + 2^-24 (the kernel rounds the uniform to fp32), and have a non-zero probability in the kernel's own output.
At most 1e-5 of the rows may draw another action than the fp64 inverse CDF, and only a neighbouring one.
"""
import ctypes as C
import math

import numpy as np
import pytest
import torch

from philox_ref import philox4x32_10, u53

from marl_uavs_targets_tracking_b200 import _cabi

DEV = "cuda:0"
U = 2.0 ** -24
MASK64 = (1 << 64) - 1
SEED_HI = 0x9E3779B97F4A7C15  # both 32-bit halves of the seed non-zero
KEYS = {"k0": (99, 5), "ctr2^32+5": (99, (1 << 32) + 5), "ctr2^64-1": (99, MASK64), "seedhi": (SEED_HI, 5)}

# draw edge cases at seed 99, row 0, counter high word 0 (recomputed and asserted by test_draw_edge_counters)
CLAMP_COUNTERS = (6_838_284, 9_792_843, 16_943_529)  # u53 >= 1 - 2^-25: rounds to 1.0f
TINY_U_COUNTER = 20_278_259                           # u53 = 1.66e-8


def gamma(n):
    return n * U / (1 - n * U)


def uniforms(rows, seed, counter):
    """The kernel's u53 of rows 0 .. rows-1 at (seed, counter), float64 numpy."""
    r = np.arange(rows, dtype=np.uint64)
    c = counter & MASK64
    v = philox4x32_10(r & np.uint64(0xFFFFFFFF), r >> np.uint64(32), c & 0xFFFFFFFF, c >> 32, seed)
    return u53(v[0], v[1])


def reference(net, x, chunk=1 << 20):
    """fp64 probabilities [B,A] and their error bound [B,A] (module docstring), float64 on the device of x."""
    w1, b1, w2, b2 = (p.detach().double() for p in (net.fc1.weight, net.fc1.bias, net.fc2.weight, net.fc2.bias))
    H, A = w1.shape[0], w2.shape[0]
    g_h, g_l = gamma(13), gamma((H + 1) // 2 + 2)
    aw1, aw2 = w1.abs().T, w2.abs().T
    ps, bs = [], []
    for s in range(0, x.shape[0], chunk):
        xs = x[s:s + chunk].double()
        h = (xs @ w1.T + b1).clamp_min(0)
        e = g_h * (b1.abs() + xs.abs() @ aw1)
        delta = g_l * (h @ aw2 + b2.abs()) + (e @ aw2) * (1 + U)
        p = torch.softmax(h @ w2.T + b2, dim=1)
        ps.append(p)
        bs.append(2 * (p * (2 * delta.max(1, keepdim=True).values + (A + 4) * 2.0 ** -23) + 2.0 ** -126))
    return torch.cat(ps), torch.cat(bs)


def check_probs(probs, p64, bound, tag):
    """|p - p64| <= bound everywhere; returns the worst error / bound ratio."""
    ratio = ((probs.double() - p64).abs() / bound)
    worst = float(ratio.max())
    r = int(ratio.max(1).values.argmax())
    print("%s: worst |p - p64| / bound = %.3g" % (tag, worst))
    assert worst <= 1.0, (tag, worst, r, probs[r].tolist(), p64[r].tolist())
    return worst


def check_draw(act, probs, p64, bound, u, tag):
    """The draw of every row against the fp64 inverse CDF of its uniform (module docstring).  Returns the number of rows
    that differ from the fp64 rule."""
    B, A = p64.shape
    a = act.long()
    assert int(a.min()) >= 0 and int(a.max()) < A, tag
    ud = torch.from_numpy(np.ascontiguousarray(u)).to(p64.device)
    cdf = p64.cumsum(1)
    tau = bound.sum(1) + U
    lo = torch.where(a > 0, cdf.gather(1, (a - 1).clamp_min(0)[:, None])[:, 0], torch.zeros_like(ud))
    hi = torch.where(a < A - 1, cdf.gather(1, a[:, None])[:, 0], torch.full_like(ud, math.inf))
    bad = ~((lo - tau <= ud) & (ud <= hi + tau))
    if bool(bad.any()):
        r = int(bad.nonzero()[0])
        raise AssertionError("%s: row %d draws %d with u53 = %.17g, fp64 cdf %s" % (tag, r, int(a[r]), float(ud[r]),
                                                                                  cdf[r].tolist()))
    if probs is not None:
        assert bool((probs.gather(1, a[:, None]) > 0).all()), tag + ": an action of probability 0 was drawn"
    expect = (cdf[:, :-1] <= ud[:, None]).sum(1)
    differ = int((a != expect).sum())
    assert differ <= 1e-5 * B, (tag, differ, B)
    assert int((a - expect).abs().max()) <= 1, tag
    return differ


def make_net(H, A, weights="fresh", seed=0):
    from marl_uavs_targets_tracking_b200.rollout import PolicyNet
    torch.manual_seed(seed)
    net = PolicyNet(12, H, A).to(DEV)
    with torch.no_grad():
        if weights == "fc2x8":     # peaked softmax
            net.fc2.weight.mul_(8)
        elif weights == "fc2x64":  # nearly one-hot
            net.fc2.weight.mul_(64)
        elif weights == "zero-prob":  # the first, a middle and the last action at probability exactly 0 in fp32
            net.fc2.bias[[0, A // 2, A - 1]] = -200.0
        else:
            assert weights == "fresh"
    return net


def make_inputs(kind, rows, seed):
    g = torch.Generator(device=DEV).manual_seed(seed)
    if kind == "randn":
        return torch.randn(rows, 12, device=DEV, generator=g)
    if kind == "zero":
        return torch.zeros(rows, 12, device=DEV)
    x = torch.rand(rows, 12, device=DEV, generator=g) * 2 - 1
    if kind == "far":  # far-away UAVs: relative coordinates up to +-200
        return x * 200
    assert kind == "obs"  # observation-shaped: entries in [-1, 1], self terms up to +-4, absent entities as -1 blocks
    x[:, :4] *= 4
    absent = torch.rand(rows, 2, device=DEV, generator=g) < 0.3
    x[:, 4:8][absent[:, 0]] = -1.0
    x[:, 8:12][absent[:, 1]] = -1.0
    return x


def multipass_rows():
    """Enough 512-row iterations that every CTA of the persistent grid makes >= 3 passes even at 16 CTAs per SM (2048 /
    128 threads, the most an SM can hold), plus 3 so the row count is not a multiple of 4."""
    sms = torch.cuda.get_device_properties(DEV).multi_processor_count
    return 3 * sms * 16 * 512 + 3


# ------------------------------------------------------------------------------------------------ CPU: argument checks
def _weights(hidden=64, n_actions=12, state_dim=12, null=False):
    """UavSimPolicyWeights with fake, 16-byte aligned pointers (never dereferenced by a refused call)."""
    w = _cabi.UavSimPolicyWeights()
    w.state_dim, w.hidden, w.n_actions = state_dim, hidden, n_actions
    w.w1, w.b1, w.w2, w.b2 = (0, 0, 0, 0) if null else (0x1000, 0x2000, 0x3000, 0x4000)
    return w


BAD_SIZES = [dict(hidden=0), dict(hidden=513), dict(n_actions=1), dict(n_actions=17), dict(state_dim=11)]


def _sample(lib, obs, rows, w):
    return lib.uavsim_policy_sample(C.c_void_p(obs), rows, C.byref(w) if w is not None else None, C.c_uint64(1),
                                    C.c_uint64(1), C.c_void_p(0x5000), None, 0, None)


def test_policy_sample_refuses_unsupported_weights():
    """With rows = 0 these are refused before anything else could happen, so the call is safe with or without a device."""
    lib = _cabi.load()
    for kw in BAD_SIZES:
        assert _sample(lib, 0x100, 0, _weights(**kw)) == -3, kw  # UAVSIM_ERR_UNSUPPORTED
    assert _sample(lib, 0x100, 0, _weights(null=True)) == -1      # UAVSIM_ERR_ARG
    assert _sample(lib, 0x100, 0, None) == -1
    assert b"NULL" in lib.uavsim_last_error()


@pytest.mark.skipif(torch.cuda.is_available(), reason="fake pointers: must never reach a launch")
def test_policy_sample_argument_checks_come_before_the_device():
    lib = _cabi.load()
    for kw in BAD_SIZES:
        assert _sample(lib, 0x100, 8, _weights(**kw)) == -3, kw
    assert _sample(lib, 0x100, 8, _weights(null=True)) == -1
    assert _sample(lib, 0, 8, _weights()) == -1                   # NULL obs
    assert _sample(lib, 0x100, 0, _weights()) == 0                # nothing to do
    for off in (4, 8, 12):                                        # obs off a 16-byte boundary
        assert _sample(lib, 0x100 + off, 8, _weights()) == -1, off
        assert b"aligned" in lib.uavsim_last_error()
    assert _sample(lib, 0x100, 8, _weights()) > 0                 # valid arguments: the missing device is reported


def test_draw_edge_counters():
    """The counters the draw edge tests use give the uniforms they claim (seed 99, row 0)."""
    for c in CLAMP_COUNTERS:
        u = float(uniforms(1, 99, c)[0])
        # rounds to 1.0f: without the clamp u * sum == sum and a zero-probability last action would be drawn
        assert u >= 1 - 2.0 ** -25 and np.float32(u) == np.float32(1.0), (c, u)
    u = float(uniforms(1, 99, TINY_U_COUNTER)[0])
    assert 1.6e-8 < u < 1.7e-8, u


# ------------------------------------------------------------------------------------------------ GPU: the plain kernel
# (A, H, rows, inputs, weights, key).  Every A of every AP instance with and without padding (AP = 4: 2..4, 8: 5..8,
# 12: 9..12, 16: 13..16), odd H (a zero padding unit), H > 384 (more than 48 KB of shared memory), row tails, the clamped
# reads of the last row, and the multi-pass grid.
CASES = [
    (2, 1, 1, "randn", "fresh", "k0"),
    (3, 2, 2, "obs", "fresh", "ctr2^32+5"),
    (4, 3, 3, "randn", "fc2x8", "k0"),
    (5, 127, 4, "randn", "zero-prob", "ctr2^64-1"),
    (8, 128, 5, "zero", "fresh", "seedhi"),
    (9, 129, 511, "obs", "fc2x64", "k0"),
    (12, 384, 512, "far", "fresh", "ctr2^64-1"),
    (13, 385, 513, "randn", "zero-prob", "k0"),
    (16, 511, 100_003, "obs", "zero-prob", "ctr2^32+5"),
    (16, 512, 100_003, "randn", "fc2x8", "seedhi"),
    (2, 512, 100_003, "randn", "fc2x64", "ctr2^64-1"),
    (3, 385, 100_003, "obs", "fc2x8", "seedhi"),
    (5, 1, 513, "far", "fresh", "k0"),
    (9, 3, 100_003, "zero", "fc2x64", "ctr2^32+5"),
    (13, 129, 100_003, "far", "fc2x8", "k0"),
    (8, 2, 511, "obs", "fc2x64", "seedhi"),
    # the four cases of the earlier torch-forward test
    (12, 128, 100_003, "randn", "fresh", "k0"),
    (12, 64, 7, "randn", "fresh", "k0"),
    (5, 128, 4097, "randn", "fresh", "k0"),
    (16, 256, 1000, "randn", "fresh", "k0"),
    # every CTA makes >= 3 passes (13 at AP = 4, 25 at AP = 8..16 with today's register counts on 148 SMs)
    (4, 128, "multipass", "obs", "fresh", "ctr2^64-1"),
    (16, 128, "multipass", "randn", "fc2x8", "seedhi"),
]


def case_id(c):
    return "A%s-H%s-rows%s-%s-%s-%s" % c


@pytest.mark.gpu
@pytest.mark.parametrize("A,H,rows,inputs,weights,key", CASES, ids=[case_id(c) for c in CASES])
def test_policy_kernel_matches_fp64_reference(A, H, rows, inputs, weights, key):
    from marl_uavs_targets_tracking_b200.rollout import fused_policy_sample
    rows = multipass_rows() if rows == "multipass" else rows
    seed, counter = KEYS[key]
    net = make_net(H, A, weights, seed=31 * H + A)
    x = make_inputs(inputs, rows, seed=7 * H + A)
    act, probs = fused_policy_sample(net, x, seed, counter, want_probs=True)
    assert act.dtype == torch.int32 and act.shape == (rows,) and probs.shape == (rows, A)
    act_only, none = fused_policy_sample(net, x, seed, counter)
    assert none is None and torch.equal(act, act_only)  # the probability output does not change the draw
    tag = case_id((A, H, rows, inputs, weights, key))
    p64, bound = reference(net, x)
    check_probs(probs, p64, bound, tag)
    if weights == "zero-prob":
        assert bool((probs[:, [0, A // 2, A - 1]] == 0).all())
    if weights == "fresh" and inputs == "randn":  # torch's own fp32 forward, as before
        with torch.no_grad():
            assert float((probs - net(x)).abs().max()) <= 2e-6
    differ = check_draw(act, probs, p64, bound, uniforms(rows, seed, counter), tag)
    # the next counter (2^64 - 1 wraps to 0) draws from its own uniforms; the same counter again is reproducible
    nxt = (counter + 1) & MASK64
    act2, _ = fused_policy_sample(net, x, seed, nxt)
    differ += check_draw(act2, probs, p64, bound, uniforms(rows, seed, nxt), tag + " next counter")
    assert torch.equal(act, fused_policy_sample(net, x, seed, counter)[0])
    if weights == "fresh" and rows > 1000:
        assert float((act != act2).float().mean()) > 0.5
    print("%s: %d draws differ from the fp64 inverse CDF" % (tag, differ))


@pytest.mark.gpu
def test_hidden_sizes_alternate_on_one_instance():
    """H = 512, 128, 512, 385 on the AP = 16 instance: the dynamic shared memory limit raised for 64 KB stays raised."""
    from marl_uavs_targets_tracking_b200.rollout import fused_policy_sample
    x = make_inputs("obs", 4099, seed=3)
    u = uniforms(4099, 99, 5)
    for H in (512, 128, 512, 385):
        net = make_net(H, 16, seed=H)
        act, probs = fused_policy_sample(net, x, 99, 5, want_probs=True)
        p64, bound = reference(net, x)
        check_probs(probs, p64, bound, "H%d" % H)
        check_draw(act, probs, p64, bound, u, "H%d" % H)


@pytest.mark.gpu
@pytest.mark.parametrize("H,A,weights", [(128, 12, "fresh"), (128, 5, "fresh"), (256, 16, "fresh"), (128, 9, "fc2x8")])
def test_action_frequencies(H, A, weights):
    """Over 2^20 rows with their own distributions, the count of every action against sum_r p64[r, a] (z < 5); and one row
    repeated 200 000 times, chi-square against its probabilities."""
    from marl_uavs_targets_tracking_b200.rollout import fused_policy_sample
    rows = 1 << 20
    net = make_net(H, A, weights, seed=H + A)
    x = make_inputs("randn", rows, seed=H + A)
    act, _ = fused_policy_sample(net, x, 1234, 77)
    p64, _ = reference(net, x)
    cnt = torch.bincount(act.long(), minlength=A).double()
    mean, var = p64.sum(0), (p64 * (1 - p64)).sum(0)
    z = (cnt - mean) / var.sqrt()
    print("H%d A%d %s: max |z| = %.2f" % (H, A, weights, float(z.abs().max())))
    assert float(z.abs().max()) < 5, z.tolist()
    reps = 200_000
    xr = x[:1].repeat(reps, 1).contiguous()
    a, p = fused_policy_sample(net, xr, 1, 1, want_probs=True)
    cnt = torch.bincount(a.long(), minlength=A).double().cpu().numpy()
    e = p64[0].cpu().numpy() * reps
    keep = e > 5
    chi2 = (((cnt - e) ** 2 / np.maximum(e, 1e-30))[keep]).sum()
    assert chi2 < 60, (chi2, cnt, e)


@pytest.mark.gpu
@pytest.mark.parametrize("A", [5, 13, 16])
def test_a_uniform_rounded_to_one_does_not_draw_a_zero_probability_last_action(A):
    """u53 >= 1 - 2^-25 rounds to 1.0f; the kernel clamps it below 1, so the last action, at probability exactly 0, is
    never drawn: the draw is the last action with a non-zero probability, as in fp64."""
    from marl_uavs_targets_tracking_b200.rollout import fused_policy_sample
    net = make_net(64, A, seed=A)
    with torch.no_grad():
        net.fc2.weight.zero_()
        net.fc2.bias.zero_()
        net.fc2.bias[A - 1] = -200.0
    x = make_inputs("randn", 1, seed=A)
    p64, bound = reference(net, x)
    for c in CLAMP_COUNTERS:
        act, probs = fused_policy_sample(net, x, 99, c, want_probs=True)
        assert float(probs[0, A - 1]) == 0.0 and int(act[0]) == A - 2, (c, int(act[0]))
        assert check_draw(act, probs, p64, bound, uniforms(1, 99, c), "A%d counter %d" % (A, c)) == 0


@pytest.mark.gpu
def test_a_tiny_uniform_draws_a_rare_first_action():
    """u53 = 1.66e-8 below p0 ~ 1e-6: action 0."""
    from marl_uavs_targets_tracking_b200.rollout import fused_policy_sample
    net = make_net(64, 5, seed=1)
    with torch.no_grad():
        net.fc2.weight.zero_()
        net.fc2.bias.zero_()
        net.fc2.bias[0] = -12.5  # p0 = e^-12.5 / (e^-12.5 + 4) = 9.3e-7
    x = make_inputs("randn", 1, seed=1)
    act, probs = fused_policy_sample(net, x, 99, TINY_U_COUNTER, want_probs=True)
    p64, bound = reference(net, x)
    assert 5e-7 < float(p64[0, 0]) < 2e-6
    assert int(act[0]) == 0
    assert check_draw(act, probs, p64, bound, uniforms(1, 99, TINY_U_COUNTER), "tiny u") == 0


# ------------------------------------------------------------------------------------------------ GPU: the PDL kernel
@pytest.mark.gpu
@pytest.mark.parametrize("n,E,H,na,first_counter", [
    (10, 1000, 128, 12, (1 << 32) - 3),   # the step counter crosses into the high word
    (64, 64, 128, 12, MASK64 - 2),        # ... and wraps to 0, 1, 2 (64x64 on the default step path)
    (10, 37, 1, 2, MASK64 - 2),
    (10, 37, 385, 13, (1 << 32) - 3),
    (10, 37, 512, 16, 7),
], ids=["10x10-E1000", "64x64-E64", "H1-na2", "H385-na13", "H512-na16"])
def test_run_policy_draws_match_the_plain_kernel_and_fp64(n, E, H, na, first_counter):
    """uavsim_run_policy (the PDL instance) over T = 6 steps with obs and action trajectories: the actions of slot k are
    bit-equal to uavsim_policy_sample on obs slot k with counter first_counter + k, and consistent with fp64 + Philox."""
    from marl_uavs_targets_tracking_b200 import BatchedEnvironment, default_config
    from marl_uavs_targets_tracking_b200.rollout import fused_policy_sample
    T, seed = 6, SEED_HI
    cfg = default_config("MAAC-G", n, n)
    env = BatchedEnvironment(n, n, 2000, 2000, na, n_envs=E, device=DEV, seed=5)
    env.reset(cfg)
    net = make_net(H, na, seed=H + na)
    obs = torch.full((T + 1, E, n, 12), float("nan"), device=DEV)
    acts = torch.full((T, E, n), -7, dtype=torch.int32, device=DEV)
    env.run_policy(cfg, None, net, seed, first_counter, T, obs=obs, actions=acts)
    for k in range(T):
        ck = (first_counter + k) & MASK64
        x = obs[k].view(E * n, 12)
        plain, probs = fused_policy_sample(net, x, seed, ck, want_probs=True)
        assert torch.equal(acts[k].view(-1), plain), k
        p64, bound = reference(net, x)
        check_probs(probs, p64, bound, "step %d" % k)
        check_draw(acts[k].view(-1), probs, p64, bound, uniforms(E * n, seed, ck), "step %d" % k)
    env.close()


# ------------------------------------------------------------------------------------------------ host-side fixes
@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [torch.float64, torch.float16], ids=["double", "half"])
def test_weights_of_another_dtype_are_converted(dtype):
    """A .double() or .half() PolicyNet draws exactly what the same net cast to float32 draws, in fused_policy_sample and
    in run_policy (the kernel reads float32)."""
    import copy
    from marl_uavs_targets_tracking_b200 import BatchedEnvironment, default_config
    from marl_uavs_targets_tracking_b200.rollout import fused_policy_sample
    net = make_net(128, 12, "fc2x8", seed=2).to(dtype)
    net32 = copy.deepcopy(net).float()
    x = make_inputs("obs", 4099, seed=2)
    a, p = fused_policy_sample(net, x, 99, 5, want_probs=True)
    a32, p32 = fused_policy_sample(net32, x, 99, 5, want_probs=True)
    assert torch.equal(a, a32) and torch.equal(p, p32)
    cfg = default_config("MAAC-G", 10, 10)
    trajs = []
    for m in (net, net32):
        env = BatchedEnvironment(10, 10, 2000, 2000, 12, n_envs=64, device=DEV, seed=5)
        env.reset(cfg)
        obs = torch.empty((6, 64, 10, 12), device=DEV)
        acts = torch.empty((5, 64, 10), dtype=torch.int32, device=DEV)
        env.run_policy(cfg, None, m, 3, 1, 5, obs=obs, actions=acts)
        trajs.append((obs, acts))
        env.close()
    assert torch.equal(trajs[0][0], trajs[1][0]) and torch.equal(trajs[0][1], trajs[1][1])


@pytest.mark.gpu
def test_sizes_beyond_the_kernel_take_the_stock_path():
    """hidden_dim = 640 (above the kernel's 512) or a single action: the agent does not use the fused kernel, and an
    episode runs on the stock torch path."""
    from marl_uavs_targets_tracking_b200 import BatchedEnvironment, default_config
    from marl_uavs_targets_tracking_b200.rollout import BatchedActorCritic, operate_epoch_batched
    dev = torch.device(DEV)
    agent = BatchedActorCritic(12, 640, 12, 1e-3, 1e-3, 0.95, dev)
    assert agent.fused is False
    assert BatchedActorCritic(12, 64, 1, 1e-3, 1e-3, 0.95, dev).fused is False
    assert BatchedActorCritic(12, 512, 16, 1e-3, 1e-3, 0.95, dev).fused is True
    cfg = default_config("MAAC-G", 10, 10)
    env = BatchedEnvironment(10, 10, 2000, 2000, 12, n_envs=16, device=DEV, seed=1)
    env.reset(cfg)
    tr, summary = operate_epoch_batched(cfg, env, agent, None, 4)
    assert tr["actions"].shape == (4 * 16 * 10,) and 0 <= int(tr["actions"].min()) and int(tr["actions"].max()) < 12
    assert 0 <= summary["average_covered_targets"] <= 10
    env.close()


@pytest.mark.gpu
def test_a_misaligned_observation_view_is_copied():
    """A contiguous float32 view 4 bytes off a 16-byte boundary draws what its aligned copy draws."""
    from marl_uavs_targets_tracking_b200.rollout import fused_policy_sample
    B = 1001
    buf = torch.empty(12 * B + 1, device=DEV)
    xv = buf[1:].view(B, 12)
    xv.copy_(make_inputs("obs", B, seed=4))
    assert xv.storage_offset() == 1 and xv.data_ptr() % 16 != 0
    net = make_net(128, 12, seed=4)
    a, p = fused_policy_sample(net, xv, 99, 5, want_probs=True)
    a0, p0 = fused_policy_sample(net, xv.clone(), 99, 5, want_probs=True)
    assert torch.equal(a, a0) and torch.equal(p, p0)
