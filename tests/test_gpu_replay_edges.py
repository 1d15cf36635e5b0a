"""Device prioritized replay (csrc/replay.cuh) against a float64 reference at its edges.

The reference restates what `PrioritizedReplayBuffer.sample` must compute -- p = q / sum(q), q = priority^alpha, the
inverse CDF of p and the weights (n p)^-beta / max -- in float64, and accepts the device's results within bounds derived
from the kernels' arithmetic (DESIGN.md section 3.3), not tuned constants:

* probabilities: powf's error, the float32 rounding of the fp64 total and the float32 division;
* indices: every draw.  With S the prefix sums of the device's own p (computed exactly on the host), index i is accepted
  for uniform u only when S[i-1]/S[-1] - delta <= u < S[i]/S[-1] + delta and p[i] > 0, where delta bounds the fp64
  rounding of the scan's longest addition chain.  Nothing here depends on the order in which the device sums.
* weights: (n p[idx])^-beta / max in fp64 within powf's error and the float32 roundings around it.

The cases are the sizes around the scan's 8-slot thread chunks, 2048-slot blocks and the 303 104-thread grid of the
grid-stride kernels, buffers that are not full, alpha in {0, 1e-3, 0.6, 1}, priorities from the smallest subnormal to
1e30, zero runs placed on chunk / warp / block boundaries, uniforms exactly on exact CDF boundaries, the windows in which
the earlier scan let a zero-probability slot be drawn, 64-bit Philox counters and seeds, and a -0.0 priority.
"""
import math

import numpy as np
import pytest
import torch

from philox_ref import philox4x32_10, u53

DEV = "cuda:0"
U = 2.0 ** -53                        # unit roundoff of float64
SCAN_ELEMS, SCAN_NT, SCAN_PER = 2048, 256, 8   # replay_scan_kernel: slots per block, threads, slots per thread
GRID_THREADS = 148 * 8 * 256          # replay_grid's cap: every grid-stride kernel makes a second pass beyond this
# powf's maximum error: 4 ulp over the full range (CUDA C++ Programming Guide, "Mathematical Functions" appendix,
# single-precision table).  Quoted, not measured here.
POWF_ULP = 4


def _buffer(capacity, alpha, **kw):
    from marl_uavs_targets_tracking_b200 import PrioritizedReplayBuffer
    return PrioritizedReplayBuffer(capacity, alpha=alpha, state_dim=1, device=DEV, **kw)


# ---- host helpers (no device) ------------------------------------------------------------------------------------
def wide_priorities(rng, n):
    """float32 priorities log-uniform from the smallest subnormal (2^-149) to 1e30, both ends included."""
    pri = (10.0 ** rng.uniform(-44.8, 30.0, n)).astype(np.float32)
    pri[rng.randint(0, n, max(1, n // 1000))] = np.float32(2.0 ** -149)
    pri[rng.randint(0, n, max(1, n // 1000))] = np.float32(1e30)
    return np.maximum(pri, np.float32(2.0 ** -149))


def kraft_depths(rng, m, max_depth=50):
    """Depths of the leaves of a random full binary tree with m leaves, none deeper than max_depth: sum 2^-d == 1."""
    d = np.zeros(1, np.int64)
    while d.size < m:
        ok = np.flatnonzero(d < max_depth)
        pick = rng.choice(ok, min(m - d.size, max(1, d.size // 2), ok.size), replace=False)
        d = np.concatenate([np.delete(d, pick), d[pick] + 1, d[pick] + 1])
    return rng.permutation(d)


def exact_prefix(p):
    """float64 of the EXACT prefix sums of the float32 array p >= 0 (relative error <= 4 U each).

    Every float32 in [0, 1] is an integer multiple of 2^-149 below 2^151: the integers are summed in 32-bit limbs held in
    int64 (5 M terms of < 2^32 stay below 2^55), carried, and converted from the top limb down."""
    bits = np.ascontiguousarray(p, np.float32).view(np.uint32).astype(np.int64)
    assert (bits >> 31 == 0).all() and ((bits >> 23) <= 127).all(), "p must lie in [0, 1]"
    e, m = bits >> 23, bits & 0x7FFFFF
    m = np.where(e > 0, m | 0x800000, m)
    sh = np.maximum(e - 1, 0)                      # p * 2^149 = m << sh
    k, val = sh // 32, m << (sh % 32)              # val < 2^55 spans limbs k and k + 1 <= 4
    limbs = np.zeros((p.size, 5), np.int64)
    rows = np.arange(p.size)
    limbs[rows, k] = val & 0xFFFFFFFF
    limbs[rows, k + 1] += val >> 32
    c = np.cumsum(limbs, axis=0)
    for j in range(4):
        c[:, j + 1] += c[:, j] >> 32
        c[:, j] &= 0xFFFFFFFF
    s = np.zeros(p.size)
    for j in range(4, -1, -1):
        s = s + c[:, j].astype(np.float64) * 2.0 ** (32 * j - 149)
    return s


def scan_chain(n):
    """Longest chain of fp64 roundings behind one CDF value of replay_scan_kernel, for n slots.
    Block sum S_b (replay_norm_kernel): 7 adds per thread + 5 butterfly + 7 over warps = 19; block offsets B_b: one add per
    earlier block (replay_scan_blocks_kernel); in-block x: 7 per thread + 5 warp scan + 7 over warps + (inc - run) + the
    slot's own running sum = 21; the final add B_b + x: 1."""
    return 19 + (n + SCAN_ELEMS - 1) // SCAN_ELEMS + 21 + 1


def draw_delta(n):
    """|cdf_i / cdf_last - S_i / S_last| bound: every device CDF value is within gamma_K * total of the exact prefix sum
    (sums of non-negative terms: each rounding errs by at most U times a partial sum <= total), so the normalised value
    is within 2 gamma_K / (1 - gamma_K) plus the device division (U); the host's S_i / S_last adds 4 U + 4 U + U."""
    K = scan_chain(n)
    g = K * U / (1 - K * U)
    return 2 * g / (1 - g) + U + 9 * U


def parent_zero_windows(p):
    """Chooses inputs only.  Emulates the float64 operation order of the scan this file's zero-window test was written
    against (replay_norm_kernel's block sums, the serial block offsets, and a CDF written as
    fl(fl(B_b + warp totals + (inc - run)) + v_k)) and the draw kernel's binary search; returns uniforms u (and the slots
    that search returned) for which it lands on a slot with p == 0."""
    n = p.size
    nb = (n + SCAN_ELEMS - 1) // SCAN_ELEMS
    x = np.zeros(nb * SCAN_ELEMS)
    x[:n] = p.astype(np.float64)
    # replay_norm_kernel: thread t sums slots t, t + 256, ... in order; xor butterfly; warp totals in order
    acc = np.zeros((nb, SCAN_NT))
    for j in range(SCAN_PER):
        acc = acc + x.reshape(nb, SCAN_PER, SCAN_NT)[:, j, :]
    a = acc.reshape(nb, 8, 32)
    for o in (16, 8, 4, 2, 1):
        a = a + a[:, :, np.arange(32) ^ o]
    S = np.zeros(nb)
    for w in range(8):
        S = S + a[:, w, 0]
    B = np.zeros(nb + 1)
    for b in range(nb):
        B[b + 1] = B[b] + S[b]
    # replay_scan_kernel as it was: 8 contiguous slots per thread
    xs = x.reshape(nb, SCAN_NT, SCAN_PER)
    v = np.zeros_like(xs)
    run = np.zeros((nb, SCAN_NT))
    for k in range(SCAN_PER):
        run = run + xs[:, :, k]
        v[:, :, k] = run
    inc = run.reshape(nb, 8, 32).copy()
    lane = np.arange(32)
    for o in (1, 2, 4, 8, 16):
        up = np.concatenate([np.zeros((nb, 8, o)), inc[:, :, :32 - o]], axis=2)
        inc = np.where(lane >= o, inc + up, inc)
    offw = np.repeat(B[:nb, None], 8, axis=1)
    for w in range(1, 8):                            # off = B_b; off += warp_tot[w'] for w' < wid, in order
        acc_w = B[:nb].copy()
        for ww in range(w):
            acc_w = acc_w + inc[:, ww, 31]
        offw[:, w] = acc_w
    off = offw[:, :, None] + (inc - run.reshape(nb, 8, 32))
    cdf = (off.reshape(nb, SCAN_NT, 1) + v).reshape(-1)[:n]
    last = cdf[n - 1]
    # candidate windows: a zero slot whose value rises above its predecessor's
    zero = np.flatnonzero(p == 0)
    zero = zero[zero > 0]
    cand = zero[cdf[zero] > cdf[zero - 1]]
    u = cdf[cand - 1] / last
    lo, hi = np.zeros(u.size, np.int64), np.full(u.size, n, np.int64)
    while (lo < hi).any():                           # replay_draw_kernel's search on that CDF
        act = lo < hi
        mid = (lo + hi) >> 1
        le = cdf[np.minimum(mid, n - 1)] / last <= u
        lo = np.where(act & le, mid + 1, lo)
        hi = np.where(act & ~le, mid, hi)
    idx = np.minimum(lo, n - 1)
    hit = p[idx] == 0
    return u[hit], idx[hit]


# ---- checks against the float64 reference --------------------------------------------------------------------------
def check_probabilities(p_dev, pri, alpha):
    """p_dev (float32, device) against p64 = q64 / fsum(q64), q64 = pri^alpha in float64.

    q_dev = powf(pri, alpha) errs by at most POWF_ULP ulp: eq = POWF_ULP * max(2^-23 q, 2^-149).  The device total,
    fp64 over q_dev then rounded to float32, lies within T (1 +- relT), relT = sum(eq) / T + gamma_K + 2^-24 (+ 2^-150 / T
    for a subnormal total).  p_dev = fl32(q_dev / total) adds one float32 rounding: relative 2^-24 or absolute 2^-150.
    alpha is the float32 the buffer stores, as numpy uses for a float32 array ** alpha (float32(0.6) - 0.6 = 2.4e-8
    moves 1e-30^alpha by 1.6e-6)."""
    n = pri.size
    q64 = pri.astype(np.float64) ** float(np.float32(alpha))
    T = math.fsum(q64)
    p64 = q64 / T
    eq = POWF_ULP * np.maximum(2.0 ** -23 * q64, 2.0 ** -149)
    K = scan_chain(n) - 22                           # the pow kernel's chain: block sums + serial total
    relT = math.fsum(eq) / T + K * U / (1 - K * U) + 2.0 ** -24 + 2.0 ** -150 / T
    hi = (q64 + eq) / (T * (1 - relT))
    lo = np.maximum(q64 - eq, 0) / (T * (1 + relT))
    hi = hi * (1 + 2.0 ** -24) + 2.0 ** -150
    lo = lo * (1 - 2.0 ** -24) - 2.0 ** -150
    pd = p_dev.astype(np.float64)
    bad = np.flatnonzero((pd < lo) | (pd > hi))
    assert bad.size == 0, ("probability outside the bound", bad[:5], pd[bad[:5]], p64[bad[:5]])
    if alpha > 0:
        assert (p_dev[pri == 0] == 0).all()          # powf(0, alpha > 0) == +0 exactly
    else:
        assert (p_dev[pri == 0] > 0).all()           # powf(0, 0) == 0 ** 0 == 1
    return p64


def check_draws(p_dev, u, idx, S=None):
    """Every drawn index against the exact prefix sums S of the device's own p (no tolerated misses)."""
    n = p_dev.size
    S = exact_prefix(p_dev) if S is None else S
    d = draw_delta(n)
    lo = np.where(idx > 0, S[np.maximum(idx - 1, 0)], 0.0) / S[-1] - d
    hi = S[idx] / S[-1] + d
    assert ((idx >= 0) & (idx < n)).all()
    bad = np.flatnonzero(~((lo <= u) & (u < hi)))
    assert bad.size == 0, ("draw outside its CDF interval", bad[:5], u[bad[:5]], idx[bad[:5]])
    zero = np.flatnonzero(p_dev[idx] == 0)
    assert zero.size == 0, ("drew a slot of probability 0", u[zero[:5]], idx[zero[:5]])


def check_weights(p_dev, idx, w, beta):
    """w = (n p[idx])^-beta / max in float64.  Device: a = fl32(n p) (2^-24, or exact when subnormal: n p is then an
    integer multiple of 2^-149), powf(a, -beta) (beta 2^-23 from a, POWF_ULP ulp), the same for the maximum, one float32
    division (2^-24)."""
    n = p_dev.size
    if beta == 0:
        assert (w == 1.0).all()                       # powf(x, -0) == 1: every weight exactly 1
        return
    raw = (n * p_dev[idx].astype(np.float64)) ** -beta
    ref = raw / raw.max()
    e = beta * 2.0 ** -23 + POWF_ULP * 2.0 ** -23
    rel = (1 + e) / (1 - e) * (1 + 2.0 ** -24) - 1
    err = np.abs(w.astype(np.float64) - ref)
    assert (err <= rel * ref).all(), ("weight outside the bound", float((err / ref).max()), rel)


def fill(C, n, pri, alpha, **kw):
    """A buffer of capacity C holding n transitions (action k in slot k) with priorities pri (one update of n indices)."""
    buf = _buffer(C, alpha, **kw)
    k = torch.arange(n, device=DEV)
    buf.add({"states": k.float()[:, None], "actions": k.int(), "rewards": torch.zeros(n, device=DEV),
             "next_states": k.float()[:, None]})
    buf.update_priorities(k, torch.as_tensor(pri, device=DEV))
    return buf


def draw(buf, u, beta=0.4):
    """Sample with caller uniforms; more uniforms than buf.size() are drawn in several calls."""
    n, out = buf.size(), []
    for s in range(0, u.size, n):
        smp, idx, w = buf.sample(min(n, u.size - s), beta, uniforms=torch.as_tensor(u[s:s + n], device=DEV))
        assert torch.equal(smp["actions"].long(), idx)                       # the gathered row is the drawn slot's
        out.append((idx.cpu().numpy(), w.cpu().numpy()))
    return np.concatenate([o[0] for o in out]), [o[1] for o in out]


def sample_and_check(buf, pri, alpha, beta, u):
    idx, ws = draw(buf, u, beta)
    p_dev = buf.export()["probabilities"].numpy()
    check_probabilities(p_dev, pri, alpha)
    S = exact_prefix(p_dev)
    check_draws(p_dev, u, idx, S)
    s = 0
    for w in ws:
        check_weights(p_dev, idx[s:s + w.size], w, beta)
        s += w.size
    return p_dev, S, idx


def boundary_uniforms(S):
    """u = S_i / S_last for every slot i and the next double below: the edges of every slot's interval (u < 1)."""
    b = S[:-1] / S[-1]
    b = b[b < 1]
    return np.concatenate([b, np.nextafter(b, 0), [0.0, 1 - U]])


# ---- CPU tests of the helpers ---------------------------------------------------------------------------------------
def test_exact_prefix_and_kraft_depths_without_a_device():
    from fractions import Fraction
    rng = np.random.RandomState(0)
    p = np.concatenate([[2.0 ** -149, 0, 1.0, 2.0 ** -126, np.nextafter(np.float32(2.0 ** -126), 0)],
                        10.0 ** rng.uniform(-40, 0, 300)]).astype(np.float32)
    ex = np.cumsum([Fraction(float(x)) for x in p])
    S = exact_prefix(p)
    assert all(abs(Fraction(float(s)) - e) <= 4 * U * e for s, e in zip(S, ex))
    for m in (1, 2, 7, 2049):
        d = kraft_depths(rng, m)
        assert d.size == m and d.max() <= 50 and sum(Fraction(1, 2 ** int(x)) for x in d) == 1


def test_parent_scan_emulation_finds_zero_windows_without_a_device():
    """The inputs of test_zero_slot_windows_are_never_drawn, with a float32 model of the device's p: the emulation of
    the earlier scan finds zero slots with a drawable interval."""
    rng = np.random.RandomState(11)
    pri = wide_priorities(rng, 4 * SCAN_ELEMS + 5)
    pri[::SCAN_PER] = 0
    q = (pri.astype(np.float64) ** 0.6).astype(np.float32)
    p = (q / np.float32(q.astype(np.float64).sum())).astype(np.float32)
    u, slots = parent_zero_windows(p)
    assert u.size > 20 and (p[slots] == 0).all()


# ---- device ---------------------------------------------------------------------------------------------------------
SIZES = (1, 2, 7, 2047, 2048, 2049, 4097, GRID_THREADS - 1, GRID_THREADS, GRID_THREADS + 1, 1 << 20, 5_000_001)
ALPHAS = (0.0, 1e-3, 0.6, 1.0)
CASES = [(n, a) for n in SIZES for a in ALPHAS if n <= 4097 or a in (0.6, 1.0)]


@pytest.mark.gpu
@pytest.mark.parametrize("n,alpha", CASES)
def test_sample_against_fp64_reference(n, alpha):
    """Full buffers of every size, wide-range priorities with some zeros: probabilities, every draw, weights."""
    rng = np.random.RandomState(n % 100_003 + int(alpha * 1000))
    pri = wide_priorities(rng, n)
    if n > 2:
        pri[rng.randint(0, n, max(1, n // 50))] = 0
        pri[rng.randint(0, n)] = 1.0
    if alpha == 1.0:                                # the float32 total must stay finite
        assert math.fsum(pri.astype(np.float64)) < 3e38
    buf = fill(n, n, pri, alpha)
    u = rng.random_sample(min(n, 1_000_003))
    p_dev, S, _ = sample_and_check(buf, pri, alpha, 0.4, u)
    if n <= 4097:                                   # and every slot's interval edges
        idx, _ = draw(buf, boundary_uniforms(S), 0.4)
        check_draws(p_dev, boundary_uniforms(S), idx, S)


@pytest.mark.gpu
@pytest.mark.parametrize("C,n,alpha", [(8, 3, 0.6), (2049, 2048, 1.0), (5000, 4097, 1e-3), (GRID_THREADS + 7, 2049, 0.6),
                                       (1 << 20, GRID_THREADS + 1, 1.0)])
def test_partly_filled_buffer_and_updates_beyond_size(C, n, alpha):
    """Priorities written by update_priorities at or beyond size count in the next add's maximum, as in the reference;
    sampling reads slots [0, size) only."""
    rng = np.random.RandomState(C + n)
    pri = wide_priorities(rng, n)
    buf = fill(C, n, pri, alpha)
    ref = np.zeros(C, np.float32)
    ref[:n] = pri
    assert np.array_equal(buf.export()["priorities"].numpy(), ref)
    beyond = np.unique(np.concatenate([[n, C - 1], rng.randint(n, C, 5)]))
    vals = np.float32(2e30) * (1 + np.arange(beyond.size, dtype=np.float32)) / beyond.size
    buf.update_priorities(torch.as_tensor(beyond, device=DEV), torch.as_tensor(vals, device=DEV))
    ref[beyond] = vals
    k = min(2, C - n)
    t = torch.arange(n, n + k, device=DEV)
    buf.add({"states": t.float()[:, None], "actions": t.int(), "rewards": torch.zeros(k, device=DEV),
             "next_states": t.float()[:, None]})
    ref[n:n + k] = ref.max()                        # numpy: priorities.max() over the whole array
    assert np.array_equal(buf.export()["priorities"].numpy(), ref)
    assert buf.size() == n + k
    sample_and_check(buf, ref[:n + k], alpha, 0.7, rng.random_sample(min(n + k, 100_000)))


@pytest.mark.gpu
@pytest.mark.parametrize("n", (1, 2, 7, 2047, 2049, 4097, GRID_THREADS + 1, 1 << 20))
def test_exact_cdf_boundaries(n):
    """alpha = 1 and power-of-two priorities summing to 1 (a random full binary tree's leaf weights, depth <= 50), with
    zero slots between them: every prefix sum is exact in any order.  u on a boundary gives the next slot with p > 0
    (side='right'), the double below gives this slot; u = 0 and u = 1 - 2^-53 give the first and last slot with p > 0."""
    rng = np.random.RandomState(n)
    m = max(1, n - n // 5)
    pri = np.zeros(n, np.float32)
    slots = np.sort(rng.choice(n, m, replace=False))
    pri[slots] = 2.0 ** -kraft_depths(rng, m).astype(np.float64)
    buf = fill(n, n, pri, 1.0)
    draw(buf, np.zeros(1), 0.0)
    p_dev = buf.export()["probabilities"].numpy()
    assert np.array_equal(p_dev, pri)               # powf(2^-d, 1) is exact and the total is exactly 1
    S = np.cumsum(pri.astype(np.float64))           # exact: dyadic values of <= 50 bits
    assert S[-1] == 1.0
    b = S[slots[:-1]]
    u = np.concatenate([b, np.nextafter(b, 0), [0.0, 1 - U]])
    idx, w = draw(buf, u, 0.0)
    assert np.array_equal(idx, np.searchsorted(S, u, side="right"))
    assert np.array_equal(idx[:b.size], slots[1:]) and np.array_equal(idx[b.size:2 * b.size], slots[:-1])
    assert idx[-2] == slots[0] and idx[-1] == slots[-1]
    assert all((x == 1.0).all() for x in w)


ZERO_RUNS = {
    "start": [(0, 9)], "start_block": [(0, SCAN_ELEMS + 8)],
    "chunk": [(8, 16), (21, 43)], "warp": [(256, 512), (250, 270), (1023, 1025)],
    "block": [(SCAN_ELEMS, 2 * SCAN_ELEMS), (2 * SCAN_ELEMS + 2040, 2 * SCAN_ELEMS + 2056)],
    "span_blocks": [(SCAN_ELEMS - 3, 2 * SCAN_ELEMS + 2049)], "end": [(-3000, None)], "end_chunk": [(-8, None)],
    "single": [(0, 2049), (2050, None)],
}


@pytest.mark.gpu
@pytest.mark.parametrize("alpha", (1e-3, 0.6, 1.0))
@pytest.mark.parametrize("layout", sorted(ZERO_RUNS))
def test_zero_runs(layout, alpha):
    """Runs of zero priorities at the start, in the middle and at the end, on or across chunk (8), warp (256) and block
    (2048) boundaries, and a single positive slot among zeros: never drawn, even by uniforms on every interval edge."""
    n = 3 * SCAN_ELEMS + 123
    rng = np.random.RandomState(len(layout) + int(alpha * 10))
    pri = wide_priorities(rng, n)
    for a, b in ZERO_RUNS[layout]:
        pri[a:b] = 0
    buf = fill(n, n, pri, alpha)
    p_dev, S, _ = sample_and_check(buf, pri, alpha, 0.4, rng.random_sample(n))
    u = boundary_uniforms(S)
    idx, _ = draw(buf, u)
    check_draws(p_dev, u, idx, S)
    if layout == "single":
        assert (idx == 2049).all()


@pytest.mark.gpu
@pytest.mark.parametrize("alpha", (0.6, 1.0))
def test_zero_slot_windows_are_never_drawn(alpha):
    """Wide-range priorities with a zero at every chunk start (so at every warp and block start too), and uniforms on
    the windows in which an emulation of the earlier scan's summation order draws a zero slot."""
    n = 4 * SCAN_ELEMS + 5
    rng = np.random.RandomState(11)
    pri = wide_priorities(rng, n)
    pri[::SCAN_PER] = 0
    buf = fill(n, n, pri, alpha)
    draw(buf, np.zeros(1))
    p_dev = buf.export()["probabilities"].numpy()
    u, _ = parent_zero_windows(p_dev)
    assert u.size > 0, "no window to test"
    idx, _ = draw(buf, u)
    check_draws(p_dev, u, idx)


@pytest.mark.gpu
def test_grid_stride_draws_and_updates():
    """Batches of GRID_THREADS + 1 and 1 000 003 draws; an update of more than GRID_THREADS indices whose positions k and
    k + GRID_THREADS repeat an index (the later one must win); the maximum in the last slot of a capacity above
    GRID_THREADS."""
    n = 1 << 20
    rng = np.random.RandomState(3)
    pri = wide_priorities(rng, n)
    buf = fill(n, n, pri, 0.6)
    sample_and_check(buf, pri, 0.6, 0.4, rng.random_sample(GRID_THREADS + 1))
    sample_and_check(buf, pri, 0.6, 0.4, rng.random_sample(1_000_003))
    cnt = GRID_THREADS + 5000
    idx = rng.randint(0, n, cnt)
    idx[GRID_THREADS:] = idx[:5000]
    vals = rng.uniform(0.5, 2.0, cnt).astype(np.float32)
    buf.update_priorities(torch.as_tensor(idx, device=DEV), torch.as_tensor(vals, device=DEV))
    ref = pri.copy()
    rev = idx[::-1]
    uniq, first = np.unique(rev, return_index=True)
    ref[uniq] = vals[cnt - 1 - first]               # sequential assignment: the last write to an index wins
    assert np.array_equal(buf.export()["priorities"].numpy(), ref)
    assert not np.array_equal(ref[idx[:5000]], vals[:5000])
    for C in (GRID_THREADS + 1, 1_000_003):
        b = fill(C, C - 1, np.ones(C - 1, np.float32), 0.6)
        b.update_priorities(torch.tensor([C - 1], device=DEV), torch.tensor([3.5], device=DEV))
        b.add({"states": torch.zeros(2, 1, device=DEV), "actions": torch.zeros(2, dtype=torch.int32, device=DEV),
               "rewards": torch.zeros(2, device=DEV), "next_states": torch.zeros(2, 1, device=DEV)})
        pr = b.export()["priorities"].numpy()
        assert pr[C - 1] == 3.5 and pr[0] == 3.5 and b.size() == C  # slots C - 1 and, wrapping, 0


@pytest.mark.gpu
@pytest.mark.parametrize("counter,seed", [(2 ** 32 - 1, 77), (2 ** 32, 77), (2 ** 64 - 1, 77),
                                          (5, 0x9E3779B97F4A7C15), (2 ** 64 - 1, 0xFFFFFFFF00000001)])
def test_philox_uniforms(counter, seed):
    """Equal priorities on 2^20 slots make the CDF exactly k 2^-20, so the drawn index is floor(u 2^20): the device's
    uniforms must be philox_ref's for (draw index; counter) under the 64-bit seed, over 1 000 003 draws."""
    n, batch = 1 << 20, 1_000_003
    buf = fill(n, n, np.ones(n, np.float32), 0.6, seed=seed)
    assert buf.seed == seed
    buf._draws = counter
    _, idx, w = buf.sample(batch, 0.4)
    k = np.arange(batch, dtype=np.uint64)
    x = philox4x32_10(k, k >> np.uint64(32), counter & 0xFFFFFFFF, counter >> 32, seed)
    u = u53(x[0], x[1])
    assert np.array_equal(idx.cpu().numpy(), np.floor(u * n).astype(np.int64))
    assert (w == 1).all()
    _, idx2, _ = buf.sample(batch, 0.4, uniforms=torch.as_tensor(u, device=DEV))
    assert torch.equal(idx, idx2)


@pytest.mark.gpu
@pytest.mark.parametrize("C,slots,vals", [
    (8, [0, 1, 2, 3], [0.5, -0.0, 2.0, 0.25]),        # -0.0 among positive priorities
    (8, [0, 1, 2, 3], [-0.0, -0.0, 0.0, -0.0]),        # all zero, signs mixed: the maximum is a zero
    (8, [1, 6], [-0.0, 0.75]),                          # the maximum beyond size
    (GRID_THREADS + 1, [GRID_THREADS, 5], [-0.0, 1.5]),  # -0.0 in the last slot, on the grid's second pass
])
def test_negative_zero_priority_then_add(C, slots, vals):
    """update_priorities(i, -0.0) then add: the stored priority is numpy's priorities.max()."""
    buf = fill(C, 4, np.ones(4, np.float32), 0.6)
    ref = np.zeros(C, np.float32)
    ref[:4] = 1
    v = np.array(vals, np.float32)
    buf.update_priorities(torch.tensor(slots, device=DEV), torch.as_tensor(v, device=DEV))
    ref[slots] = v
    buf.add({"states": torch.zeros(2, 1, device=DEV), "actions": torch.zeros(2, dtype=torch.int32, device=DEV),
             "rewards": torch.zeros(2, device=DEV), "next_states": torch.zeros(2, 1, device=DEV)})
    ref[4:6] = ref.max()
    got = buf.export()["priorities"].numpy()
    assert np.array_equal(got, ref) and got[4] == ref.max()
    if ref[:6].max() > 0:
        _, idx, w = buf.sample(6, 0.4, uniforms=torch.linspace(0, 1 - U, 6, dtype=torch.float64, device=DEV))
        assert (ref[idx.cpu().numpy()] > 0).all() and torch.isfinite(w).all()


@pytest.mark.gpu
@pytest.mark.parametrize("bad", (float("nan"), float("inf"), float("-inf"), -1e-30, -1.0))
def test_update_rejects_nan_infinite_and_negative_priorities(bad):
    """ValueError before anything is written; an index out of range is still an IndexError."""
    buf = fill(16, 16, np.arange(1, 17, dtype=np.float32), 0.6)
    before = buf.export()["priorities"].numpy()
    with pytest.raises(ValueError):
        buf.update_priorities(torch.tensor([0, 3, 5], device=DEV), torch.tensor([2.0, bad, 4.0], device=DEV))
    assert np.array_equal(buf.export()["priorities"].numpy(), before)
    with pytest.raises(IndexError):
        buf.update_priorities(torch.tensor([0, 16], device=DEV), torch.tensor([2.0, 3.0], device=DEV))
    buf.update_priorities(torch.tensor([0, 3], device=DEV), torch.tensor([-0.0, 0.0], device=DEV))   # zeros are fine
    assert np.array_equal(buf.export()["priorities"].numpy()[[0, 3]], [0, 0])
