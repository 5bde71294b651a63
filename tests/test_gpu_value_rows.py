"""K4 at every row count it accepts (n = Hmax + Smax from 1 to 64), against the fp64 restatement of the value network,
and K5's first-maximum rule on hand-built ties and NaN.  Needs a B200.

K4 picks its code from n: how the mean of H1 is reduced (n == 16, n | 32, segmented runs, one partial per warp for
n > 32), how softmax and pooling run (n == 16, several states per warp, whole warps per state through a scratch),
and how many states share a 128-row tile.  Every such path is pinned here with n in the test id, in every value
mode, with padding rows that hold garbage (the ABI excludes them from the mean and the softmax), the attention
weights, and bit-identity under permutation and for prefixes of the batch."""
import numpy as np
import pytest
import torch

import oracle_backend as ob
from ebc import synth
from ebc.actions import build_action_space
from ebc.config import SimConfig
from ebc.engine import BatchedSim
from test_gpu_parity import VALUE_TOL, assert_same_bits, np_, pair, random_batch, random_cfg
from test_gpu_value_tc import torch_value

pytestmark = pytest.mark.gpu

# value error bars relative to max(1, |ref|max), as in test_gpu_value_tc.test_tc_modes_vs_fp64, except tc_fp32: 3e-5
# instead of 2e-5.  Over ~10^4 states its maximum error is a rounding tail, not a structural error.  On a B200 the
# relative error of the 64 EB-CADRL row counts ranged from 0.7e-5 to 2.1e-5.  The largest was at n = 10, with 1.6e-5 at
# n = 9 and 0.8e-5 at n = 11, and at every n it stayed 2-9x the FFMA error on the same batch.  Wrong padding masks
# planted in the kernel gave errors of 2.6e-4 and more.
BARS = {"fp32": 1e-4, "tc_fp32": 3e-5, "tc_fp16x2": 4e-5, "tc_bf16": 0.1}
ACCURATE = ("fp32", "tc_fp32", "tc_fp16x2")
TC_MODES = ("tc_fp32", "tc_fp16x2", "tc_bf16")
ATTN_TOL = 2e-5                 # test_attention_weights.py
BOUNDARY_N = (1, 2, 3, 4, 5, 7, 8, 9, 15, 16, 17, 31, 32, 33, 48, 63, 64)
# partial first and last tiles at every states-per-tile count the launchers pick
PREFIXES = (1, 2, 3, 7, 8, 9, 15, 16, 17, 31, 32, 33, 129)
STATE_KEYS = ("hum_pv", "hum_gr", "hum_type", "hum_count", "stat", "stat_count", "rect", "rect_count", "rob_pv", "rob_gr",
              "rob_theta", "time")


def _sm_count():
    return torch.cuda.get_device_properties(0).multi_processor_count


def _batch_size():
    """The smallest prime above 2 * SMs * 32: every persistent CTA runs at least two tiles (the next tile's input is
    staged early) at every states-per-tile count up to 32, and the last tile is partial whenever a tile holds > 1 state."""
    k = 2 * _sm_count() * 32 + 1
    while any(k % p == 0 for p in range(2, int(k ** 0.5) + 1)):
        k += 1
    return k


def _random_local_net():
    """The dims of test_gpu_value_tc.test_tc_random_networks without the global state (no global K chunk, no G cap)."""
    rng = np.random.default_rng(7)
    dims = {"mlp1": [13, 168, 120], "mlp2": [120, 104, 52], "attention": [120, 88, 72, 1], "mlp3": [58, 180, 90, 70, 1]}
    w = {}
    for name, ds in dims.items():
        for i in range(len(ds) - 1):
            b = 1.0 / np.sqrt(ds[i])
            w["%s.%d.weight" % (name, 2 * i)] = rng.uniform(-b, b, (ds[i + 1], ds[i])).astype(np.float32)
            w["%s.%d.bias" % (name, 2 * i)] = rng.uniform(-b, b, ds[i + 1]).astype(np.float32)
    return w


NETS = {   # name -> (weights, typed input, with_global_state)
    "ebcadrl": (lambda: ob.load_weights("weights_ebcadrl.npz"), True, True),
    "sarl": (lambda: ob.load_weights("weights_sarl_baseline.npz"), False, True),
    "local": (_random_local_net, False, False),
}
SWEEP = [("ebcadrl", n) for n in range(1, 65)] + [(net, n) for net in ("sarl", "local") for n in BOUNDARY_N]


def _row_batch(n_states, n, D, seed):
    """Random rows, random row counts, and the counts that sit on a boundary forced at the start, middle and end of
    the batch: 1 and n, and for n > 32 also 31, 32 and 33 (the state's second warp empty, fully masked, or one real
    row).  Returns the zero-padded batch and the same batch with every padding row filled with garbage: normal(0, 4),
    and some rows at +-1e6 (beyond the fp16 range)."""
    rng = np.random.default_rng(seed)
    x = rng.normal(0, 1, (n_states, n, D)).astype(np.float32)
    cnt = rng.integers(1, n + 1, n_states).astype(np.int32)
    forced = [1, n] + ([31, 32, 33] if n > 32 else [])
    for j, c in enumerate(forced):
        cnt[[j, n_states // 2 + j, n_states - 1 - j]] = c
    pad = np.arange(n)[None, :] >= cnt[:, None]
    x[pad] = 0.0
    dirty = x.copy()
    dirty[pad] = rng.normal(0, 4, (int(pad.sum()), D)).astype(np.float32)
    partial = np.nonzero(cnt < n)[0]
    if len(partial):
        pick = rng.choice(partial, min(len(partial), 64), replace=False)
        dirty[pick, cnt[pick]] = np.where(rng.random((len(pick), D)) < 0.5, -1e6, 1e6).astype(np.float32)
    dev = lambda a: torch.as_tensor(a, device="cuda:0")  # noqa: E731
    return dev(x), dev(dirty), dev(cnt)


def _ragged_batch(N, H, S, R, seed):
    """random_batch with the extreme counts present: episode 0 has one human and no disc, episode 1 is full."""
    b = random_batch(N, H, S, R, seed)
    b["hum_count"][0], b["stat_count"][0] = 1, 0
    b["hum_count"][1], b["stat_count"][1] = H, S
    b["hum_type"][1] = np.sort(b["hum_type"][1])       # types stay sorted over the live humans
    return b


def _fp64_reference(w, x, cnt, with_global):
    """torch_value in chunks of <= 2^17 rows (the widest activation at n = 64 and 10^4 states is ~1.5 GB of doubles)."""
    step = max(1, (1 << 17) // x.shape[1])
    vs, ws = [], []
    for i in range(0, x.shape[0], step):
        v, a = torch_value(w, x[i:i + step], cnt[i:i + step], with_global, return_weights=True)
        vs.append(v)
        ws.append(a)
    return torch.cat(vs), torch.cat(ws)


def _same(a, b, cnt, what):
    """Bit-identity of two per-state tensors; on failure name the states and their row counts."""
    if torch.equal(a, b):
        return
    bad = (a != b).reshape(a.shape[0], -1).any(1).nonzero()[:, 0]
    raise AssertionError("%s: %d states differ, first %s with row counts %s" % (
        what, len(bad), bad[:8].tolist(), cnt[bad[:8]].tolist()))


@pytest.mark.parametrize("net,n", SWEEP, ids=["%s-n%d" % s for s in SWEEP])
def test_value_rows_vs_fp64(net, n):
    """Values and attention weights against fp64 at every row count; garbage in the padding rows changes no bit;
    a permuted batch gives the permuted values and every prefix the prefix, bit for bit; in every value mode."""
    make_w, typed, wg = NETS[net]
    w = make_w()
    cfg = SimConfig()
    cfg.with_agent_type = typed
    N = _batch_size()
    x, dirty, cnt = _row_batch(N, n, cfg.D, seed=1000 * n + len(net))
    ref, ref_w = _fp64_reference(w, x, cnt, wg)
    scale = max(1.0, ref.abs().max().item())
    real = torch.arange(n, device="cuda:0")[None, :] < cnt[:, None].long()
    perm = torch.as_tensor(np.random.default_rng(n).permutation(N), device="cuda:0")
    sim = BatchedSim(cfg, 1, n, 0, 0, 81, device="cuda:0")
    sim.set_weights(w, with_global_state=wg)
    att = sim.enable_attention(N)
    errs = {}
    for mode in ("fp32",) + TC_MODES:
        sim.set_value_mode(mode)
        v = sim.value(x, cnt).clone()
        a = att[:N].clone()
        err = (v.double() - ref).abs().max().item()
        a_err = (a.double() - ref_w)[real].abs().max().item()
        errs[mode] = (err, a_err)
        assert err < BARS[mode] * scale, (net, n, mode, err, scale)
        assert (a[~real] == 0).all(), (net, n, mode, "attention on a padding row")
        if mode in ACCURATE:
            assert a_err <= ATTN_TOL, (net, n, mode, a_err)
            s_err = (a.double().sum(1) - 1.0).abs().max().item()
            assert s_err <= 1e-5, (net, n, mode, s_err)
        vd = sim.value(dirty, cnt).clone()
        _same(vd, v, cnt, "%s n=%d %s: values with garbage padding" % (net, n, mode))
        _same(att[:N], a, cnt, "%s n=%d %s: attention with garbage padding" % (net, n, mode))
        vp = sim.value(x[perm], cnt[perm])
        _same(vp, v[perm], cnt[perm], "%s n=%d %s: permuted batch" % (net, n, mode))
        for k in PREFIXES:
            vk = sim.value(x[:k], cnt[:k])
            _same(vk, v[:k], cnt[:k], "%s n=%d %s: prefix of %d states" % (net, n, mode, k))
    print("value-rows %-8s n=%2d states=%d scale=%.3g  " % (net, n, N, scale)
          + "  ".join("%s |dV| %.2e |dw| %.2e" % (m, e, ae) for m, (e, ae) in errs.items()))


FUSED_SHAPES = [(1, 0), (2, 0), (2, 1), (3, 0), (4, 4), (7, 1), (9, 0), (12, 5), (20, 0), (25, 7), (31, 2), (32, 1), (33, 0),
                (40, 8), (50, 14), (64, 0)]


@pytest.mark.parametrize("H,S", FUSED_SHAPES, ids=["H%d-S%d" % s for s in FUSED_SHAPES])
def test_fused_input_across_shapes(H, S):
    """decide(fused=True) builds K4's rows from the bound state (human, static disc or padding, from the ragged counts)
    and must equal decide(fused=False) bit for bit: values, action values, argmax and attention weights, in every
    tensor-core mode.  Enough episodes that every CTA runs at least two entity tiles."""
    N = _batch_size() // 81 + 1
    cfg = random_cfg()
    sim = BatchedSim(cfg, N, H, S, 0, 81, device="cuda:0")
    sim.set_actions(build_action_space(0.8))
    sim.set_weights(ob.load_weights("weights_ebcadrl.npz"))
    sim.load_episodes(0, **_ragged_batch(N, H, S, 0, seed=H * 100 + S))
    att = sim.enable_attention()
    for mode in TC_MODES:
        sim.set_value_mode(mode)
        sim.decide(fused=False)
        want = {k: getattr(sim, k).clone() for k in ("values", "action_values", "argmax")}
        want["attention"] = att.clone()
        att.fill_(7.0)
        sim.decide(fused=True)
        torch.cuda.synchronize()
        for k, t in want.items():
            assert_same_bits(getattr(sim, k), t, "H=%d S=%d %s: fused %s" % (H, S, mode, k))


END_TO_END = [(1, 0, 0), (2, 0, 0), (2, 1, 0), (33, 0, 0), (40, 24, 3), (64, 0, 0), "ONE_STATIC"]


@pytest.mark.parametrize("shape", END_TO_END, ids=[s if isinstance(s, str) else "H%d-S%d-R%d" % s for s in END_TO_END])
def test_decide_and_step_vs_oracle_at_extremes(oracle, shape):
    """A whole decision and one committed step at the smallest and largest entity counts (and on the reference's
    one-static-human scenes from the device generator), against the oracle with test_full_size_other_configs' rule:
    ORCA and lookahead events exact, values within VALUE_TOL, argmax equal unless the oracle's two action values are
    closer than 2e-4, step events and human states exact, no NaN."""
    N = 256
    cfg = random_cfg()
    if shape == "ONE_STATIC":
        sh = synth.ONE_STATIC
        cfg.map_size_m, cfg.map_resolution = sh.map_size_m, sh.map_resolution
        g, r = pair(cfg, N, sh.H, sh.Smax, sh.Rmax, oracle, actions=build_action_space(sh.robot_v_pref),
                    weights=ob.load_weights("weights_ebcadrl.npz"))
        g.generate(sh, torch.arange(N, dtype=torch.int64, device="cuda:0"))
        torch.cuda.synchronize()
        for k in STATE_KEYS:
            getattr(r, k).copy_(getattr(g, k).cpu())
        assert g.n == 2 and (np_(g.hum_count) == 2).all()
    else:
        H, S, R = shape
        g, r = pair(cfg, N, H, S, R, oracle, actions=build_action_space(0.8), weights=ob.load_weights("weights_ebcadrl.npz"))
        batch = _ragged_batch(N, H, S, R, seed=7 * H + S)
        for s in (g, r):
            s.load_episodes(0, **batch)
    ga, ra = np_(g.decide().clone()), np_(r.decide().clone())
    torch.cuda.synchronize()
    assert_same_bits(g.hum_nv, r.hum_nv, "ORCA velocities")
    assert_same_bits(g.la_event, r.la_event, "lookahead events")
    dv = np.abs(np_(g.values) - np_(r.values)).max()
    assert dv < VALUE_TOL, dv
    av = np_(r.action_values)
    for i in np.nonzero(ga != ra)[0]:
        assert abs(av[i, ga[i]] - av[i, ra[i]]) < 2e-4, (i, ga[i], ra[i])
    assert (ga != ra).mean() <= 0.02
    assert (np_(g.nan_flag) == 0).all() and (np_(r.nan_flag) == 0).all()
    g.step(action_idx=g.argmax)
    r.step(action_idx=torch.as_tensor(ga.astype(np.int32)))
    torch.cuda.synchronize()
    assert_same_bits(g.event, r.event, "step events")
    assert_same_bits(g.hum_pv, r.hum_pv, "human states after the step")
    print("extremes", shape, "max |dV| %.2e" % dv, "argmax flips", int((ga != ra).sum()))


def _select_cases(A, rng):
    """Hand-built (reward, value, inside-goal) rows for K5 and the action each must select: -1 = none (nan_flag)."""
    cases = []

    def base():
        rew = np.round(rng.uniform(-1, 0, A), 3)
        val = np.round(rng.uniform(-1, 0, A), 3).astype(np.float32)
        return rew, val

    def tie(idx):                 # the same (reward, value) pair at every index (mod A): equal action values
        rew, val = base()
        idx = sorted(set(int(i) % A for i in idx))
        rew[idx], val[idx] = 0.5, 0.25
        cases.append((rew, val, False, idx[0]))

    tie([0])
    tie([A - 1])
    tie([5, 5 + 32, 5 + 64])                          # one lane's stride
    tie([3, 17, 30])                                  # different lanes, first pass
    tie([40, 7])                                      # lane 8 (second pass) and lane 7
    tie([33, 2])                                      # lane 1 holds the higher index: ties break by index, not lane
    tie([31, 32, 63, 64, 255])
    tie(list(rng.choice(A, min(A, 4), replace=False)))
    rew, val = np.zeros(A), np.zeros(A, np.float32)   # every action equal, signed zeros mixed in
    rew[1::2] = -0.0
    cases.append((rew, val, False, 0))
    rew, val = base()                                 # one NaN among finite values, at the would-be maximum
    k, k1 = A // 2, (A // 2 + 1) % A
    rew[k1], val[k1] = 0.75, 0.0
    rew[k], val[k] = 2.0, np.nan
    cases.append((rew, val, False, k1 if A > 1 else -1))
    rew, val = base()
    cases.append((rew, np.full(A, np.nan, np.float32), False, -1))
    cases.append((rew, np.full(A, -np.inf, np.float32), False, -1))
    rew, val = base()                                 # +inf wins, the first of two
    val[(A - 1) // 2] = val[A - 1] = np.inf
    cases.append((rew, val, False, (A - 1) // 2))
    rew, val = base()                                 # the robot is inside its goal radius: action 0
    rew[A - 1] = 1.0
    cases.append((rew, val, True, 0))
    return cases


@pytest.mark.parametrize("A", [1, 31, 32, 33, 81, 256])
def test_select_ties_and_nan(oracle, A):
    """K5 (a lane-strided scan, then a shuffle reduction that breaks ties by the lower index) against the oracle's
    sequential first-maximum scan, bit for bit: action values, argmax and nan_flag."""
    rng = np.random.default_rng(A)
    cases = _select_cases(A, rng)
    N = len(cases)
    g, r = pair(random_cfg(), N, 1, 0, 0, oracle, A=A)
    rew = np.stack([c[0] for c in cases])
    val = np.stack([c[1] for c in cases])
    rob_pv = np.zeros((N, 4), np.float32)
    rob_gr = np.tile(np.array([4.0, 3.0, 1.0, 0.3], np.float32), (N, 1))
    rob_gr[1::3, 2] = 0.6                             # two discount factors: gamma ** (dt * v_pref)
    inside = np.array([c[2] for c in cases])
    rob_gr[inside, :2] = rob_pv[inside, :2] + 0.1
    for s in (g, r):
        s.rob_pv.copy_(torch.as_tensor(rob_pv))
        s.rob_gr.copy_(torch.as_tensor(rob_gr))
        s.la_reward.copy_(torch.as_tensor(rew))
        s.values.copy_(torch.as_tensor(val))
        s.select()
    torch.cuda.synchronize()
    assert_same_bits(g.action_values, r.action_values, "action values")
    assert_same_bits(g.nan_flag, r.nan_flag, "nan_flag")
    assert_same_bits(g.argmax, r.argmax, "argmax")
    want = np.array([c[3] for c in cases])
    assert np.array_equal(np_(g.argmax), np.maximum(want, 0)), (np_(g.argmax), want)
    assert np.array_equal(np_(g.nan_flag), (want < 0).astype(np.uint8))
