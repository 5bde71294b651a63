"""K4 on the tensor cores (tcgen05): fp32-accurate mode and bf16 fast mode against a torch fp64
restatement of rl/policy/sarl.py:38-82 and against the FFMA path.  Needs a B200."""
import numpy as np
import pytest
import torch

import oracle_backend as ob
from ebc.config import SimConfig
from ebc.engine import BatchedSim

pytestmark = pytest.mark.gpu


def torch_value(w, x, cnt, with_global=True, return_weights=False):
    """fp64 reference of the value network with ragged row counts.  `return_weights`: also return the softmax
    attention weights [n_states, n] (0 on padding rows)."""
    W = {k: torch.as_tensor(v, device=x.device, dtype=torch.float64) for k, v in w.items()}
    n = x.shape[1]

    def lin(t, k, relu):
        y = t @ W[k + ".weight"].T + W[k + ".bias"]
        return torch.relu(y) if relu else y

    xd = x.double()
    h1 = lin(lin(xd, "mlp1.0", True), "mlp1.2", True)
    h2 = lin(lin(h1, "mlp2.0", True), "mlp2.2", False)
    mask = (torch.arange(n, device=x.device)[None] < cnt[:, None]).double()
    g = (h1 * mask[..., None]).sum(1, keepdim=True) / cnt[:, None, None].double()
    att_in = torch.cat([h1, g.expand(-1, n, -1)], 2) if with_global else h1
    a = lin(lin(lin(att_in, "attention.0", True), "attention.2", True), "attention.4", False)[..., 0]
    e = torch.exp(a) * (a != 0) * mask
    wts = e / e.sum(1, keepdim=True)
    f = (wts[..., None] * h2).sum(1)
    j = torch.cat([xd[:, 0, :6], f], 1)
    v = lin(lin(lin(lin(j, "mlp3.0", True), "mlp3.2", True), "mlp3.4", True), "mlp3.6", False)[:, 0]
    return (v, wts) if return_weights else v


def make_inputs(n_states, n, D, seed, ragged=True):
    rng = np.random.default_rng(seed)
    x = rng.normal(0, 1, (n_states, n, D)).astype(np.float32)
    cnt = rng.integers(1, n + 1, n_states).astype(np.int32) if ragged else np.full(n_states, n, np.int32)
    for i in range(n_states):
        x[i, cnt[i]:] = 0
    return torch.as_tensor(x, device="cuda:0"), torch.as_tensor(cnt, device="cuda:0")


@pytest.mark.parametrize("weights,H,S,typed", [("weights_ebcadrl.npz", 10, 6, True),
                                                ("weights_sarl_baseline.npz", 5, 0, False),
                                                ("weights_ebcadrl.npz", 24, 6, True)])
@pytest.mark.parametrize("n_states", [37, 3000])
def test_tc_modes_vs_fp64(weights, H, S, typed, n_states):
    w = ob.load_weights(weights)
    cfg = SimConfig()
    cfg.with_agent_type = typed
    sim = BatchedSim(cfg, 1, H, S, 0, 81, device="cuda:0")
    sim.set_weights(w)
    assert sim.value_mode() == "tc_fp16x2"        # default when the network fits the tiling
    x, cnt = make_inputs(n_states, H + S, cfg.D, seed=n_states + H)
    ref = torch_value(w, x, cnt)
    scale = max(1.0, ref.abs().max().item())
    out = {}
    for mode in ("fp32", "tc_fp32", "tc_fp16x2", "tc_bf16"):
        sim.set_value_mode(mode)
        out[mode] = sim.value(x, cnt).double()
        torch.cuda.synchronize()
    err = {m: (v - ref).abs().max().item() for m, v in out.items()}
    print(weights, H + S, n_states, err)
    assert err["fp32"] < 1e-4 * scale
    assert err["tc_fp32"] < 2e-5 * scale, err     # fp32-accurate: as good as (or better than) FFMA
    assert err["tc_fp16x2"] < 4e-5 * scale, err   # two fp16 parts (22 bits), 3 MMAs per product
    assert err["tc_bf16"] < 0.1 * scale, err      # bf16 operands: percent-level
    assert err["tc_bf16"] > err["tc_fp32"]


def test_tc_matches_golden_argmax(oracle):
    """End to end on a reference trace: tensor-core fp32-accurate values keep the reference's argmax."""
    name = "trace_cfg2_h10_seed7"
    tr = ob.Trace(name)
    H, S, R = tr.dims()
    N = tr.n_steps
    g = BatchedSim(tr.sim_config(), N, H, S, R, 81, device="cuda:0")
    g.set_actions(tr.z["actions"])
    g.set_weights(ob.load_weights(ob.TRACE_WEIGHTS[name]))
    for t in range(N):
        tr.load_into(g, t, episode=t)
    res = {}
    for mode in ("tc_fp32", "tc_fp16x2", "tc_bf16"):
        g.set_value_mode(mode)
        g.decide()
        torch.cuda.synchronize()
        has = [t for t in range(N) if tr.has(t, "la_value")]
        ref_val = np.stack([tr.get(t, "la_value") for t in has])
        dv = np.abs(g.values.cpu().numpy()[has] - ref_val).max()
        flips = sum(int(g.argmax[t]) != tr.steps[t]["argmax"] for t in has)
        big = sum(int(g.argmax[t]) != tr.steps[t]["argmax"] and tr.steps[t]["top2_gap"] >= 5e-4 for t in has)
        res[mode] = (dv, flips, big, len(has))
    print(res)
    assert res["tc_fp32"][0] < 2e-4 and res["tc_fp32"][2] == 0 and res["tc_fp32"][1] <= 2
    assert res["tc_fp16x2"][0] < 2e-4 and res["tc_fp16x2"][2] == 0 and res["tc_fp16x2"][1] <= 2
    assert res["tc_bf16"][0] < 0.1


@pytest.mark.parametrize("n_states", [0, 1, 127, 128, 129, 257])
def test_tc_ragged_batch_sizes(n_states):
    """Batch sizes around the 128-state tiles of the pooled-feature scratch (an empty batch launches nothing; partial last
    tiles of both kernels; the state right after a tile boundary); every state's value must equal the value the same
    state gets inside a large batch, bit for bit, in every mode."""
    w = ob.load_weights("weights_ebcadrl.npz")
    cfg = SimConfig()
    cfg.with_agent_type = True
    sim = BatchedSim(cfg, 1, 10, 6, 0, 81, device="cuda:0")
    sim.set_weights(w)
    x, cnt = make_inputs(300, 16, cfg.D, seed=5)
    for mode in ("tc_fp16x2", "tc_fp32", "tc_bf16", "fp32"):
        sim.set_value_mode(mode)
        big = sim.value(x, cnt).clone()
        small = sim.value(x[:n_states], cnt[:n_states]).clone()
        torch.cuda.synchronize()
        assert small.shape[0] == n_states
        assert torch.equal(small, big[:n_states]), mode


@pytest.mark.parametrize("n,with_global", [(16, False), (7, False), (8, True), (32, True)])
def test_tc_random_networks(n, with_global):
    """Shapes the shipped checkpoints do not cover: no global state (sarl.py:28-32 with_global_state = False,
    the MMA schedule then has no global K chunk), odd widths (padding columns that alias a neighbouring
    accumulator must stay exact zeros), row counts that do / do not divide the warp."""
    rng = np.random.default_rng(100 + n)
    D = 13
    dims = {"mlp1": [D, 250 if with_global else 168, 120], "mlp2": [120, 104, 52], "attention": [240 if with_global else 120, 88, 72, 1],
            "mlp3": [58, 180, 90, 70, 1]}
    w = {}
    for name, ds in dims.items():
        for i in range(len(ds) - 1):
            b = 1.0 / np.sqrt(ds[i])
            w["%s.%d.weight" % (name, 2 * i)] = rng.uniform(-b, b, (ds[i + 1], ds[i])).astype(np.float32)
            w["%s.%d.bias" % (name, 2 * i)] = rng.uniform(-b, b, ds[i + 1]).astype(np.float32)
    cfg = SimConfig()
    cfg.with_agent_type = False
    sim = BatchedSim(cfg, 1, n, 0, 0, 81, device="cuda:0")
    sim.set_weights(w, with_global_state=with_global)
    x, cnt = make_inputs(1111, n, cfg.D, seed=n)
    ref = torch_value(w, x, cnt, with_global)
    scale = max(1.0, ref.abs().max().item())
    for mode in ("fp32", "tc_fp16x2", "tc_fp32"):
        sim.set_value_mode(mode)
        out = sim.value(x, cnt).double()
        torch.cuda.synchronize()
        err = (out - ref).abs().max().item()
        print(n, with_global, mode, err)
        assert err < 5e-5 * scale, (mode, err)


def test_nan_and_overflow_stay_visible():
    """A NaN (or, in the fp16-split mode, an activation beyond the fp16 range) must come out as NaN for that state --
    the ReLU keeps NaN, nothing clamps -- so that K5's nan_flag / the reference's ValueError can fire; the other
    states of the same tile are unaffected."""
    w = ob.load_weights("weights_ebcadrl.npz")
    cfg = SimConfig()
    cfg.with_agent_type = True
    sim = BatchedSim(cfg, 1, 10, 6, 0, 81, device="cuda:0")
    sim.set_weights(w)
    x, cnt = make_inputs(300, 16, cfg.D, seed=5, ragged=False)
    clean = {}
    for mode in ("fp32", "tc_fp16x2", "tc_fp32"):
        sim.set_value_mode(mode)
        clean[mode] = sim.value(x, cnt).clone()
    x[7, 3, 2] = float("nan")
    x[130, 0, 1] = 1e30          # overflows every 16-bit part and the fp32 products
    for mode in ("fp32", "tc_fp16x2", "tc_fp32"):
        sim.set_value_mode(mode)
        out = sim.value(x, cnt)
        torch.cuda.synchronize()
        assert torch.isnan(out[7]), mode
        assert not torch.isfinite(out[130]) or out[130].abs() > 1e6, (mode, out[130])
        ok = torch.ones(300, dtype=torch.bool, device="cuda:0")
        ok[7] = ok[130] = False
        assert torch.equal(out[ok], clean[mode][ok]), mode
