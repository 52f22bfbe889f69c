"""Dispatch plan and router backward at the shapes of the multi-CTA paths: the plan bit for bit against the oracle's
replay of the reference rule, the router gradients against autograd through the oracle's router."""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import apertis_oracle as O

pytestmark = pytest.mark.gpu


def dev():
    return torch.device("cuda:0")


def _plan_case(S, E, K, cap, ties, inactive, seed):
    rng = np.random.default_rng(seed)
    idx = np.stack([rng.permutation(E)[:K] for _ in range(S)]).astype(np.int32)
    idx[: S // 3, 0] = 1 % E                            # skew: one expert overflows
    w = rng.random((S, K)).astype(np.float32) * 0.9 + 0.05
    if ties:
        w = np.round(w * 4) / 4 + 0.0625                # few distinct weights: long runs of ties at the threshold
    active = None
    if inactive:
        active = np.ones(E, dtype=bool)
        active[inactive] = False
    return idx, w, active


def _check_plan(idx, w, E, cap, active, fixed_seg=0):
    from apertis_llm_b200 import ops
    S, K = idx.shape
    kept, counts, groups = O.moe_plan(idx, w, E, min(cap, S), active)
    d = dev()
    act_t = torch.from_numpy(active.astype(np.int32)).to(d) if active is not None else None
    p = ops.moe_plan(torch.from_numpy(idx).to(d), torch.from_numpy(w).to(d), E, cap, act_t, fixed_seg=fixed_seg)
    torch.cuda.synchronize()
    assert np.array_equal(p["counts"].cpu().numpy(), counts.astype(np.int32)), "per-expert counts"
    row_of = p["row_of"].cpu().numpy()
    assert np.array_equal(row_of >= 0, kept), "kept (token, slot) sets"
    seg = p["seg_off"].cpu().numpy()
    # positions: inside an expert's segment, slot k's kept tokens follow slot k-1's, each in token order
    for e in range(E):
        expect = [(s, k) for k in range(K) for s in groups.get((k, e), [])]
        if not expect:
            continue
        ss, kk = np.array(expect).T
        assert np.array_equal(row_of[ss, kk], seg[e] + np.arange(len(expect))), f"row positions of expert {e}"
    tok, slot = p["tok_of_row"].cpu().numpy(), p["slot_of_row"].cpu().numpy()
    rows = row_of[kept]
    s_idx, k_idx = np.nonzero(kept)
    assert np.array_equal(tok[rows], s_idx) and np.array_equal(slot[rows], k_idx)
    if fixed_seg:
        assert np.array_equal(seg, np.arange(E + 1) * fixed_seg)


@pytest.mark.parametrize("S", [1, 4095, 32768, 131072])
@pytest.mark.parametrize("E,K", [(2, 1), (8, 2), (32, 3)])
def test_plan_bit_exact_multichunk(S, E, K):
    cap = max(1, int(S * K / E * 0.6))                  # most experts overflow
    idx, w, active = _plan_case(S, E, K, cap, ties=False, inactive=None, seed=S + E)
    _check_plan(idx, w, E, cap, active)


@pytest.mark.parametrize("S,E,K,cap,inactive", [(32768, 8, 2, 5120, None), (131072, 8, 3, 20000, [2, 5]),
                                                (4095, 32, 2, 100, [0]), (32768, 2, 1, 9000, None)])
def test_plan_heavy_ties_and_inactive(S, E, K, cap, inactive):
    idx, w, active = _plan_case(S, E, K, cap, ties=True, inactive=inactive, seed=cap)
    _check_plan(idx, w, E, cap, active)


@pytest.mark.parametrize("cap_limited", [True, False])
def test_plan_fixed_seg(cap_limited):
    from apertis_llm_b200 import _lib
    S, E, K = 32768, 8, 2
    cap = 5120 if cap_limited else S
    idx, w, active = _plan_case(S, E, K, cap, ties=True, inactive=[3], seed=7)
    RA = _lib.ROW_ALIGN
    if cap_limited:
        seg = (cap + RA - 1) // RA * RA
    else:
        seg = (int(np.bincount(idx.reshape(-1), minlength=E).max()) + RA - 1) // RA * RA
    _check_plan(idx, w, E, cap, active, fixed_seg=seg)


def _router_case(x_dtype, seed=0):
    """C2 router dims with a capacity-limited plan; returns kernel inputs and the oracle's autograd gradients."""
    from apertis_llm_b200 import ops
    S, Dm, E, K, alpha = 4096, 704, 8, 2, 0.1
    sd = O.make_layer_params(Dm, 11, 256, E, seed=seed)
    _, moe, _ = O.split_layer_params(sd)
    x, noise = O.make_inputs(1, S, Dm, E, seed=seed)
    x2 = x.reshape(S, Dm).to(x_dtype).float()           # the kernel and the oracle see the same (rounded) input
    d = dev()
    ns = F.softplus(moe["w_noise"]) * alpha
    r = ops.moe_route(x2.to(x_dtype).to(d), moe["router_norm.weight"].to(d), moe["router_norm.bias"].to(d), 1e-12,
                      moe["router.weight"].to(d), moe["router.bias"].to(d), noise.to(d), ns.to(d), K)
    cap = int(S / E * 1.25)
    plan = ops.moe_plan(r["idx"], r["w"], E, cap)
    g = torch.Generator().manual_seed(seed + 1)
    max_rows = plan["max_rows"]
    dw_row = torch.randn(max_rows, generator=g)
    dxrow = torch.randn(max_rows, Dm, generator=g)
    scal = torch.tensor([0.3, 0.02])
    fvec = (r["aux"][E:2 * E] / S).cpu()
    row_of = plan["row_of"].cpu().long()

    # reference: autograd through the oracle's router, with the same routing decisions and upstream gradients
    p = {k: moe[k].clone().double().requires_grad_(True) for k in ("router_norm.weight", "router_norm.bias", "router.weight",
                                                                   "router.bias", "w_noise")}
    xr = x2.double().clone().requires_grad_(True)
    logits, gates, probs, idx, wts = O.moe_router(p, xr, eps=1e-12, noise=noise.double(), alpha=alpha, K=K)
    assert torch.equal(idx.int(), r["idx"].cpu()), "routing differs from the oracle"
    keptm = row_of >= 0
    dw = torch.where(keptm, dw_row.double()[row_of.clamp(min=0)], torch.zeros((), dtype=torch.float64))
    gx = torch.where(keptm.unsqueeze(-1), dxrow.double()[row_of.clamp(min=0)], torch.zeros((), dtype=torch.float64)).sum(1)
    lse = torch.logsumexp(logits, -1)
    loss = (wts * dw).sum() + scal[0].double() * (gates * fvec.double()).sum() + scal[1].double() * (lse ** 2).sum() + (xr * gx).sum()
    loss.backward()
    ref = dict(dx=xr.grad, dWr=p["router.weight"].grad, dbr=p["router.bias"].grad, drn_w=p["router_norm.weight"].grad,
               drn_b=p["router_norm.bias"].grad, dns=p["w_noise"].grad / (torch.sigmoid(p["w_noise"].detach()) * alpha))
    inputs = dict(x2=x2.to(x_dtype).to(d), r=r, plan=plan, moe={k: v.to(d) for k, v in moe.items()}, noise=noise.to(d),
                  fvec=fvec.to(d), scal=scal.to(d), dw_row=dw_row.to(d), dxrow=dxrow.to(d), S=S, Dm=Dm, E=E, K=K)
    return inputs, ref


def _router_bwd(a):
    from apertis_llm_b200._lib import call, query, ptr, dt, stream_ptr
    S, Dm, E, K = a["S"], a["Dm"], a["E"], a["K"]
    d = dev()
    f32 = dict(dtype=torch.float32, device=d)
    r, moe = a["r"], a["moe"]
    out = dict(dx=torch.empty_like(a["x2"]), dWr=torch.empty(E, Dm, **f32), dbr=torch.empty(E, **f32),
               drn_w=torch.empty(Dm, **f32), drn_b=torch.empty(Dm, **f32), dns=torch.empty(E, **f32))
    nws = query("ab_moe_router_bwd_workspace_bytes", S, Dm, E)
    ws = torch.empty(nws, dtype=torch.uint8, device=d)
    call("ab_moe_router_bwd", ptr(a["x2"]), ptr(r["stats"]), ptr(moe["router_norm.weight"]), ptr(moe["router_norm.bias"]),
         ptr(moe["router.weight"]), ptr(moe["router.bias"]), ptr(r["gates"]), ptr(r["idx"]), ptr(r["probs"]), ptr(r["lse"]),
         ptr(r["lclean"]), ptr(a["noise"]), ptr(a["fvec"]), ptr(a["scal"]), ptr(a["dw_row"]), ptr(a["dxrow"]),
         ptr(a["plan"]["row_of"]), ptr(out["dx"]), ptr(out["dWr"]), ptr(out["dbr"]), ptr(out["drn_w"]), ptr(out["drn_b"]),
         ptr(out["dns"]), ptr(ws), ws.numel(), S, Dm, E, K, dt(a["x2"]), stream_ptr())
    torch.cuda.synchronize()
    return out


def _rel(a, b):
    a, b = a.detach().double().cpu(), b.detach().double().cpu()
    return float((a - b).norm() / b.norm().clamp(min=1e-30))


@pytest.mark.parametrize("x_dtype", [torch.float32, torch.bfloat16])
def test_router_bwd_vs_oracle_autograd(x_dtype):
    a, ref = _router_case(x_dtype)
    out = _router_bwd(a)
    tol = dict(dx=1e-5 if x_dtype == torch.float32 else 8e-3)      # dx is stored in x's dtype
    for name in ("dx", "dWr", "dbr", "drn_w", "drn_b", "dns"):
        assert _rel(out[name], ref[name]) < tol.get(name, 1e-4), f"{name}: rel err {_rel(out[name], ref[name]):.3g}"


@pytest.mark.parametrize("x_dtype", [torch.float32, torch.bfloat16])
def test_router_bwd_is_deterministic(x_dtype):
    a, _ = _router_case(x_dtype, seed=3)
    o1, o2 = _router_bwd(a), _router_bwd(a)
    for name in o1:
        assert torch.equal(o1[name], o2[name]), f"{name} differs between two identical calls"
