"""The MoE router, dispatch plan, combine and expert-LayerNorm kernels across the expert counts, top-k and hidden sizes that
AdaptiveExpertSystem accepts (num_experts <= 32, experts_per_token <= 8, hidden sizes up to the router's shared-memory
bound).  Each launcher picks a template instance by E, K and the hidden size; every instance is run here against a float64
reference of the same operation, and the sub-layer end to end against the oracle."""
import itertools

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import apertis_oracle as O
from tests.util import rel_err

TOL = {torch.float32: 1e-4, torch.bfloat16: 2e-2}
EPS = 1e-12
ALPHA = 0.1
f32, bf16 = torch.float32, torch.bfloat16
gpu = pytest.mark.gpu


def dev():
    return torch.device("cuda:0")


def _lib():
    from apertis_llm_b200 import _lib as L
    return L


# ------------------------------------------------------------------------------------------------
# host: hidden sizes the router cannot stage are refused at construction
# ------------------------------------------------------------------------------------------------
def test_router_shared_memory_bound_is_checked_at_construction():
    from apertis_llm_b200 import AdaptiveExpertSystem, BlockConfig
    from apertis_llm_b200.modules import ROUTER_SMEM_LIMIT, router_max_hidden, router_smem_bytes
    cfg = lambda E, Dm: BlockConfig(hidden_size=Dm, num_attention_heads=1, intermediate_size=8, num_experts=E, experts_per_token=2)
    assert [router_max_hidden(E) for E in (8, 16, 32)] == [5792, 3208, 1688]
    for E in (1, 2, 8, 16, 32):
        Dm = router_max_hidden(E)
        assert router_smem_bytes(E, Dm) <= ROUTER_SMEM_LIMIT < router_smem_bytes(E, Dm + 8)
    for E, Dm in ((32, 1696), (16, 3216), (8, 5800), (16, 4096)):
        with pytest.raises(ValueError, match=f"hidden_size must be <= {router_max_hidden(E)}"):
            AdaptiveExpertSystem(cfg(E, Dm))
    for E, Dm in ((32, 1688), (16, 3208), (8, 5792)):
        AdaptiveExpertSystem(cfg(E, Dm))


# ------------------------------------------------------------------------------------------------
# router forward against float64
# ------------------------------------------------------------------------------------------------
def _router_params(E, Dm, seed):
    g = torch.Generator().manual_seed(seed)
    return {"router_norm.weight": 1.0 + 0.1 * torch.randn(Dm, generator=g), "router_norm.bias": 0.1 * torch.randn(Dm, generator=g),
            "router.weight": torch.randn(E, Dm, generator=g) / Dm ** 0.5, "router.bias": 0.2 * torch.randn(E, generator=g),
            "w_noise": torch.randn(E, generator=g)}


def _router_inputs(S, E, Dm, dtype, seed):
    """x [S, Dm] rounded to `dtype` (returned as fp32, the values the kernel reads) and the routing noise draw [S, E]."""
    g = torch.Generator().manual_seed(10_000 + seed)
    x = (torch.randn(S, Dm, generator=g) * 1.5 + 0.3).to(dtype).float()
    return x, torch.randn(S, E, generator=g)


def _route(x, p, noise, K, dtype, quant=0):
    from apertis_llm_b200 import ops
    d = dev()
    ns = F.softplus(p["w_noise"]) * ALPHA
    r = ops.moe_route(x.to(dtype).to(d), p["router_norm.weight"].to(d), p["router_norm.bias"].to(d), EPS, p["router.weight"].to(d),
                      p["router.bias"].to(d), noise.to(d) if noise is not None else None, ns.to(d) if noise is not None else None,
                      K, quant)
    torch.cuda.synchronize()
    return {k: v.cpu() for k, v in r.items()}


def _route_ref(x, p, noise):
    """The router forward in float64: LayerNorm, Linear, noise * softplus(w_noise) * alpha, softmax, logsumexp."""
    xd = x.double()
    mean = xd.mean(-1)
    rstd = (xd.var(-1, unbiased=False) + EPS).rsqrt()
    xn = (xd - mean[:, None]) * rstd[:, None] * p["router_norm.weight"].double() + p["router_norm.bias"].double()
    lclean = xn @ p["router.weight"].double().t() + p["router.bias"].double()
    logits = lclean if noise is None else lclean + noise.double() * (F.softplus(p["w_noise"].double()) * ALPHA)
    return dict(stats=torch.stack([mean, rstd], -1), lclean=lclean, logits=logits, gates=torch.softmax(logits, -1),
                lse=torch.logsumexp(logits, -1))


def _check_selection(r, K):
    """Top-K on the kernel's own gates (descending, ties to the lower expert id), probs the selected gates exactly."""
    _, idx_ref = O.topk_lowest_index(r["gates"].numpy(), K)
    assert np.array_equal(r["idx"].numpy(), idx_ref.astype(np.int32)), "top-k selection on the kernel's gates"
    assert torch.equal(r["probs"], r["gates"].gather(1, r["idx"].long()))


def _check_route(r, ref, S, E, K):
    for name in ("stats", "lclean", "logits", "gates", "lse"):
        assert rel_err(r[name], ref[name]) < 1e-5, f"{name}: {rel_err(r[name], ref[name]):.3g}"
    _check_selection(r, K)
    pk = ref["gates"].gather(1, r["idx"].long())
    assert rel_err(r["w"], pk / (pk.sum(-1, keepdim=True) + 1e-6)) < 1e-5, "w"
    aux = r["aux"]
    assert rel_err(aux[:E], ref["gates"].sum(0)) < 1e-5, "aux: gate sums"
    assert torch.equal(aux[E:2 * E], torch.bincount(r["idx"].reshape(-1).long(), minlength=E).float()), "aux: selection counts"
    assert rel_err(aux[2 * E:], (ref["lse"] ** 2).sum().reshape(1)) < 1e-5, "aux: sum of lse^2"


# (E, K, Dm, dtype) -> the instance ab_moe_router_fwd launches: EM = 8 / 16 / 32 by E, NV = 4 / 6 / 8 / 16 by
# ceil(Dm / (32 * V)) with V = 4 (fp32) or 8 (bf16); the streaming kernel when the row does not fit in registers
ROUTER_FWD_CASES = [
    (1, 1, 64, f32),        # EM 8, NV 4; one expert
    (8, 8, 704, f32),       # EM 8, NV 6; K = E
    (8, 3, 1024, f32),      # EM 8, NV 8
    (8, 2, 1600, f32),      # EM 8, NV 16
    (8, 1, 2048, f32),      # EM 8, NV 16, full
    (8, 2, 2560, f32),      # streaming, EM 8
    (16, 3, 448, f32),      # EM 16, NV 4
    (16, 8, 704, f32),      # EM 16, NV 6
    (16, 2, 1024, f32),     # EM 16, NV 8
    (16, 4, 1600, f32),     # streaming, EM 16
    (32, 8, 448, f32),      # EM 32, NV 4
    (32, 2, 704, f32),      # EM 32, NV 6
    (32, 3, 1024, f32),     # EM 32, NV 8
    (32, 8, 1688, f32),     # streaming, EM 32, at the shared-memory bound
    (2, 2, 512, bf16),      # EM 8, NV 4; K = E
    (8, 2, 704, bf16),      # EM 8, NV 4 (nv 3)
    (8, 3, 1536, bf16),     # EM 8, NV 6
    (8, 2, 2048, bf16),     # EM 8, NV 8
    (8, 8, 4096, bf16),     # EM 8, NV 16; K = E
    (8, 2, 5120, bf16),     # streaming, EM 8
    (16, 2, 256, bf16),     # EM 16, NV 4
    (16, 4, 1536, bf16),    # EM 16, NV 6
    (16, 4, 1600, bf16),    # EM 16, NV 8
    (16, 1, 3208, bf16),    # streaming, EM 16, at the shared-memory bound
    (32, 8, 1024, bf16),    # EM 32, NV 4
    (32, 2, 1536, bf16),    # EM 32, NV 6
    (32, 8, 1688, bf16),    # EM 32, NV 8, at the shared-memory bound
]


def _case_id(c):
    return f"E{c[0]}-K{c[1]}-Dm{c[2]}-{'f32' if c[3] == f32 else 'bf16'}"


@gpu
@pytest.mark.parametrize("noise", [True, False])
@pytest.mark.parametrize("E,K,Dm,dtype", ROUTER_FWD_CASES, ids=[_case_id(c) for c in ROUTER_FWD_CASES])
def test_router_fwd_vs_fp64(E, K, Dm, dtype, noise):
    S = 1000
    p = _router_params(E, Dm, seed=E * 7 + Dm)
    x, nz = _router_inputs(S, E, Dm, dtype, seed=Dm + K)
    nz = nz if noise else None
    r = _route(x, p, nz, K, dtype)
    _check_route(r, _route_ref(x, p, nz), S, E, K)


@gpu
@pytest.mark.parametrize("S,E,K,Dm,dtype", [(1, 32, 8, 1688, f32), (1, 8, 2, 704, bf16), (1, 1, 1, 64, f32),
                                            (65537, 32, 8, 64, f32), (65537, 16, 4, 256, bf16), (65537, 8, 2, 128, f32)])
def test_router_fwd_one_token_and_capped_grid(S, E, K, Dm, dtype):
    """S = 1: a single warp; S = 65537: more rows than the capped grid has warps, so every warp loops (the register
    kernel prefetches its next row) and the aux sums add many rows per CTA."""
    p = _router_params(E, Dm, seed=S + E)
    x, nz = _router_inputs(S, E, Dm, dtype, seed=S)
    r = _route(x, p, nz, K, dtype)
    _check_route(r, _route_ref(x, p, nz), S, E, K)


# ------------------------------------------------------------------------------------------------
# router forward with the logits rounded like an autocast Linear (ROUTER_BF16 / ROUTER_FP16)
# ------------------------------------------------------------------------------------------------
def _ulp(v, dtype):
    """Spacing of `dtype` at |v| (float64 in, float64 out); fp16's subnormal spacing below its smallest normal."""
    mant, emin = (7, -126) if dtype == bf16 else (10, -14)
    _, e = torch.frexp(v.abs().clamp(min=1e-300))
    return torch.ldexp(torch.ones_like(v), (e - 1).clamp(min=emin) - mant)


# rounded logits that differ from the float64 emulation at all: the kernel accumulates the dot product in fp32, so a
# logit within that error of a rounding midpoint lands on the neighbouring value.  Measured on a B200 over the cases
# below: at most 0.012 % (bf16) and 0.104 % (fp16) of the logits; bound 0.5 %.
QUANT_MISMATCH_MAX = 0.005


@gpu
@pytest.mark.parametrize("mode", ["bf16", "fp16"])
@pytest.mark.parametrize("E,K,Dm,dtype", [(8, 2, 704, f32), (8, 2, 704, bf16), (16, 4, 1024, f32), (32, 8, 448, bf16),
                                          (16, 2, 1600, f32), (32, 8, 1688, bf16)],
                         ids=["E8-Dm704-f32", "E8-Dm704-bf16", "E16-Dm1024-f32", "E32-Dm448-bf16", "E16-Dm1600-f32-streaming",
                              "E32-Dm1688-bf16"])
def test_router_fwd_autocast_rounding(E, K, Dm, dtype, mode):
    L = _lib()
    quant, tdt = (L.ROUTER_BF16, torch.bfloat16) if mode == "bf16" else (L.ROUTER_FP16, torch.float16)
    S = 4096
    p = _router_params(E, Dm, seed=E + Dm)
    x, _ = _router_inputs(S, E, Dm, dtype, seed=E * Dm)
    r = _route(x, p, None, K, dtype, quant)
    assert rel_err(r["stats"], _route_ref(x, p, None)["stats"]) < 1e-5
    # reference: the fp32 LayerNorm with the kernel's own mean and rstd (checked just above), evaluated as the kernel does,
    # ((x - mean) * rstd) * w + b with one rounding for the last multiply-add.  A different fp32 normalisation would round
    # an element of the row to the neighbouring bf16 / fp16 value now and then, and on a logit that cancels to near zero
    # that shows as many ulps.  Then the normalised row, the weight and the bias rounded to the autocast dtype, the dot
    # product in float64, the logit rounded once.
    mean, rstd = r["stats"][:, :1], r["stats"][:, 1:]
    t = (x - mean) * rstd
    xn = (t.double() * p["router_norm.weight"].double() + p["router_norm.bias"].double()).float()
    xq, Wq, bq = xn.to(tdt).double(), p["router.weight"].to(tdt).double(), p["router.bias"].to(tdt).double()
    ref = (xq @ Wq.t() + bq).to(tdt).double()
    # before its one rounding the kernel's fp32 dot product may be off by the summation bound (Dm/32 + 6 additions in a
    # chain: per lane, then the warp's tree) * 2^-24 * sum |terms|: on a logit that cancels to near zero that can exceed
    # the target dtype's spacing.  So: one ulp (two half-ulp roundings) plus that bound.
    acc = (Dm / 32 + 8) * 2.0 ** -24 * (xq.abs() @ Wq.abs().t() + bq.abs())
    lg = r["lclean"].double()
    assert torch.equal(r["logits"], r["lclean"])
    assert torch.equal(lg, lg.to(tdt).double()), "every logit is a value of the autocast dtype"
    tol = _ulp(torch.maximum(lg.abs(), ref.abs()), tdt) + acc
    assert bool(((lg - ref).abs() <= tol).all()), f"max |diff| / bound {float(((lg - ref).abs() / tol).max()):.3g}"
    frac = float((lg != ref).double().mean())
    assert frac <= QUANT_MISMATCH_MAX, f"{frac:.4f} of the logits differ from the emulation"
    _check_selection(r, K)                 # rounded logits tie often: the lower-index rule decides
    r0 = _route(x, p, None, K, dtype, L.ROUTER_EXACT)
    assert not torch.equal(r0["lclean"], r["lclean"])


# ------------------------------------------------------------------------------------------------
# router backward: unfused (E > 8 or Dm > 1024) and the fused column kernel with KM = 8 (K > 2)
# ------------------------------------------------------------------------------------------------
def _router_case(E, K, Dm, x_dtype, S=4096, seed=0):
    """A capacity-limited plan on the kernel's routing; returns the kernel inputs and the gradients of fp64 autograd
    through the oracle's router, with the kernel's selection."""
    from apertis_llm_b200 import ops
    moe = _router_params(E, Dm, seed=seed + E + Dm)
    x2, noise = _router_inputs(S, E, Dm, x_dtype, seed=seed)
    d = dev()
    ns = F.softplus(moe["w_noise"]) * ALPHA
    r = ops.moe_route(x2.to(x_dtype).to(d), moe["router_norm.weight"].to(d), moe["router_norm.bias"].to(d), EPS,
                      moe["router.weight"].to(d), moe["router.bias"].to(d), noise.to(d), ns.to(d), K)
    # the plan fills the experts slot by slot: a capacity just under the mean load drops some of the last slot's rows
    # and keeps most of them (at 1.25 S / E every slot past the second would be dropped whole for K > 2)
    cap = int(S * K / E * 0.95)
    plan = ops.moe_plan(r["idx"], r["w"], E, cap)
    g = torch.Generator().manual_seed(seed + 1)
    max_rows = plan["max_rows"]
    dw_row = torch.randn(max_rows, generator=g)
    dxrow = torch.randn(max_rows, Dm, generator=g)
    scal = torch.tensor([0.3, 0.02])
    fvec = (r["aux"][E:2 * E] / S).cpu()
    row_of = plan["row_of"].cpu().long()
    assert (row_of < 0).any() and (row_of[:, K - 1] >= 0).float().mean() > 0.5, "last slot mostly kept, some rows dropped"
    idx = r["idx"].cpu().long()

    p = {k: v.clone().double().requires_grad_(True) for k, v in moe.items()}
    xr = x2.double().clone().requires_grad_(True)
    logits, gates, _, _, _ = O.moe_router(p, xr, eps=EPS, noise=noise.double(), alpha=ALPHA, K=K)
    probs = gates.gather(1, idx)                       # the kernel's selection (fp32 near-ties may order differently)
    wts = probs / (probs.sum(-1, keepdim=True) + 1e-6)
    keptm = row_of >= 0
    dw = torch.where(keptm, dw_row.double()[row_of.clamp(min=0)], torch.zeros((), dtype=torch.float64))
    gx = torch.where(keptm.unsqueeze(-1), dxrow.double()[row_of.clamp(min=0)], torch.zeros((), dtype=torch.float64)).sum(1)
    lse = torch.logsumexp(logits, -1)
    loss = (wts * dw).sum() + scal[0].double() * (gates * fvec.double()).sum() + scal[1].double() * (lse ** 2).sum() + (xr * gx).sum()
    loss.backward()
    ref = dict(dx=xr.grad, dWr=p["router.weight"].grad, dbr=p["router.bias"].grad, drn_w=p["router_norm.weight"].grad,
               drn_b=p["router_norm.bias"].grad, dns=p["w_noise"].grad / (torch.sigmoid(p["w_noise"].detach()) * ALPHA))
    inputs = dict(x2=x2.to(x_dtype).to(d), r=r, plan=plan, moe={k: v.to(d) for k, v in moe.items()}, noise=noise.to(d),
                  fvec=fvec.to(d), scal=scal.to(d), dw_row=dw_row.to(d), dxrow=dxrow.to(d), S=S, Dm=Dm, E=E, K=K)
    return inputs, ref


def _router_bwd(a):
    from apertis_llm_b200._lib import call, query, ptr, dt, stream_ptr
    S, Dm, E, K = a["S"], a["Dm"], a["E"], a["K"]
    d = dev()
    f = dict(dtype=torch.float32, device=d)
    r, moe = a["r"], a["moe"]
    out = dict(dx=torch.empty_like(a["x2"]), dWr=torch.empty(E, Dm, **f), dbr=torch.empty(E, **f),
               drn_w=torch.empty(Dm, **f), drn_b=torch.empty(Dm, **f), dns=torch.empty(E, **f))
    ws = torch.empty(query("ab_moe_router_bwd_workspace_bytes", S, Dm, E), dtype=torch.uint8, device=d)
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


@gpu
@pytest.mark.parametrize("x_dtype", [f32, bf16])
@pytest.mark.parametrize("E,K,Dm", [(16, 4, 704), (32, 8, 1024), (8, 3, 704), (8, 2, 1600)],
                         ids=["unfused-EM16", "unfused-EM32", "fused-KM8", "unfused-EM8-Dm1600"])
def test_router_bwd_vs_fp64_autograd(E, K, Dm, x_dtype):
    a, ref = _router_case(E, K, Dm, x_dtype)
    out = _router_bwd(a)
    tol = dict(dx=1e-5 if x_dtype == f32 else 8e-3)      # dx is stored in x's dtype
    for name in ("dx", "dWr", "dbr", "drn_w", "drn_b", "dns"):
        assert _rel(out[name], ref[name]) < tol.get(name, 1e-4), f"{name}: rel err {_rel(out[name], ref[name]):.3g}"
    again = _router_bwd(a)
    for name in out:
        assert torch.equal(out[name], again[name]), f"{name} differs between two identical calls"


# ------------------------------------------------------------------------------------------------
# combine (unpermute) and expert LayerNorm through the C ABI on a real plan
# ------------------------------------------------------------------------------------------------
def _dispatch(S, E, K, seed, inactive=()):
    """Distinct random experts per token, gate weights, and the device plan with a capacity that drops slots."""
    from apertis_llm_b200 import ops
    g = torch.Generator().manual_seed(seed)
    idx = torch.argsort(torch.rand(S, E, generator=g), dim=1)[:, :K].to(torch.int32)
    w = torch.rand(S, K, generator=g) * 0.9 + 0.05
    d = dev()
    active = None
    if inactive:
        active = torch.ones(E, dtype=torch.int32)
        active[list(inactive)] = 0
        active = active.to(d)
    cap = max(1, int(S * K / E * 0.95))               # just under the mean load: the last slot is kept in part
    plan = ops.moe_plan(idx.to(d), w.to(d), E, cap, active)
    torch.cuda.synchronize()
    row_of = plan["row_of"].cpu().long()
    assert (row_of < 0).any() and (row_of[:, K - 1] >= 0).float().mean() > 0.5, "last slot mostly kept, some rows dropped"
    return idx, w, plan, row_of


def _kept_rows(plan, idx):
    """Valid permuted rows (< n_rows[0], token >= 0), their token, slot and expert."""
    n0 = int(plan["n_rows"][0])
    tok = plan["tok_of_row"][:n0].cpu().long()
    slot = plan["slot_of_row"][:n0].cpu().long()
    rv = torch.nonzero(tok >= 0).squeeze(1)
    return n0, rv, tok[rv], slot[rv], idx.long()[tok[rv], slot[rv]]


def _out_tol(dtype):
    # fp32: a few fp32 roundings; bf16: the final rounding, at most half a bf16 ulp = 2^-8 (3.9e-3) of the value, plus those
    return 1e-6 if dtype == f32 else 4e-3


@gpu
@pytest.mark.parametrize("Dm", [96, 704])
@pytest.mark.parametrize("K", [1, 2, 3, 4, 5, 8])
def test_unpermute_fwd_bwd_every_slot_count(K, Dm):
    """unpermute_kernel<KM = 2, 4, 8> for every (y, out) dtype pair, with and without the fp32 residual, and the combine
    backward for every (dout, y, dy) dtype triple, against float64 on a plan that drops slots."""
    from apertis_llm_b200._lib import call, dt, ptr, stream_ptr
    S, E = 1500, 16
    idx, w, plan, row_of = _dispatch(S, E, K, seed=K * 1000 + Dm)
    d = dev()
    max_rows = plan["max_rows"]
    g = torch.Generator().manual_seed(K + Dm)
    y32 = torch.randn(max_rows, Dm, generator=g)
    res = torch.randn(S, Dm, generator=g)
    dout32 = torch.randn(S, Dm, generator=g)
    kept = row_of >= 0
    wk = w.double() * kept
    n0, rv, tok, slot, _ = _kept_rows(plan, idx)
    wd, resd = w.to(d), res.to(d)          # device copies held by name: a kernel must not see their memory reused
    for ydt in (f32, bf16):
        y = y32.to(ydt)
        yd = y.to(d)
        ref = (y.double()[row_of.clamp(min=0)] * wk[..., None]).sum(1)
        for odt, with_res in itertools.product((f32, bf16), (False, True)):
            out = torch.empty(S, Dm, dtype=odt, device=d)
            call("ab_moe_unpermute", ptr(yd), ptr(plan["row_of"]), ptr(wd), ptr(resd) if with_res else None, ptr(out),
                 0.0, None, S, K, Dm, dt(ydt), dt(odt), stream_ptr())
            want = ref + res.double() if with_res else ref
            assert rel_err(out.float(), want) < _out_tol(odt), (ydt, odt, with_res)
    for ddt, ydt, dydt in itertools.product((f32, bf16), repeat=3):
        dout, y = dout32.to(ddt), y32.to(ydt)
        doutd, yd = dout.to(d), y.to(d)
        dy = torch.full((max_rows, Dm), float("nan"), dtype=dydt, device=d)
        dw_row = torch.full((max_rows,), float("nan"), device=d)
        call("ab_moe_unpermute_bwd", ptr(doutd), ptr(yd), ptr(wd), ptr(plan["tok_of_row"]), ptr(plan["slot_of_row"]),
             ptr(plan["n_rows"]), ptr(dy), ptr(dw_row), 0.0, None, K, Dm, max_rows, dt(ddt), dt(ydt), dt(dydt), stream_ptr())
        dy_ref = torch.zeros(n0, Dm, dtype=torch.float64)
        dy_ref[rv] = w.double()[tok, slot][:, None] * dout.double()[tok]
        dw_ref = torch.zeros(n0, dtype=torch.float64)
        dw_ref[rv] = (dout.double()[tok] * y.double()[rv]).sum(-1)
        assert rel_err(dy[:n0].float(), dy_ref) < _out_tol(dydt), ("dy", ddt, ydt, dydt)
        assert rel_err(dw_row[:n0], dw_ref) < 1e-5, ("dw_row", ddt, ydt, dydt)


@gpu
def test_unpermute_output_dropout_forward_and_backward_share_the_mask():
    from apertis_llm_b200._lib import call, dt, ptr, stream_ptr
    S, E, K, Dm, p = 2000, 16, 5, 704, 0.25
    idx, w, plan, row_of = _dispatch(S, E, K, seed=77)
    d = dev()
    max_rows = plan["max_rows"]
    g = torch.Generator().manual_seed(78)
    y = torch.randn(max_rows, Dm, generator=g).to(d)
    res = torch.randn(S, Dm, generator=g).to(d)
    dout = torch.randn(S, Dm, generator=g)
    seed = torch.tensor([123457, 99], dtype=torch.int32, device=d)
    wd = w.to(d)

    def fwd(res_t):
        out = torch.empty(S, Dm, device=d)
        call("ab_moe_unpermute", ptr(y), ptr(plan["row_of"]), ptr(wd), ptr(res_t), ptr(out), p, ptr(seed), S, K, Dm, dt(y), dt(out), stream_ptr())
        torch.cuda.synchronize()
        return out.cpu()

    out, out_res = fwd(None), fwd(res)
    ref = (y.cpu().double()[row_of.clamp(min=0)] * (w.double() * (row_of >= 0))[..., None]).sum(1)
    keep = out != 0
    frac = 1.0 - float(keep.double().mean())
    assert abs(frac - p) < 5 * (p * (1 - p) / keep.numel()) ** 0.5, frac
    assert rel_err(out[keep], (ref / (1 - p))[keep]) < 1e-6, "kept elements are the combine scaled by 1 / (1 - p)"
    assert rel_err(out_res - res.cpu(), out) < 1e-6, "the residual is added after the same mask"
    n0, rv, tok, slot, _ = _kept_rows(plan, idx)
    dy = torch.empty(max_rows, Dm, device=d)
    dw_row = torch.empty(max_rows, device=d)
    doutd = dout.to(d)
    call("ab_moe_unpermute_bwd", ptr(doutd), ptr(y), ptr(wd), ptr(plan["tok_of_row"]), ptr(plan["slot_of_row"]), ptr(plan["n_rows"]),
         ptr(dy), ptr(dw_row), p, ptr(seed), K, Dm, max_rows, dt(dout), dt(y), dt(dy), stream_ptr())
    gmask = dout.double() * keep / (1 - p)                  # the upstream gradient through the forward's mask
    dy_ref = torch.zeros(n0, Dm, dtype=torch.float64)
    dy_ref[rv] = w.double()[tok, slot][:, None] * gmask[tok]
    dw_ref = torch.zeros(n0, dtype=torch.float64)
    dw_ref[rv] = (gmask[tok] * y.cpu().double()[rv]).sum(-1)
    assert rel_err(dy[:n0], dy_ref) < 1e-6 and rel_err(dw_row[:n0], dw_ref) < 1e-5


@gpu
@pytest.mark.parametrize("Dm", [64, 448, 704, 1000, 1600], ids=["NIT2", "NIT4", "NIT6", "NIT8", "rows+cols"])
def test_permute_ln_fwd_bwd_every_width(Dm):
    """permute_ln_kernel for the four (x, xn) dtype pairs and the expert-LayerNorm backward - the fused kernel at
    NIT = 2/4/6/8 and the rows + cols pair above 1024 - for the four (x, dxn) dtype pairs.  The padding rows of dxn hold
    garbage, which the backward must not read into the sums."""
    from apertis_llm_b200._lib import ROW_ALIGN, call, dt, ptr, query, stream_ptr
    S, E, K = 2000, 8, 2
    idx, w, plan, row_of = _dispatch(S, E, K, seed=Dm, inactive=(5,))
    d = dev()
    max_rows = plan["max_rows"]
    g = torch.Generator().manual_seed(Dm + 1)
    x32 = torch.randn(S, Dm, generator=g) * 1.5 + 0.3
    ln_w, ln_b = 1 + 0.1 * torch.randn(E, Dm, generator=g), 0.1 * torch.randn(E, Dm, generator=g)
    dxn32 = torch.randn(max_rows, Dm, generator=g)
    n0, rv, tok, _, e_of = _kept_rows(plan, idx)
    lw, lb = ln_w.double()[e_of], ln_b.double()[e_of]
    ws = torch.empty(query("ab_moe_permute_ln_bwd_workspace_bytes", Dm, ROW_ALIGN, max_rows), dtype=torch.uint8, device=d)
    lnwd, lnbd = ln_w.to(d), ln_b.to(d)
    for xdt in (f32, bf16):
        x = x32.to(xdt)
        xd = x.double()
        stats = torch.stack([xd.mean(-1), (xd.var(-1, unbiased=False) + EPS).rsqrt()], -1).float()
        x_d, stats_d = x.to(d), stats.to(d)
        xh = (xd[tok] - stats[tok, 0:1].double()) * stats[tok, 1:2].double()
        for odt in (f32, bf16):
            xn = torch.full((max_rows, Dm), float("nan"), dtype=odt, device=d)
            call("ab_moe_permute_ln", ptr(x_d), ptr(stats_d), ptr(lnwd), ptr(lnbd), ptr(plan["tok_of_row"]),
                 ptr(plan["tile_expert"]), ptr(plan["n_rows"]), ptr(xn), Dm, ROW_ALIGN, max_rows, dt(xdt), dt(odt), stream_ptr())
            xn = xn[:n0].float().cpu()
            assert rel_err(xn[rv], xh * lw + lb) < _out_tol(odt), ("permute_ln", xdt, odt)
            pad = torch.ones(n0, dtype=torch.bool)
            pad[rv] = False
            assert bool((xn[pad] == 0).all()), "padding rows are written as zeros"
        for gdt in (f32, bf16):
            dxn = dxn32.to(gdt)
            dxn_d = dxn.to(d)
            dxrow = torch.empty(max_rows, Dm, device=d)
            dln_w, dln_b = torch.empty(E, Dm, device=d), torch.empty(E, Dm, device=d)
            call("ab_moe_permute_ln_bwd", ptr(dxn_d), ptr(x_d), ptr(stats_d), ptr(lnwd), ptr(plan["tok_of_row"]),
                 ptr(plan["tile_expert"]), ptr(plan["n_rows"]), ptr(dxrow), ptr(dln_w), ptr(dln_b), ptr(ws), ws.numel(), Dm, E,
                 ROW_ALIGN, max_rows, dt(xdt), dt(gdt), stream_ptr())
            gv = dxn.double()[rv]
            dh = gv * lw
            m1, m2 = dh.mean(-1, keepdim=True), (dh * xh).mean(-1, keepdim=True)
            dx_ref = stats[tok, 1:2].double() * (dh - m1 - xh * m2)
            dlw_ref = torch.zeros(E, Dm, dtype=torch.float64).index_add_(0, e_of, gv * xh)
            dlb_ref = torch.zeros(E, Dm, dtype=torch.float64).index_add_(0, e_of, gv)
            assert rel_err(dxrow.cpu()[rv], dx_ref) < 1e-5, ("dxrow", xdt, gdt)
            assert rel_err(dln_w, dlw_ref) < 1e-5 and rel_err(dln_b, dlb_ref) < 1e-5, ("dln_w / dln_b", xdt, gdt)


@gpu
@pytest.mark.parametrize("C", [96, 1408])
@pytest.mark.parametrize("dtype", [f32, bf16])
def test_segment_colsum(dtype, C):
    """Per-expert column sums of the permuted rows (the expert bias gradients); padding rows are zero, as the combine
    backward and the GEMMs leave them."""
    from apertis_llm_b200._lib import ROW_ALIGN, call, dt, ptr, query, stream_ptr
    S, E, K = 3000, 8, 2
    idx, w, plan, row_of = _dispatch(S, E, K, seed=C, inactive=(2,))
    d = dev()
    max_rows = plan["max_rows"]
    n0, rv, _, _, e_of = _kept_rows(plan, idx)
    g = torch.Generator().manual_seed(C)
    a = torch.zeros(max_rows, C)
    a[rv] = torch.randn(rv.numel(), C, generator=g)
    a = a.to(dtype)
    a_d = a.to(d)
    out = torch.empty(E, C, device=d)
    ws = torch.empty(query("ab_moe_segment_colsum_workspace_bytes", C, ROW_ALIGN, max_rows), dtype=torch.uint8, device=d)
    call("ab_moe_segment_colsum", ptr(a_d), ptr(plan["tile_expert"]), ptr(plan["n_rows"]), ptr(out), ptr(ws), ws.numel(), C, E,
         ROW_ALIGN, max_rows, dt(dtype), stream_ptr())
    ref = torch.zeros(E, C, dtype=torch.float64).index_add_(0, e_of, a.double()[rv])
    assert rel_err(out, ref) < 1e-5
    assert float(out[2].abs().max()) == 0.0, "an inactive expert has no rows"


# ------------------------------------------------------------------------------------------------
# plan and top-k at the large end
# ------------------------------------------------------------------------------------------------
def _plan_case(S, E, K, ties, inactive, seed):
    rng = np.random.default_rng(seed)
    idx = np.argsort(rng.random((S, E)), axis=1)[:, :K].astype(np.int32)    # K distinct experts per token
    head = idx[: S // 3]                                # skew: one expert overflows (slot 0 of a third of the tokens) ...
    dup = head[:, 1:] == 1 % E
    head[:, 1:][dup] = np.broadcast_to(head[:, :1], dup.shape)[dup]     # ... and the token's experts stay distinct
    head[:, 0] = 1 % E
    w = rng.random((S, K)).astype(np.float32) * 0.9 + 0.05
    if ties:
        w = np.round(w * 4) / 4 + 0.0625                # few distinct weights: long runs of ties at the threshold
    active = None
    if inactive:
        active = np.ones(E, dtype=bool)
        active[inactive] = False
    return idx, w, active


def _check_plan(idx, w, E, cap, active):
    from apertis_llm_b200 import ops
    S, K = idx.shape
    kept, counts, groups = O.moe_plan(idx, w, E, min(cap, S), active)
    d = dev()
    act_t = torch.from_numpy(active.astype(np.int32)).to(d) if active is not None else None
    p = ops.moe_plan(torch.from_numpy(idx).to(d), torch.from_numpy(w).to(d), E, cap, act_t)
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


@gpu
@pytest.mark.parametrize("S", [4095, 131072])
@pytest.mark.parametrize("E,K,inactive", [(32, 8, [0, 7, 31]), (16, 5, [3])])
def test_plan_bit_exact_large_topk(S, E, K, inactive):
    cap = max(1, int(S * K / E * 0.6))                  # most experts overflow
    idx, w, active = _plan_case(S, E, K, ties=True, inactive=inactive, seed=S + E)
    _check_plan(idx, w, E, cap, active)


@gpu
def test_topk_from_logits_32_experts_top8_with_ties():
    from apertis_llm_b200 import ops
    g = torch.Generator().manual_seed(32)
    S, E, K = 4096, 32, 8
    logits = torch.randn(S, E, generator=g)
    logits[::5] = torch.round(logits[::5] * 2) / 2      # many exact ties
    logits[7] = 0.5                                     # an all-equal row
    logits[11, 3::4] = 5.0                              # eight equal maxima
    gates, idx, probs, w, lse = ops.moe_topk_from_logits(logits.to(dev()), K)
    torch.cuda.synchronize()
    r = dict(gates=gates.cpu(), idx=idx.cpu(), probs=probs.cpu())
    _check_selection(r, K)
    ld = logits.double()
    assert rel_err(r["gates"], torch.softmax(ld, -1)) < 1e-6
    pk = torch.softmax(ld, -1).gather(1, r["idx"].long())
    assert rel_err(w, pk / (pk.sum(-1, keepdim=True) + 1e-6)) < 1e-6
    assert rel_err(lse, torch.logsumexp(ld, -1)) < 1e-6
    assert idx[7].tolist() == list(range(8)) and idx[11].tolist() == list(range(3, 32, 4))


# ------------------------------------------------------------------------------------------------
# ReLU and SiLU epilogues of the grouped GEMM, element by element
# ------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("act", [1, 2], ids=["relu", "silu"])
def test_grouped_gemm_relu_silu_accuracy_per_element(act):
    """One pre-activation value per row over [-12, 12] (bf16-exact), the forward epilogue (act) and the d-activation
    epilogue (EPI_DACT with an accumulator of 1) against the exact function and its derivative in float64.
    ReLU is exact.  SiLU is x * rcp.approx(1 + ex2.approx(-x log2 e)): the rounding of the exponent's argument (|x| log2 e
    2^-24 <= 1.1e-6 relative in exp) and the two approximations (2^-22 each) stay below 1.5e-6 relative in the sigmoid.
    fp32 bounds: 2e-6 |silu| for the value, 2e-6 (|silu'| + |x| s (1 - s)) for the derivative (its two terms carry the
    sigmoid's error separately).  Measured on a B200: 7.5e-7 and 6.4e-7 of those scales.  bf16 adds the output rounding,
    half an ulp = at most 2^-8 of the value (measured 3.7e-3 and 3.9e-3 of |silu| and |silu'|)."""
    L = _lib()
    from apertis_llm_b200 import ops
    d = dev()
    RA = L.ROW_ALIGN
    N, K, E = 64, 64, 1
    rows = 4 * RA
    plan = dict(tile_expert=torch.zeros(rows // RA, dtype=torch.int32, device=d), n_rows=torch.tensor([rows, rows], dtype=torch.int32, device=d))
    xs = torch.linspace(-12, 12, rows).to(torch.bfloat16)
    A = torch.zeros(rows, K, dtype=torch.bfloat16)
    A[:, 0] = xs
    W = torch.zeros(E, N, K, dtype=torch.bfloat16)
    W[0, :, 0] = 1.0                                    # pre[r, n] = xs[r]
    bias = torch.zeros(E, N)
    x32 = xs.float()[:, None].expand(rows, N)
    x = x32.double()
    s = torch.sigmoid(x)
    if act == 1:
        want, want_d = torch.relu(x), (x > 0).double()
        scale_v, scale_d = torch.zeros_like(x), torch.zeros_like(x)
    else:
        want, want_d = x * s, s * (1 + x * (1 - s))
        scale_v, scale_d = 2e-6 * want.abs(), 2e-6 * (want_d.abs() + x.abs() * s * (1 - s))
    ones = torch.zeros(rows, K, dtype=torch.bfloat16)
    ones[:, 0] = 1.0                                    # accumulator of the dact GEMM = 1
    for odt in (torch.bfloat16, torch.float32):
        h, pre = ops.grouped_gemm("nt", A.to(d), W.to(d), plan, N, K, E, bias=bias.to(d), epi=L.EPI_BIAS_ACT, act=act, out_dtype=odt, want_c2=True)
        dact = ops.grouped_gemm("nt", ones.to(d), W.to(d), plan, N, K, E, aux=x32.to(odt).to(d), epi=L.EPI_DACT, act=act, out_dtype=odt)
        torch.cuda.synchronize()
        assert torch.equal(pre.float().cpu(), x32)
        rnd = 2.0 ** -8 if odt == torch.bfloat16 else 0.0
        eh = (h.double().cpu() - want).abs()
        ed = (dact.double().cpu() - want_d).abs()
        assert bool((eh <= scale_v + rnd * want.abs()).all()), (odt, float(eh.max()))
        assert bool((ed <= scale_d + rnd * want_d.abs()).all()), (odt, float(ed.max()))


# ------------------------------------------------------------------------------------------------
# the sub-layer end to end against the oracle
# ------------------------------------------------------------------------------------------------
def _moe_module(E, K, act, Dm, I, seed):
    from apertis_llm_b200 import AdaptiveExpertSystem, BlockConfig
    sd = O.make_layer_params(Dm, 1, I, E, seed=seed)
    _, moe, _ = O.split_layer_params(sd)
    m = AdaptiveExpertSystem(BlockConfig(hidden_size=Dm, num_attention_heads=1, intermediate_size=I, num_experts=E,
                                         experts_per_token=K, hidden_act=act, hidden_dropout_prob=0.0))
    m.load_state_dict(moe, strict=True)
    m = m.to(dev()).train()
    ndrop = int(np.floor(E * 0.1))                       # whole-expert dropout of core.py:514-521 at p = 0.1
    active = None
    if ndrop:
        perm = torch.randperm(E, generator=torch.Generator().manual_seed(seed))
        active = np.ones(E, dtype=bool)
        active[perm[:ndrop].numpy()] = False
    act_t = torch.from_numpy(active.astype(np.int32)) if active is not None else None
    m._draw_active_mask = lambda device: act_t.to(device) if act_t is not None else None
    return m, moe, active


def _grad(t):
    """A leaf's gradient; zeros for an expert the oracle never ran (inactive, or no token kept)."""
    return t.grad if t.grad is not None else torch.zeros_like(t)


def _module_grads(m):
    """Gradients keyed like the reference's named_parameters() of the expert system."""
    out = {}
    for k, p in m.named_parameters():
        g = p.grad if p.grad is not None else torch.zeros_like(p)
        if k in m._STACKED:
            for e in range(g.shape[0]):
                out[f"experts.{e}.{m._STACKED[k]}"] = g[e]
        else:
            out[k] = g
    return out


@gpu
@pytest.mark.parametrize("E,K,act,Dm,I,B,L", [(1, 1, "gelu", 64, 128, 2, 256), (4, 4, "relu", 96, 160, 1, 1000),
                                               (16, 4, "silu", 704, 1408, 2, 1024), (32, 8, "gelu", 256, 512, 2, 512),
                                               (32, 8, "silu", 1688, 256, 1, 512)])
def test_moe_sublayer_fp32_vs_oracle(E, K, act, Dm, I, B, L):
    """AdaptiveExpertSystem alone, training with routing noise, the capacity limit and whole-expert dropout, fp32 inputs
    (the fp32-accurate GEMMs): routing and post-capacity counts bit for bit, output, aux losses, dx and every parameter
    gradient within the fp32 tolerance."""
    seed = E * 100 + K
    m, moe, active = _moe_module(E, K, act, Dm, I, seed)
    x, noise = O.make_inputs(B, L, Dm, E, seed=seed)
    m._draw_noise = lambda S, E_, device: noise.to(device)
    p = {k: v.clone().requires_grad_(True) for k, v in moe.items()}
    xr = x.clone().requires_grad_(True)
    out_r, lb_r, rz_r, parts = O.moe_forward(p, xr, E=E, K=K, act=act, training=True, noise=noise, active=active, return_parts=True)
    O.block_loss(out_r, lb_r, rz_r).backward()
    xg = x.to(dev()).requires_grad_(True)
    out, lb, rz = m(xg)
    O.block_loss(out, lb, rz).backward()
    torch.cuda.synchronize()
    idx_g, row_of = (t.cpu().numpy() for t in m.last_routing)
    assert np.array_equal(idx_g, parts["idx"].numpy()), "router indices"
    assert np.array_equal(row_of >= 0, parts["kept"]), "kept (token, slot) sets"
    assert np.array_equal(m.last_counts.cpu().numpy(), parts["counts"].astype(np.int32)), "expert_token_counts_post_capacity"
    tol = TOL[f32]
    assert rel_err(out, out_r.detach()) < tol, "out"
    assert abs(float(lb) - float(lb_r)) < tol * max(abs(float(lb_r)), 1e-3)
    assert abs(float(rz) - float(rz_r)) < tol * max(abs(float(rz_r)), 1e-3)
    assert rel_err(xg.grad, xr.grad) < tol, "dx"
    bad = [(k, e) for k, gr in _module_grads(m).items() if not (e := rel_err(gr, _grad(p[k]))) < tol]
    assert not bad, bad


@gpu
def test_moe_sublayer_bf16_autocast_rounded_routing_vs_oracle():
    """Under bf16 autocast with the router's logit rounding on (the default), against the oracle run under CUDA bf16
    autocast: both route on bf16-rounded logits.  The two differ in their bf16 arithmetic, so a few near-tied tokens route
    differently; the output and dx are compared on the identically routed tokens.  Measured on a B200 (all tokens routed
    identically): out 4.8e-3, dx 2.9e-3 (L2), parameter gradients at most 6.3e-3."""
    E, K, act, Dm, I, B, L = 16, 4, "silu", 704, 1408, 2, 1024
    S = B * L
    seed = 5
    m, moe, active = _moe_module(E, K, act, Dm, I, seed)
    assert m.router_autocast_rounding
    x, noise = O.make_inputs(B, L, Dm, E, seed=seed)
    d = dev()
    m._draw_noise = lambda S_, E_, device: noise.to(device)
    p = {k: v.to(d).requires_grad_(True) for k, v in moe.items()}
    xr = x.to(d).requires_grad_(True)
    with torch.autocast("cuda", dtype=torch.bfloat16):
        out_r, lb_r, rz_r, parts = O.moe_forward(p, xr, E=E, K=K, act=act, training=True, noise=noise.to(d), active=active,
                                                 return_parts=True)
    O.block_loss(out_r.float(), lb_r.float(), rz_r.float()).backward()
    xg = x.to(d).requires_grad_(True)
    with torch.autocast("cuda", dtype=torch.bfloat16):
        out, lb, rz = m(xg)
    O.block_loss(out.float(), lb.float(), rz.float()).backward()
    torch.cuda.synchronize()
    idx_g, row_of = (t.cpu().numpy() for t in m.last_routing)
    same = (idx_g == parts["idx"].cpu().numpy()).all(1) & ((row_of >= 0) == parts["kept"]).all(1)
    assert same.mean() > 0.97, f"routing agreement {same.mean():.4f}"
    same_t = torch.from_numpy(same)
    tol = TOL[bf16]
    o, o_r = out.float().reshape(S, Dm).cpu(), out_r.detach().float().reshape(S, Dm).cpu()
    assert rel_err(o[same_t], o_r[same_t]) < tol, "out (identically routed tokens)"
    assert abs(float(lb) - float(lb_r)) < tol * abs(float(lb_r))
    assert abs(float(rz) - float(rz_r)) < tol * abs(float(rz_r))
    counts = m.last_counts.cpu().numpy()
    assert int(counts.max()) <= parts["cap"] and abs(int(counts.sum()) - int(parts["counts"].sum())) <= 8
    dg, dr = xg.grad.reshape(S, Dm)[same_t.to(d)].double(), xr.grad.reshape(S, Dm)[same_t.to(d)].double()
    assert float((dg - dr).norm() / dr.norm()) < tol, "dx (identically routed tokens)"
    bad = [(k, e) for k, gr in _module_grads(m).items() if not (e := rel_err(gr, _grad(p[k]))) < tol]
    assert not bad, bad
