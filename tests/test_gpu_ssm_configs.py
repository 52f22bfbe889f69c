"""The SSM layer across the state sizes and conv widths SelectiveLinearAttention accepts (ssm_d_state 16 / 32 / 64,
ssm_conv_kernel 2..8).  The rounds scan picks its instance by heads per 64-channel slab (4 / 2 / 1) and the causal conv
by the conv width; every new instance is run here against a float64 reference of the same operation, and the layer and
the block end to end against the oracle."""
import math

import pytest
import torch
import torch.nn.functional as F

from oracle import apertis_oracle as O
from tests.util import rel_err

TOL = {torch.float32: 1e-4, torch.bfloat16: 2e-2}
f32, bf16 = torch.float32, torch.bfloat16
gpu = pytest.mark.gpu
EPS = 1e-12


def dev():
    return torch.device("cuda:0")


def _cfg(N, Kc, Dm=64, H=2, I=64, E=4, K=2, **kw):
    from apertis_llm_b200 import BlockConfig
    return BlockConfig(hidden_size=Dm, num_attention_heads=H, intermediate_size=I, num_experts=E, experts_per_token=K,
                       ssm_d_state=N, ssm_conv_kernel=Kc, hidden_dropout_prob=0.0, **kw)


# ------------------------------------------------------------------------------------------------
# host: which configurations construct, and with which parameters
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("N", [16, 32, 64])
@pytest.mark.parametrize("Kc", list(range(2, 9)))
def test_supported_configs_construct_with_reference_parameters(N, Kc):
    from apertis_llm_b200 import ApertisLayerB200
    layer = ApertisLayerB200(_cfg(N, Kc, H=3))
    ref = O.make_layer_params(64, 3, 64, 4, N=N, Kc=Kc)
    sd = layer.state_dict()
    assert set(sd) == set(ref)
    for k, v in ref.items():
        assert sd[k].shape == v.shape, k
    layer.load_state_dict(ref, strict=True)


@pytest.mark.parametrize("N", [8, 12, 24, 48, 128])
def test_unsupported_d_state_is_refused_at_construction(N):
    from apertis_llm_b200 import SelectiveLinearAttention
    with pytest.raises(NotImplementedError, match=r"ssm_d_state in \(16, 32, 64\)"):
        SelectiveLinearAttention(_cfg(N, 4))


@pytest.mark.parametrize("Kc", [1, 9])
def test_unsupported_conv_kernel_is_refused_at_construction(Kc):
    from apertis_llm_b200 import SelectiveLinearAttention
    with pytest.raises(NotImplementedError, match="ssm_conv_kernel in 2..8"):
        SelectiveLinearAttention(_cfg(16, Kc))


# ------------------------------------------------------------------------------------------------
# rounds scan at N = 32 / 64 against the float64 recurrent oracle
# ------------------------------------------------------------------------------------------------
def _scan_case(B, L, H, N, dtype, seed, h0=True):
    Di = N * H
    g = torch.Generator().manual_seed(seed)
    q = lambda t: t.to(dtype).float()
    return dict(xa=q(torch.randn(B, L, Di, generator=g)), z=q(torch.randn(B, L, Di, generator=g)),
                BC=q(torch.randn(B, L, 2 * Di, generator=g) * 0.5), dlog=q(torch.randn(B, L, H, generator=g) - 3.0),
                A_log=torch.rand(H, N, generator=g) * (math.log(0.99) - math.log(0.5)) + math.log(0.5),
                D=1.0 + 0.1 * torch.randn(Di, generator=g), h0=torch.randn(B, H, N, generator=g) if h0 else None,
                dy=q(torch.randn(B, L, Di, generator=g)), dys=q(torch.randn(B, L, Di, generator=g) * 0.3))


def _scan_oracle(c, heads=None, chunk=8192, want_yssm=True):
    """Outputs and gradients of scan + skip + gate from O.scan_recurrent in float64 for a subset of heads (independent
    chains), the time loop cut into chunks whose boundary state and its gradient are handed on explicitly."""
    B, L, Di = c["xa"].shape
    H, N = c["A_log"].shape
    hs = list(range(H)) if heads is None else list(heads)
    ch = torch.tensor([h * N + n for h in hs for n in range(N)])
    Hs = len(hs)
    sel = lambda t: t[..., ch].double()
    xa, z, dy, dys = sel(c["xa"]), sel(c["z"]), sel(c["dy"]), sel(c["dys"])
    Bm, Cm = sel(c["BC"][..., :Di]), sel(c["BC"][..., Di:])
    dlog = c["dlog"][..., hs].double()
    A_log, D = c["A_log"][hs].double(), c["D"][ch].double()
    h0 = c["h0"][:, hs].double() if c["h0"] is not None else torch.zeros(B, Hs, N, dtype=torch.float64)
    heads_of = lambda t, a, b: t[:, a:b].reshape(B, b - a, Hs, N).transpose(1, 2)
    bounds = list(range(0, L, chunk)) + [L]
    states, ys_all, y_all = [h0], [], []
    with torch.no_grad():
        for a, b in zip(bounds[:-1], bounds[1:]):
            delta = F.softplus(dlog[:, a:b]).transpose(1, 2).unsqueeze(-1)
            ys, hl = O.scan_recurrent(delta, A_log, heads_of(Bm, a, b), heads_of(Cm, a, b), states[-1])
            ys = ys.transpose(1, 2).reshape(B, b - a, Hs * N)
            ys_all.append(ys)
            y_all.append((ys + D * xa[:, a:b]) * F.silu(z[:, a:b]))
            states.append(hl)
    out = dict(y=torch.cat(y_all, 1), y_ssm=torch.cat(ys_all, 1), h_last=states[-1].reshape(B, Hs * N), ch=ch, hs=hs)
    g = {k: torch.zeros_like(v) for k, v in dict(xa=xa, z=z, Bm=Bm, Cm=Cm, dlog=dlog, A_log=A_log, D=D).items()}
    dh = torch.zeros_like(h0)
    for i in range(len(bounds) - 2, -1, -1):
        a, b = bounds[i], bounds[i + 1]
        lv = dict(xa=xa[:, a:b], z=z[:, a:b], Bm=Bm[:, a:b], Cm=Cm[:, a:b], dlog=dlog[:, a:b], A_log=A_log, D=D, h=states[i])
        lv = {k: v.detach().clone().requires_grad_(True) for k, v in lv.items()}
        delta = F.softplus(lv["dlog"]).transpose(1, 2).unsqueeze(-1)
        ys, hl = O.scan_recurrent(delta, lv["A_log"], heads_of(lv["Bm"], 0, b - a), heads_of(lv["Cm"], 0, b - a), lv["h"])
        ys = ys.transpose(1, 2).reshape(B, b - a, Hs * N)
        y = (ys + lv["D"] * lv["xa"]) * F.silu(lv["z"])
        loss = (y * dy[:, a:b]).sum() + (hl * dh).sum()
        if want_yssm:
            loss = loss + (ys * dys[:, a:b]).sum()
        loss.backward()
        for k in ("xa", "z", "Bm", "Cm", "dlog"):
            g[k][:, a:b] = lv[k].grad
        g["A_log"] += lv["A_log"].grad
        g["D"] += lv["D"].grad
        dh = lv["h"].grad
    out["grads"] = g
    return out


def _scan_gpu(c, dtype, fused, want_yssm=True, dt_bias=None):
    """fused: the layout ssm_core uses - xa / z as column slices of one [xa | z] buffer, [dt (no bias) | pad | B | C] as
    one buffer, the dt bias applied inside the kernel; otherwise separate contiguous tensors."""
    from apertis_llm_b200 import ops
    B, L, Di = c["xa"].shape
    H = c["dlog"].shape[-1]
    d = dev()
    A_log = c["A_log"].to(d).requires_grad_(True)
    D = c["D"].to(d).requires_grad_(True)
    h0 = c["h0"].to(d) if c["h0"] is not None else None
    bias = dt_bias.to(d).requires_grad_(True) if dt_bias is not None else None
    dl_in = c["dlog"] - (dt_bias if dt_bias is not None else 0.0)
    if fused:
        xz = torch.cat([c["xa"], c["z"]], dim=-1).to(d, dtype).requires_grad_(True)
        xa, z = xz[..., :Di], xz[..., Di:]
        Hp = (H + 7) // 8 * 8
        prm = torch.cat([dl_in, torch.full((B, L, Hp - H), 7.0), c["BC"]], dim=-1).to(d, dtype).requires_grad_(True)
        y, ys, hl = ops.selective_scan_fused(xa, prm, bias, z, A_log, D, H, h0=h0, want_yssm=want_yssm, want_hlast=True)
    else:
        xa, z = c["xa"].to(d, dtype).requires_grad_(True), c["z"].to(d, dtype).requires_grad_(True)
        dlog = dl_in.to(d, dtype).requires_grad_(True)
        BC = c["BC"].to(d, dtype).requires_grad_(True)
        y, ys, hl = ops._SelectiveScanRounds.apply(xa, dlog, bias, BC, z, A_log, D, h0, want_yssm, True, H)
    outs, gos = [y], [c["dy"].to(d, dtype)]
    if want_yssm:
        outs.append(ys)
        gos.append(c["dys"].to(d, dtype))
    torch.autograd.backward(outs, gos)
    torch.cuda.synchronize()
    r = dict(y=y.detach().float().cpu(), y_ssm=ys.detach().float().cpu() if want_yssm else None, h_last=hl.cpu(),
             dA_log=A_log.grad.cpu(), dD=D.grad.cpu())
    if fused:
        r["dxa"], r["dz"] = xz.grad[..., :Di].float().cpu(), xz.grad[..., Di:].float().cpu()
        gp = prm.grad.float().cpu()
        r["ddlog"], r["dpad"], r["dBC"] = gp[..., :H], gp[..., H:Hp], gp[..., Hp:]
    else:
        r["dxa"], r["dz"] = xa.grad.float().cpu(), z.grad.float().cpu()
        r["ddlog"], r["dBC"] = dlog.grad.float().cpu(), BC.grad.float().cpu()
    if bias is not None:
        r["dbias"] = bias.grad.cpu()
    return r


def _scan_compare(r, o, dtype, want_yssm=True):
    tol = TOL[dtype]
    ch, hs = o["ch"], o["hs"]
    Di = r["y"].shape[-1]
    red = max(tol, 2e-3) if dtype == bf16 else tol         # reductions over all tokens of bf16-rounded terms
    g = o["grads"]
    checks = [("y", r["y"][..., ch], o["y"], tol), ("h_last", r["h_last"][..., ch], o["h_last"], tol),
              ("dxa", r["dxa"][..., ch], g["xa"], tol), ("dz", r["dz"][..., ch], g["z"], tol),
              ("dB", r["dBC"][..., :Di][..., ch], g["Bm"], tol), ("dC", r["dBC"][..., Di:][..., ch], g["Cm"], tol),
              ("ddlog", r["ddlog"][..., hs], g["dlog"], red), ("dA_log", r["dA_log"][hs], g["A_log"], red),
              ("dD", r["dD"][ch], g["D"], red)]
    if want_yssm:
        checks.append(("y_ssm", r["y_ssm"][..., ch], o["y_ssm"], tol))
    if "dbias" in r:
        checks.append(("d dt_bias", r["dbias"][hs], g["dlog"].sum((0, 1)), red))
    bad = [(n, rel_err(a, b)) for n, a, b, t in checks if not rel_err(a, b) < t]
    assert not bad, bad


# (N, B, L, H): odd head counts leave a tail slab (N = 32: one head in the last slab; N = 64: any H)
SCAN_CASES = [
    (32, 1, 5, 3), (32, 3, 333, 5), (32, 1, 4096, 4), (32, 2, 1, 3), (32, 1, 777, 11),
    (64, 1, 5, 2), (64, 3, 333, 3), (64, 1, 4096, 8), (64, 2, 1, 1), (64, 2, 600, 7),
]


@gpu
@pytest.mark.parametrize("dtype", [f32, bf16], ids=["f32", "bf16"])
@pytest.mark.parametrize("N,B,L,H", SCAN_CASES)
def test_rounds_scan_d_state_vs_oracle(N, B, L, H, dtype):
    """Fused strided layout with h0 and the dt bias inside the kernel (padding columns of d dt must come back zero), then
    the split layout without h0; both against float64, and the fused launch bitwise repeatable."""
    c = _scan_case(B, L, H, N, dtype, seed=N + L + H)
    bias = torch.rand(H, generator=torch.Generator().manual_seed(H)) * 2 - 5
    o = _scan_oracle(c)
    r = _scan_gpu(c, dtype, fused=True, dt_bias=bias)
    _scan_compare(r, o, dtype)
    assert not r["dpad"].any(), "padding columns of d dt"
    r2 = _scan_gpu(c, dtype, fused=True, dt_bias=bias)
    for k in ("y", "y_ssm", "h_last", "dxa", "dz", "dBC", "ddlog", "dpad", "dA_log", "dD", "dbias"):
        assert torch.equal(r[k], r2[k]), f"{k}: not bitwise repeatable"
    c = _scan_case(B, L, H, N, dtype, seed=N + L + H, h0=False)
    _scan_compare(_scan_gpu(c, dtype, fused=False), _scan_oracle(c), dtype)


@gpu
@pytest.mark.parametrize("N,H,heads", [(32, 4, (0, 3)), (64, 3, (1,))])
def test_rounds_scan_d_state_long_sequence(N, H, heads):
    """L = 65536 (many rounds, both prefix levels), bf16, against the oracle on a subset of heads."""
    c = _scan_case(1, 65536, H, N, bf16, seed=7 + N, h0=False)
    o = _scan_oracle(c, heads=heads, want_yssm=False)
    r = _scan_gpu(c, bf16, fused=True, want_yssm=False)
    _scan_compare(r, o, bf16, want_yssm=False)


# ------------------------------------------------------------------------------------------------
# causal conv + SiLU for every conv width against float64
# ------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("dtype", [f32, bf16], ids=["f32", "bf16"])
@pytest.mark.parametrize("Kc", list(range(2, 9)))
def test_causal_conv_widths_vs_float64(Kc, dtype):
    from apertis_llm_b200 import ops
    g = torch.Generator().manual_seed(Kc)
    for B, L, Di in ((2, 300, 96), (1, Kc - 1, 64), (3, 1, 32), (1, 2000, 176)):
        w = (torch.rand(Di, 1, Kc, generator=g) - 0.5)
        b = (torch.rand(Di, generator=g) - 0.5)
        # xp as the first half of a [xp | z] row (row stride 2 Di), the way the in-projection output is consumed
        buf = torch.randn(B, L, 2 * Di, generator=g).to(dtype)
        dout = torch.randn(B, L, Di, generator=g).to(dtype)
        xb = buf.to(dev()).requires_grad_(True)
        wg, bg = w.to(dev()).requires_grad_(True), b.to(dev()).requires_grad_(True)
        xa = ops.causal_conv1d_silu(xb[..., :Di], wg, bg)
        xa.backward(dout.to(dev()))
        torch.cuda.synchronize()
        xr = buf[..., :Di].double().requires_grad_(True)
        wr, br = w.double().requires_grad_(True), b.double().requires_grad_(True)
        ref = F.silu(F.conv1d(xr.transpose(1, 2), wr, br, padding=Kc - 1, groups=Di)[:, :, :L]).transpose(1, 2)
        ref.backward(dout.double())
        tol = TOL[dtype]
        case = (Kc, B, L, Di)
        assert rel_err(xa.float().cpu(), ref.detach()) < tol, ("xa", case)
        assert rel_err(xb.grad[..., :Di].float().cpu(), xr.grad) < tol, ("dxp", case)
        assert float(xb.grad[..., Di:].abs().max()) == 0.0, ("z columns", case)
        assert rel_err(wg.grad.cpu(), wr.grad) < tol, ("dw", case)
        assert rel_err(bg.grad.cpu(), br.grad) < tol, ("dbias", case)


# ------------------------------------------------------------------------------------------------
# SelectiveLinearAttention and ApertisLayerB200 against the oracle
# ------------------------------------------------------------------------------------------------
MODULE_CONFIGS = [(32, 3), (64, 2), (16, 8), (64, 4), (32, 6)]
Dm, H_MOD, I_MOD, E_MOD, K_MOD = 128, 3, 256, 4, 2


def _ssm_pair(N, Kc, seed):
    from apertis_llm_b200 import SelectiveLinearAttention
    sd = O.make_layer_params(Dm, H_MOD, I_MOD, E_MOD, N=N, Kc=Kc, seed=seed)
    ssm_sd, _, _ = O.split_layer_params(sd)
    m = SelectiveLinearAttention(_cfg(N, Kc, Dm=Dm, H=H_MOD, I=I_MOD, E=E_MOD))
    m.load_state_dict(ssm_sd, strict=True)
    return m.to(dev()), {k: v.clone().requires_grad_(True) for k, v in ssm_sd.items()}


def _grads_match(m, ref, tol, what):
    bad = []
    for k, p in m.named_parameters():
        e = rel_err(p.grad.float().cpu(), ref[k].grad)
        if not e < tol:
            bad.append((k, e))
    assert not bad, (what, bad)


@gpu
@pytest.mark.parametrize("N,Kc", MODULE_CONFIGS)
def test_ssm_layer_train_eval_vs_oracle(N, Kc):
    B, L = 2, 96
    x, _ = O.make_inputs(B, L, Dm, E_MOD, seed=N + Kc)
    for output_attentions in (False, True):
        m, ref = _ssm_pair(N, Kc, seed=Kc)
        m.train()
        xg = x.to(dev()).requires_grad_(True)
        out, y, _ = m(xg, output_attentions=output_attentions)
        xr = x.clone().requires_grad_(True)
        out_r, y_r, _ = O.ssm_forward(ref, xr, num_heads=H_MOD, d_state=N, training=True)
        loss = out.pow(2).mean() + (y.pow(2).mean() if output_attentions else 0.0)
        loss_r = out_r.pow(2).mean() + (y_r.pow(2).mean() if output_attentions else 0.0)
        loss.backward()
        loss_r.backward()
        assert rel_err(out.cpu(), out_r.detach()) < 1e-4, ("out", output_attentions)
        if output_attentions:
            assert rel_err(y.cpu(), y_r.detach()) < 1e-4, "y_ssm"
        assert rel_err(xg.grad.cpu(), xr.grad) < 1e-4, ("dx", output_attentions)
        _grads_match(m, ref, 1e-4, ("fp32 train", output_attentions))
    # bf16 autocast over fp32 masters: the fused training path against the fp32 oracle
    m, ref = _ssm_pair(N, Kc, seed=Kc)
    m.train()
    xg = x.to(dev()).requires_grad_(True)
    with torch.autocast("cuda", dtype=torch.bfloat16):
        out, _, _ = m(xg)
    out.float().pow(2).mean().backward()
    xr = x.clone().requires_grad_(True)
    out_r, _, _ = O.ssm_forward(ref, xr, num_heads=H_MOD, d_state=N, training=True)
    out_r.pow(2).mean().backward()
    assert rel_err(out.float().cpu(), out_r.detach()) < 2e-2, "bf16 out"
    assert rel_err(xg.grad.float().cpu(), xr.grad) < 2e-2, "bf16 dx"
    _grads_match(m, ref, 2e-2, "bf16 autocast")
    # evaluation: recurrent scan, y_ssm
    m.eval()
    with torch.no_grad():
        out, y, _ = m(x.to(dev()), output_attentions=True)
        out_r, y_r, _ = O.ssm_forward({k: v.detach() for k, v in ref.items()}, x, num_heads=H_MOD, d_state=N, training=False)
    assert rel_err(out.cpu(), out_r) < 1e-4 and rel_err(y.cpu(), y_r) < 1e-4, "eval"


@gpu
@pytest.mark.parametrize("N,Kc", MODULE_CONFIGS)
def test_ssm_layer_cached_decode_vs_oracle(N, Kc):
    """Prefill, then 8 single tokens with the (conv_state [B, Di, Kc-1], ssm_state [B, H, N]) cache, including the
    reference's cached-conv quirk (core.py:369-373: the state goes in front, the first L outputs are kept)."""
    B, L, steps = 2, 16, 8
    m, ref = _ssm_pair(N, Kc, seed=3 * Kc)
    m.eval()
    ref = {k: v.detach() for k, v in ref.items()}
    x, _ = O.make_inputs(B, L + steps, Dm, E_MOD, seed=N * Kc)
    xd = x.to(dev())
    with torch.no_grad():
        out, y, cache = m(xd[:, :L], output_attentions=True, use_cache=True)
        out_r, y_r, cache_r = O.ssm_forward(ref, x[:, :L], num_heads=H_MOD, d_state=N, training=False, use_cache=True)
        assert cache[0].shape == (B, N * H_MOD, Kc - 1) and cache[1].shape == (B, H_MOD, N)
        for s in range(steps + 1):
            assert rel_err(out.cpu(), out_r) < 1e-4 and rel_err(y.cpu(), y_r) < 1e-4, ("out", s)
            assert rel_err(cache[0].cpu(), cache_r[0]) < 1e-5 and rel_err(cache[1].cpu(), cache_r[1]) < 1e-4, ("cache", s)
            if s == steps:
                break
            t = L + s
            out, y, cache = m(xd[:, t:t + 1], past_key_value=cache, output_attentions=True, use_cache=True)
            out_r, y_r, cache_r = O.ssm_forward(ref, x[:, t:t + 1], num_heads=H_MOD, d_state=N, training=False, use_cache=True,
                                                past=cache_r)


@gpu
@pytest.mark.parametrize("N", [32, 64])
def test_older_scan_schedules_refuse_d_state_above_16(N):
    """scan_mode 0 / 1 / 2 select the single-pass, two-pass and pipelined schedules, which hold ssm_d_state 16 only."""
    m, _ = _ssm_pair(N, 4, seed=0)
    x = torch.randn(1, 32, Dm, device=dev())
    for mode in (0, 1, 2):
        m.scan_mode = mode
        with pytest.raises(RuntimeError, match=r"Di == 16\*H"):
            m(x)


def _block_ref(sd, x, N, noise):
    """ApertisLayer.forward (core.py:1005-1018) with dropout 0 from the oracle's SSM and MoE functions at state size N."""
    ssm, moe, norms = O.split_layer_params(sd)
    n1 = F.layer_norm(x, (Dm,), norms["attention.pre_norm.weight"], norms["attention.pre_norm.bias"], EPS)
    a, _, _ = O.ssm_forward(ssm, n1, num_heads=H_MOD, d_state=N, training=True)
    h = a + x
    n2 = F.layer_norm(h, (Dm,), norms["feed_forward.pre_norm.weight"], norms["feed_forward.pre_norm.bias"], EPS)
    m, lb, rz = O.moe_forward(moe, n2, E=E_MOD, K=K_MOD, eps=EPS, training=True, noise=noise)
    return m + h, lb, rz


@gpu
@pytest.mark.parametrize("N,Kc", MODULE_CONFIGS)
def test_block_d_state_conv_kernel_vs_oracle(N, Kc):
    from apertis_llm_b200 import ApertisLayerB200
    from tests.test_gpu_modules import named_grads
    B, L = 2, 64
    sd = O.make_layer_params(Dm, H_MOD, I_MOD, E_MOD, N=N, Kc=Kc, seed=N + Kc)
    layer = ApertisLayerB200(_cfg(N, Kc, Dm=Dm, H=H_MOD, I=I_MOD, E=E_MOD, K=K_MOD))
    layer.load_state_dict(sd, strict=True)
    layer.feed_forward.ffn.router_autocast_rounding = False      # the fp32 oracle routes on fp32 logits
    layer = layer.to(dev()).train()
    x, noise = O.make_inputs(B, L, Dm, E_MOD, seed=Kc)
    layer.feed_forward.ffn._draw_noise = lambda S, E, device: noise.to(device)
    sdr = {k: v.clone().requires_grad_(True) for k, v in sd.items()}
    xr = x.clone().requires_grad_(True)
    out_r, lb_r, rz_r = _block_ref(sdr, xr, N, noise)
    O.block_loss(out_r, lb_r, rz_r).backward()
    xg = x.to(dev()).requires_grad_(True)
    out, _, _, lb, rz = layer(xg)
    O.block_loss(out, lb, rz).backward()
    assert rel_err(out.cpu(), out_r.detach()) < 1e-4
    assert abs(float(lb) - float(lb_r)) <= 1e-4 * abs(float(lb_r)) and abs(float(rz) - float(rz_r)) <= 1e-4 * abs(float(rz_r))
    assert rel_err(xg.grad.cpu(), xr.grad) < 1e-4
    bad = [(k, rel_err(g.cpu(), sdr[k].grad)) for k, g in named_grads(layer).items() if not rel_err(g.cpu(), sdr[k].grad) < 1e-4]
    assert not bad, bad


# ------------------------------------------------------------------------------------------------
# live reference: an unmodified ApertisForCausalLM at ssm_d_state 32, ssm_conv_kernel 3
# ------------------------------------------------------------------------------------------------
@gpu
def test_patched_causal_lm_d_state_32_conv_kernel_3_vs_reference():
    import copy

    from baseline import ref_loader
    if not ref_loader.available():
        pytest.skip("baseline/_ref (the installed reference) is absent")
    import apertis_llm_b200 as ab
    from tests.test_gpu_reference_model import compare_models, text_batch
    core = ref_loader.load_core()
    cfg = core.ApertisConfig(hidden_size=128, num_attention_heads=2, intermediate_size=256, num_hidden_layers=2,
                             attention_type="selective_ssm", use_expert_system=True, num_experts=4, experts_per_token=2,
                             vocab_size=211, hidden_dropout_prob=0.0, attention_probs_dropout_prob=0.0,
                             use_noisy_top_k_routing=False, ssm_d_state=32, ssm_conv_kernel=3)
    torch.manual_seed(0)
    ref = core.ApertisForCausalLM(cfg).to(dev())
    g = torch.Generator(device="cpu").manual_seed(1)
    with torch.no_grad():
        for p in ref.parameters():
            if p.dim() == 1:
                p.add_(0.05 * torch.randn(p.shape, generator=g).to(p.device))
    mine = ab.patch_apertis_model(copy.deepcopy(ref))
    assert mine.model.layers[0].attention.attention_mechanism_impl.A_log.shape == (2, 32)
    ref.train(); mine.train()
    compare_models(ref, mine, text_batch(), 1e-4)
    ref.eval(); mine.eval()
    ids = text_batch(B=1, L=24)["input_ids"]
    with torch.no_grad():
        t_r = ref.generate(input_ids=ids, max_new_tokens=6, do_sample=False)
        t_m = mine.generate(input_ids=ids, max_new_tokens=6, do_sample=False)
    assert torch.equal(t_r, t_m), (t_r.tolist(), t_m.tolist())
