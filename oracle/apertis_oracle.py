"""CPU oracle for the Apertis SSM+MoE block hot path.

TEST INFRASTRUCTURE ONLY.  Nothing under ``apertis_llm_b200/`` may import this
module; only ``tests/``, ``__graft_entry__.smoke()`` and the ``cpu_baseline`` /
``--impl reference`` legs of ``bench.py`` do, and only as the checker / the CPU
baseline, never as the thing shipped.

It is a functional restatement (plain torch CPU ops on explicit parameter
dictionaries, plus numpy integer code for the routing plan) of the reference's
algorithm in ``/root/reference/src/model/core.py``:

* ``SelectiveLinearAttention``   core.py:295-401
* ``AdaptiveExpertSystem``       core.py:403-607
* the callers that bracket them  core.py:690-704, 836-838, 886-923, 1005-1018

Parity status: **pinned**.  The reference's own test-suite holds no golden
vector for this path (SURVEY.md section 4), so the oracle is pinned against outputs
of the unmodified reference modules executed in the build container
(``tests/golden/make_golden.py`` imports ``/root/reference`` and writes the
fixtures under ``tests/golden/``; ``tests/test_oracle_golden.py`` checks every
function here against them).

Parameter dictionaries use the reference's ``state_dict`` key names relative to
the module (``in_proj_x.weight`` ... / ``router.weight``, ``experts.0.1.weight`` ...).
Gradients come from torch autograd over these ops.
"""
from __future__ import annotations

import math
from typing import Dict, Optional, Tuple

import numpy as np
import torch
import torch.nn.functional as F

Tensor = torch.Tensor
Params = Dict[str, Tensor]


# --------------------------------------------------------------------------
# shape bookkeeping (core.py:151-167, 298-304)
# --------------------------------------------------------------------------
def ssm_dims(hidden_size: int, num_heads: int, d_state: int = 16,
             dt_rank: Optional[int] = None, conv_kernel: int = 4) -> dict:
    """Derived sizes of the SSM layer: d_inner = heads*d_state (core.py:154),
    dt_rank = ceil(hidden/16) (core.py:164)."""
    return dict(Dm=hidden_size, H=num_heads, N=d_state, Di=num_heads * d_state,
                R=dt_rank if dt_rank is not None else math.ceil(hidden_size / 16),
                Kc=conv_kernel)


# --------------------------------------------------------------------------
# selective scan, two formulations
# --------------------------------------------------------------------------
def scan_logcumsum(delta: Tensor, A_log: Tensor, Bt: Tensor, Ct: Tensor) -> Tensor:
    """Training-mode scan exactly as the reference writes it (core.py:324-335):
    P = exp(cumsum(log(abar + 1e-38))); h = P * cumsum(B / (P + 1e-38)); y = C * h.
    delta [B,H,L,1]; A_log [H,N]; Bt, Ct [B,H,L,N] -> y [B,H,L,N].
    Known to overflow to NaN for L >= 16384 (SURVEY.md section 5)."""
    A = -torch.exp(A_log)                                     # :326
    abar = torch.exp(delta * A[None, :, None, :])             # :327
    lp = torch.cumsum(torch.log(abar + 1e-38), dim=2)         # :328-329
    P = torch.exp(lp)                                         # :330
    acc = torch.cumsum(Bt / (P + 1e-38), dim=2)               # :331-332
    return Ct * (P * acc)                                     # :333-334


def scan_recurrent(delta: Tensor, A_log: Tensor, Bt: Tensor, Ct: Tensor,
                   h0: Optional[Tensor] = None) -> Tuple[Tensor, Tensor]:
    """Eval / cached scan (core.py:337-353): h_t = abar_t*h_{t-1} + B_t, y_t = C_t*h_t.
    Returns (y [B,H,L,N], h_last [B,H,N])."""
    A = -torch.exp(A_log)                                     # :339
    abar = torch.exp(delta * A[None, :, None, :])             # :340-341
    Bsz, H, L, N = Bt.shape
    h = h0 if h0 is not None else torch.zeros(Bsz, H, N, dtype=Bt.dtype)
    ys = []
    # same per-step arithmetic as the reference's indexing (abar[:, :, t, :] ...); unbind() hands autograd one
    # backward node per tensor instead of one zero-filled [B,H,L,N] gradient per step, which is what makes the
    # L >= 16K parity cases (SURVEY.md 8c caveat 1) tractable on the CPU
    a_t, b_t, c_t = abar.unbind(2), Bt.unbind(2), Ct.unbind(2)
    for t in range(L):                                        # :347
        h = a_t[t] * h + b_t[t]
        ys.append(c_t[t] * h)
    return torch.stack(ys, dim=2), h


# --------------------------------------------------------------------------
# SSM layer (SelectiveLinearAttention.forward, core.py:355-401)
# --------------------------------------------------------------------------
def ssm_forward(p: Params, x: Tensor, *, num_heads: int, d_state: int = 16,
                training: bool = True, use_cache: bool = False,
                past: Optional[Tuple[Tensor, Tensor]] = None,
                scan: Optional[str] = None, return_parts: bool = False):
    """x [B,L,Dm] -> (out [B,L,Dm], y_ssm [B,L,Di], cache|None).

    ``scan`` = "logcumsum" | "recurrent"; default follows the reference's mode
    switch (core.py:388-393): logcumsum when training and not use_cache.
    The cached-conv quirk of core.py:369-373 (the state is concatenated in front
    and the conv output truncated to the first L columns) is reproduced as is."""
    Bsz, L, _ = x.shape
    H, N = num_heads, d_state
    Di = H * N
    Kc = p["conv1d.weight"].shape[-1]
    R = p["dt_proj_head.weight"].shape[1]
    xp = F.linear(x, p["in_proj_x.weight"])                   # :366
    z = F.linear(x, p["in_proj_z.weight"])                    # :367
    xc_in = xp.transpose(1, 2)                                # :368
    conv_prev, h_prev = (past if past is not None else (None, None))
    if conv_prev is not None and use_cache:                   # :369-371
        if conv_prev.shape[1] == Di and conv_prev.shape[2] == Kc - 1:
            xc_in = torch.cat([conv_prev, xc_in], dim=2)
    conv_state = xc_in[:, :, -(Kc - 1):].detach() if use_cache else None   # :372
    xc = F.conv1d(xc_in, p["conv1d.weight"], p["conv1d.bias"],
                  padding=Kc - 1, groups=Di)[:, :, :L].transpose(1, 2)      # :373-374
    xa = F.silu(xc)                                           # :375
    prm = F.linear(xa, p["x_param_proj.weight"])              # :376
    dtf, Braw, Craw = torch.split(prm, [R, Di, Di], dim=-1)   # :377-381
    dlog = F.linear(dtf, p["dt_proj_head.weight"], p["dt_proj_head.bias"])  # :382
    delta = F.softplus(dlog).transpose(1, 2).unsqueeze(-1)    # :383
    Bt = Braw.view(Bsz, L, H, N).transpose(1, 2)              # :384
    Ct = Craw.view(Bsz, L, H, N).transpose(1, 2)              # :385
    if scan is None:
        scan = "logcumsum" if (training and not use_cache) else "recurrent"
    h_last = None
    if scan == "logcumsum":
        y = scan_logcumsum(delta, p["A_log"], Bt, Ct)         # :389
    else:
        y, h_last = scan_recurrent(delta, p["A_log"], Bt, Ct,
                                   h_prev if use_cache else None)           # :391
    y_ssm = y.transpose(1, 2).contiguous().view(Bsz, L, Di)   # :394
    gated = (y_ssm + p["D"][None, None, :] * xa) * F.silu(z)  # :395-396
    out = F.linear(gated, p["out_proj.weight"])               # :397
    cache = (conv_state, h_last.detach()) if use_cache else None            # :398-400
    if return_parts:
        return out, y_ssm, cache, dict(xp=xp, z=z, xa=xa, dlog=dlog, Braw=Braw, Craw=Craw, gated=gated)
    return out, y_ssm, cache


# --------------------------------------------------------------------------
# MoE routing: integer-exact plan (core.py:547-590) in numpy
# --------------------------------------------------------------------------
def moe_capacity(S: int, E: int, factor: float = 1.25, training: bool = True,
                 use_limit: bool = True) -> int:
    """core.py:508-511."""
    if use_limit and training and E > 0:
        return max(1, math.floor((S / E) * factor)) if S > 0 else 0
    return S


def moe_plan(idx: np.ndarray, w: np.ndarray, E: int, cap: int,
             active: Optional[np.ndarray] = None, limit: bool = True):
    """Replays the dispatch rule of core.py:547-590 on host integers.

    idx [S,K] int (expert chosen per slot), w [S,K] float32 (normalised gate
    weights).  Order: slot k outer, expert e inner; an expert keeps at most
    ``cap`` rows summed over slots; on overflow of a (k,e) group the rows with
    the largest w[:,k] are kept (core.py:578-582).  Tie policy (the reference's
    torch.topk leaves it unspecified): equal weights -> lower token index first.

    Returns kept [S,K] bool, counts [E] int64, groups {(k,e): kept token ids ascending}."""
    S, K = idx.shape
    kept = np.zeros((S, K), dtype=bool)
    counts = np.zeros(E, dtype=np.int64)
    groups = {}
    for k in range(K):
        for e in range(E):
            if active is not None and not bool(active[e]):
                continue
            cand = np.nonzero(idx[:, k] == e)[0]
            if cand.size == 0:
                continue
            n_take = cand.size
            if limit:
                rem = cap - int(counts[e])
                if rem <= 0:
                    continue
                n_take = min(cand.size, rem)
            if n_take < cand.size:
                # stable sort on -w keeps lower token ids first among equal weights
                order = np.argsort(-w[cand, k].astype(np.float64), kind="stable")
                take = np.sort(cand[order[:n_take]])
            else:
                take = cand
            if take.size == 0:
                continue
            counts[e] += take.size
            kept[take, k] = True
            groups[(k, e)] = take
    return kept, counts, groups


def topk_lowest_index(g: np.ndarray, K: int) -> Tuple[np.ndarray, np.ndarray]:
    """Top-K along the last axis, descending, ties -> lower index first (the tie
    policy the CUDA router defines; torch.topk's is unspecified)."""
    order = np.argsort(-g.astype(np.float64), axis=-1, kind="stable")[:, :K]
    return np.take_along_axis(g, order, axis=-1), order


# --------------------------------------------------------------------------
# MoE layer (AdaptiveExpertSystem.forward, core.py:470-607)
# --------------------------------------------------------------------------
def _act(name: str):
    """core.py:463-468."""
    if name == "relu":
        return F.relu
    if name in ("silu", "swish"):
        return F.silu
    return F.gelu


def moe_router(p: Params, x2: Tensor, *, eps: float, noise: Optional[Tensor],
               alpha: float, K: int):
    """core.py:480-492, 529.  x2 [S,Dm] -> logits, gates [S,E], probs/idx [S,K], w [S,K]."""
    xn = F.layer_norm(x2, (x2.shape[-1],), p["router_norm.weight"], p["router_norm.bias"], eps)
    logits = F.linear(xn, p["router.weight"], p["router.bias"]).float()     # :482
    if noise is not None:                                                   # :485-488
        logits = logits + noise * (F.softplus(p["w_noise"]) * alpha).unsqueeze(0)
    gates = F.softmax(logits, dim=-1)                                       # :491
    probs, idx = torch.topk(gates, K, dim=-1)                               # :492
    w = probs / (probs.sum(dim=-1, keepdim=True) + 1e-6)                    # :529
    return logits, gates, probs, idx, w


def moe_forward(p: Params, x: Tensor, *, E: int, K: int, eps: float = 1e-12,
                act: str = "gelu", training: bool = True,
                noise: Optional[Tensor] = None, alpha: float = 0.1,
                lb_coef: float = 0.01, rz_coef: float = 0.001,
                cap_factor: float = 1.25, use_capacity: bool = True,
                active: Optional[np.ndarray] = None, return_parts: bool = False):
    """x [B,L,Dm] -> (out [B,L,Dm], lb_loss, rz_loss).

    ``noise`` [S,E] is the standard-normal draw of core.py:487 (pass None for
    eval or when noisy routing is off); the caller owns the RNG so that both
    sides of a parity test consume the same numbers.  ``active`` is the
    whole-expert dropout mask of core.py:514-521 (None = all active; with the
    default E=8, p=0.1 the reference drops floor(0.8)=0 experts).
    Expert-internal Dropout (core.py:439) is not modelled: parity runs use
    hidden_dropout_prob = 0."""
    Bsz, L, Dm = x.shape
    S = Bsz * L
    x2 = x.reshape(S, Dm)                                                   # :480
    logits, gates, probs, idx, w = moe_router(p, x2, eps=eps, noise=noise if training else None,
                                              alpha=alpha, K=K)
    lb = torch.zeros((), dtype=x.dtype)
    rz = torch.zeros((), dtype=x.dtype)
    if training and lb_coef > 0:                                            # :499-505
        P_i = gates.mean(dim=0)
        onehot = torch.zeros_like(gates).scatter_(1, idx, 1.0)
        f_i = onehot.mean(dim=0)
        lb = lb_coef * E * torch.sum(f_i * P_i)
    cap = moe_capacity(S, E, cap_factor, training, use_capacity)            # :508-511
    if training and rz_coef > 0:                                            # :524-526
        rz = rz_coef * torch.mean(torch.logsumexp(logits, dim=-1) ** 2)
    kept, counts, groups = moe_plan(idx.cpu().numpy(), w.detach().cpu().numpy(), E, cap, active,
                                    limit=(use_capacity and training))
    out = torch.zeros_like(x2)                                              # :531
    fn = _act(act)
    for k in range(K):                                                      # :547
        for e in range(E):                                                  # :551
            take = groups.get((k, e))
            if take is None:
                continue
            rows = torch.from_numpy(take).to(x2.device)
            xe = x2[rows]                                                   # :593
            h = F.layer_norm(xe, (Dm,), p[f"experts.{e}.0.weight"], p[f"experts.{e}.0.bias"], eps)
            h = fn(F.linear(h, p[f"experts.{e}.1.weight"], p[f"experts.{e}.1.bias"]))
            y = F.linear(h, p[f"experts.{e}.4.weight"], p[f"experts.{e}.4.bias"])  # :596
            out = out.index_add(0, rows, y * w[rows, k].unsqueeze(1))       # :605
    res = (out.reshape(Bsz, L, Dm), lb, rz)
    if return_parts:
        return res + (dict(logits=logits, gates=gates, idx=idx, w=w, kept=kept, counts=counts, cap=cap),)
    return res


# --------------------------------------------------------------------------
# the block (ApertisAttention / ApertisFeedForward / ApertisLayer)
# --------------------------------------------------------------------------
def split_layer_params(sd: Params):
    """Splits an ``ApertisLayer`` state_dict into (ssm, moe, norms)."""
    a = "attention.attention_mechanism_impl."
    f = "feed_forward.ffn."
    ssm = {k[len(a):]: v for k, v in sd.items() if k.startswith(a)}
    moe = {k[len(f):]: v for k, v in sd.items() if k.startswith(f)}
    norms = {k: v for k, v in sd.items() if ".pre_norm." in k}
    return ssm, moe, norms


def block_forward(sd: Params, x: Tensor, *, num_heads: int, E: int, K: int,
                  eps: float = 1e-12, training: bool = True, noise: Optional[Tensor] = None,
                  scan: Optional[str] = None, **moe_kw):
    """ApertisLayer.forward (core.py:1005-1018) with dropout p = 0:
    h = x + SSM(LN(x)) (core.py:694-704, 836-837); out = h + MoE(LN(h)) (core.py:887-919)."""
    ssm, moe, norms = split_layer_params(sd)
    Dm = x.shape[-1]
    n1 = F.layer_norm(x, (Dm,), norms["attention.pre_norm.weight"], norms["attention.pre_norm.bias"], eps)
    a, _, _ = ssm_forward(ssm, n1, num_heads=num_heads, training=training, scan=scan)
    h = a + x
    n2 = F.layer_norm(h, (Dm,), norms["feed_forward.pre_norm.weight"], norms["feed_forward.pre_norm.bias"], eps)
    m, lb, rz = moe_forward(moe, n2, E=E, K=K, eps=eps, training=training, noise=noise, **moe_kw)
    return m + h, lb, rz


# --------------------------------------------------------------------------
# deterministic parameter / input factory shared by fixtures, tests and bench
# --------------------------------------------------------------------------
def make_layer_params(Dm: int, H: int, I: int, E: int, *, seed: int = 0, N: int = 16, Kc: int = 4,
                      dtype=torch.float32, perturb: bool = True) -> Params:
    """An ``ApertisLayer`` state_dict drawn from a seeded CPU generator.

    Follows the reference initialiser's distributions (Linear ~ N(0, 0.02), LayerNorm
    1/0, A_log ~ U(log .5, log .99), dt bias ~ U(log 1e-3, log 1e-2), D = 1, w_noise = 0;
    core.py:315-318, 1045-1062) and, with ``perturb``, jitters the constant-initialised
    tensors so that parity tests exercise non-trivial LayerNorm affines, biases and noise
    scales.  The fixtures load exactly these tensors into the reference modules."""
    g = torch.Generator().manual_seed(seed)
    Di, R = H * N, math.ceil(Dm / 16)

    def nrm(*s, std=0.02):
        return (torch.randn(*s, generator=g) * std).to(dtype)

    def uni(*s, lo, hi):
        return (torch.rand(*s, generator=g) * (hi - lo) + lo).to(dtype)

    jit = 0.1 if perturb else 0.0
    sd: Params = {}
    a = "attention.attention_mechanism_impl."
    sd[a + "A_log"] = uni(H, N, lo=math.log(0.5), hi=math.log(0.99))
    sd[a + "D"] = 1.0 + jit * nrm(Di, std=1.0)
    sd[a + "in_proj_x.weight"] = nrm(Di, Dm)
    sd[a + "in_proj_z.weight"] = nrm(Di, Dm)
    sd[a + "conv1d.weight"] = uni(Di, 1, Kc, lo=-0.5, hi=0.5)       # torch Conv1d default: U(+-1/sqrt(Kc))
    sd[a + "conv1d.bias"] = uni(Di, lo=-0.5, hi=0.5)
    sd[a + "x_param_proj.weight"] = nrm(R + 2 * Di, Di)
    sd[a + "dt_proj_head.weight"] = nrm(H, R)
    sd[a + "dt_proj_head.bias"] = uni(H, lo=math.log(1e-3), hi=math.log(1e-2))
    sd[a + "out_proj.weight"] = nrm(Dm, Di)
    for pre in ("attention.pre_norm.", "feed_forward.pre_norm."):
        sd[pre + "weight"] = 1.0 + jit * nrm(Dm, std=1.0)
        sd[pre + "bias"] = jit * nrm(Dm, std=1.0)
    f = "feed_forward.ffn."
    sd[f + "w_noise"] = jit * nrm(E, std=1.0)
    sd[f + "router_norm.weight"] = 1.0 + jit * nrm(Dm, std=1.0)
    sd[f + "router_norm.bias"] = jit * nrm(Dm, std=1.0)
    sd[f + "router.weight"] = nrm(E, Dm)
    sd[f + "router.bias"] = jit * nrm(E, std=0.2)
    for e in range(E):
        sd[f + f"experts.{e}.0.weight"] = 1.0 + jit * nrm(Dm, std=1.0)
        sd[f + f"experts.{e}.0.bias"] = jit * nrm(Dm, std=1.0)
        sd[f + f"experts.{e}.1.weight"] = nrm(I, Dm)
        sd[f + f"experts.{e}.1.bias"] = jit * nrm(I, std=0.2)
        sd[f + f"experts.{e}.4.weight"] = nrm(Dm, I)
        sd[f + f"experts.{e}.4.bias"] = jit * nrm(Dm, std=0.2)
    return sd


def make_inputs(Bsz: int, L: int, Dm: int, E: int, *, seed: int = 0):
    """x ~ N(0,1) [B,L,Dm] and the routing noise draw [B*L,E] from one seeded generator."""
    g = torch.Generator().manual_seed(1000 + seed)
    x = torch.randn(Bsz, L, Dm, generator=g)
    noise = torch.randn(Bsz * L, E, generator=g)
    return x, noise


def block_loss(out: Tensor, lb: Tensor, rz: Tensor) -> Tensor:
    """The synthetic objective of SURVEY.md section 8(d): mean(out^2) + lb + rz."""
    return out.float().pow(2).mean() + lb + rz
