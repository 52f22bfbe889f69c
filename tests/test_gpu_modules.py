"""Module-level parity on the B200: the drop-in modules against the golden fixtures recorded from the
unmodified reference (tests/golden) and against the CPU oracle on the same seeded inputs."""
import numpy as np
import pytest
import torch

from oracle import apertis_oracle as O
from tests.util import load_golden, rel_err, sample

pytestmark = pytest.mark.gpu

BLOCK_CASES = ["block_small_train", "block_small_eval", "block_relu_e4", "block_drop_expert", "block_h3_ragged", "block_c1dims"]


def dev():
    return torch.device("cuda:0")


def build_layer(spec, sd=None, dropout=0.0):
    from apertis_llm_b200 import ApertisLayerB200, BlockConfig
    cfg = BlockConfig(hidden_size=spec["Dm"], num_attention_heads=spec["H"], intermediate_size=spec["I"],
                      num_experts=spec["E"], experts_per_token=spec["K"], hidden_dropout_prob=dropout,
                      hidden_act=spec.get("act", "gelu"))
    layer = ApertisLayerB200(cfg)
    if sd is None:
        sd = O.make_layer_params(spec["Dm"], spec["H"], spec["I"], spec["E"], seed=spec["seed"])
    layer.load_state_dict(sd, strict=True)          # reference key names -> stacked expert parameters
    # these cases are checked against fp32 recordings of the reference (tests/golden) and the fp32 oracle, whose routing
    # sees fp32 logits; the autocast-rounded routing is checked against the live reference in test_gpu_reference_model.py
    layer.feed_forward.ffn.router_autocast_rounding = False
    return layer.to(dev()), sd


def set_rng_hooks(layer, spec, noise):
    ffn = layer.feed_forward.ffn
    ffn._draw_noise = lambda S, E, device: noise.to(device)
    if spec.get("perm") is not None:
        E = spec["E"]
        ndrop = int(np.floor(E * 0.1))
        act = torch.ones(E, dtype=torch.int32)
        act[torch.tensor(spec["perm"][:ndrop])] = 0
        ffn._draw_active_mask = lambda device: act.to(device)


def named_grads(layer):
    """Gradients keyed like the reference's named_parameters()."""
    sd = {}
    for k, p in layer.named_parameters():
        g = p.grad if p.grad is not None else torch.zeros_like(p)
        sd[k] = g
    out = {}
    ffn = layer.feed_forward.ffn
    for k, g in sd.items():
        leaf = k.split(".")[-1]
        if leaf in ffn._STACKED:
            for e in range(g.shape[0]):
                out[f"feed_forward.ffn.experts.{e}.{ffn._STACKED[leaf]}"] = g[e]
        else:
            out[k] = g
    return out


def run_block(spec, g, autocast):
    layer, sd = build_layer(spec)
    x, noise = O.make_inputs(spec["B"], spec["L"], spec["Dm"], spec["E"], seed=spec["seed"])
    training = spec.get("training", True)
    layer.train(training)
    set_rng_hooks(layer, spec, noise)
    xg = x.to(dev()).requires_grad_(training)
    with torch.autocast("cuda", dtype=torch.bfloat16, enabled=autocast):
        out, _, _, lb, rz = layer(xg)
    grads = None
    if training:
        O.block_loss(out, lb, rz).backward()
        grads = named_grads(layer)
    torch.cuda.synchronize()
    return layer, out, lb, rz, xg, grads


@pytest.mark.parametrize("name", BLOCK_CASES)
def test_block_fp32_matches_reference(name):
    spec, g = load_golden(name)
    layer, out, lb, rz, xg, grads = run_block(spec, g, autocast=False)
    ffn = layer.feed_forward.ffn
    # integer artefacts first: they must be bit-exact
    S = spec["B"] * spec["L"]
    training = spec.get("training", True)
    cap = O.moe_capacity(S, spec["E"], 1.25, training)
    active = None
    if spec.get("perm") is not None:
        active = np.ones(spec["E"], dtype=bool)
        active[np.array(spec["perm"][: int(np.floor(spec["E"] * 0.1))])] = False
    kept, counts, _ = O.moe_plan(g["idx"], g["w"], spec["E"], cap, active)
    assert np.array_equal(ffn.last_counts.cpu().numpy(), counts.astype(np.int32)), "expert_token_counts_post_capacity"
    assert rel_err(out.float(), g["out"]) < 1e-4, "block output"
    assert abs(float(lb) - float(g["lb"])) < 1e-4 * max(abs(float(g["lb"])), 1e-3)
    assert abs(float(rz) - float(g["rz"])) < 1e-4 * max(abs(float(g["rz"])), 1e-3)
    if not training:
        return
    assert rel_err(xg.grad, g["dx"]) < 1e-4, "dx"
    for k, gr in grads.items():
        if "grad/" + k in g:
            assert rel_err(gr, g["grad/" + k]) < 1e-4, k
        else:
            assert rel_err(sample(gr), g["gsample/" + k]) < 1e-4, k


@pytest.mark.parametrize("name", ["block_small_train", "block_h3_ragged", "block_c1dims", "block_small_eval"])
def test_block_bf16_autocast_within_tolerance(name):
    spec, g = load_golden(name)
    layer, out, lb, rz, xg, grads = run_block(spec, g, autocast=True)
    assert rel_err(out.float(), g["out"]) < 2e-2
    if not spec.get("training", True):
        return
    assert rel_err(xg.grad, g["dx"]) < 2e-2
    bad = []
    for k, gr in grads.items():
        ref = g["grad/" + k] if "grad/" + k in g else None
        err = rel_err(gr, ref) if ref is not None else rel_err(sample(gr), g["gsample/" + k])
        if err >= 2e-2:
            bad.append((k, err))
    assert not bad, bad


def test_router_indices_bit_exact_vs_reference():
    """Indices recorded from the reference's own torch.topk equal the CUDA router's on the same block input."""
    from apertis_llm_b200 import ops
    for name in BLOCK_CASES:
        spec, g = load_golden(name)
        sd = O.make_layer_params(spec["Dm"], spec["H"], spec["I"], spec["E"], seed=spec["seed"])
        _, moe, _ = O.split_layer_params(sd)
        _, noise = O.make_inputs(spec["B"], spec["L"], spec["Dm"], spec["E"], seed=spec["seed"])
        training = spec.get("training", True)
        d = dev()
        ns = (torch.nn.functional.softplus(moe["w_noise"]) * 0.1).to(d)
        r = ops.moe_route(torch.from_numpy(g["moe_in"]).to(d), moe["router_norm.weight"].to(d), moe["router_norm.bias"].to(d), 1e-12,
                          moe["router.weight"].to(d), moe["router.bias"].to(d), noise.to(d) if training else None,
                          ns if training else None, spec["K"])
        assert np.array_equal(r["idx"].cpu().numpy(), g["idx"].astype(np.int32)), name
        assert rel_err(r["w"], g["w"]) < 1e-5, name
        assert rel_err(r["logits"], g["logits"]) < 1e-5, name


def test_ssm_train_and_eval_vs_reference():
    from apertis_llm_b200 import BlockConfig, SelectiveLinearAttention
    spec, g = load_golden("ssm_scans_l512")
    sd = O.make_layer_params(spec["Dm"], spec["H"], spec["I"], spec["E"], seed=spec["seed"])
    ssm_sd, _, _ = O.split_layer_params(sd)
    cfg = BlockConfig(hidden_size=spec["Dm"], num_attention_heads=spec["H"], intermediate_size=spec["I"])
    for mode in (0, 1):
        m = SelectiveLinearAttention(cfg)
        m.load_state_dict(ssm_sd, strict=True)
        m = m.to(dev()).train()
        m.scan_mode = mode
        x, _ = O.make_inputs(spec["B"], spec["L"], spec["Dm"], spec["E"], seed=spec["seed"])
        xg = x.to(dev()).requires_grad_(True)
        out, y, _ = m(xg, output_attentions=True)
        (out.pow(2).mean() + y.pow(2).mean()).backward()
        assert rel_err(out, g["train_out"]) < 1e-4 and rel_err(y, g["train_y"]) < 1e-4
        assert rel_err(xg.grad, g["dx"]) < 1e-4
        for k, p in m.named_parameters():
            assert rel_err(p.grad, g["grad/" + k]) < 1e-4, (mode, k)
        m.eval()
        with torch.no_grad():
            out2, y2, _ = m(xg.detach(), output_attentions=True)
        assert rel_err(out2, g["eval_out"]) < 1e-4 and rel_err(y2, g["eval_y"]) < 1e-4


def test_ssm_cached_decode_vs_reference():
    from apertis_llm_b200 import BlockConfig, SelectiveLinearAttention
    spec, g = load_golden("ssm_cache_decode")
    sd = O.make_layer_params(spec["Dm"], spec["H"], spec["I"], spec["E"], seed=spec["seed"])
    ssm_sd, _, _ = O.split_layer_params(sd)
    m = SelectiveLinearAttention(BlockConfig(hidden_size=spec["Dm"], num_attention_heads=spec["H"]))
    m.load_state_dict(ssm_sd, strict=True)
    m = m.to(dev()).eval()
    x, _ = O.make_inputs(spec["B"], spec["L"] + spec["steps"], spec["Dm"], spec["E"], seed=spec["seed"])
    x = x.to(dev())
    with torch.no_grad():
        full, yfull, _ = m(x, output_attentions=True)
        assert rel_err(full, g["full_out"]) < 1e-4 and rel_err(yfull, g["full_y"]) < 1e-4
        out, y, cache = m(x[:, :spec["L"]], output_attentions=True, use_cache=True)
        assert rel_err(out, g["prefill_out"]) < 1e-4
        assert rel_err(cache[0], g["prefill_conv"]) < 1e-5 and rel_err(cache[1], g["prefill_h"]) < 1e-4
        for s in range(spec["steps"]):
            out, y, cache = m(x[:, spec["L"] + s: spec["L"] + s + 1], past_key_value=cache, output_attentions=True, use_cache=True)
            assert rel_err(out, g[f"step{s}_out"]) < 1e-4, s
            assert rel_err(cache[0], g[f"step{s}_conv"]) < 1e-5 and rel_err(cache[1], g[f"step{s}_h"]) < 1e-4, s


def test_state_dict_round_trip_uses_reference_keys():
    spec, _ = load_golden("block_small_train")
    layer, sd = build_layer(spec)
    out_sd = layer.state_dict()
    assert set(out_sd) == set(sd)
    for k in sd:
        assert torch.equal(out_sd[k].cpu(), sd[k]), k


def test_block_is_deterministic():
    """Bitwise run-to-run determinism of the whole block (forward, input and parameter gradients)."""
    spec, g = load_golden("block_small_train")
    outs = []
    for _ in range(2):
        layer, out, lb, rz, xg, grads = run_block(spec, g, autocast=True)
        outs.append((out.detach().clone(), xg.grad.clone(), {k: v.clone() for k, v in grads.items()}))
    assert torch.equal(outs[0][0], outs[1][0]) and torch.equal(outs[0][1], outs[1][1])
    for k in outs[0][2]:
        assert torch.equal(outs[0][2][k], outs[1][2][k]), k


def test_block_medium_vs_oracle_fp32():
    """C2-like widths at a reduced token count against the CPU oracle (seconds on CPU)."""
    spec = dict(Dm=704, H=11, I=2816, E=8, K=2, B=2, L=384, seed=11)
    layer, sd = build_layer(spec)
    x, noise = O.make_inputs(spec["B"], spec["L"], spec["Dm"], spec["E"], seed=spec["seed"])
    layer.train()
    set_rng_hooks(layer, spec, noise)
    sdr = {k: v.clone().requires_grad_(True) for k, v in sd.items()}
    xr = x.clone().requires_grad_(True)
    out_r, lb_r, rz_r = O.block_forward(sdr, xr, num_heads=spec["H"], E=spec["E"], K=spec["K"], training=True, noise=noise)
    O.block_loss(out_r, lb_r, rz_r).backward()
    xg = x.to(dev()).requires_grad_(True)
    out, _, _, lb, rz = layer(xg)
    O.block_loss(out, lb, rz).backward()
    assert rel_err(out, out_r.detach()) < 1e-4
    assert rel_err(xg.grad, xr.grad) < 1e-4
    grads = named_grads(layer)
    for k, gr in grads.items():
        assert rel_err(gr, sdr[k].grad) < 1e-4, k


def test_no_cpu_fallback():
    from apertis_llm_b200 import BlockConfig, SelectiveLinearAttention
    m = SelectiveLinearAttention(BlockConfig(hidden_size=64, num_attention_heads=2))
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        m(torch.randn(1, 4, 64))


def test_expert_dropout_train_vs_eval_statistics():
    """hidden_dropout_prob > 0: training output is an unbiased, noisier version of the p = 0 output; eval ignores it;
    the mask follows torch's CUDA generator (same seed -> same output), and gradients flow."""
    from apertis_llm_b200 import AdaptiveExpertSystem, BlockConfig
    spec = dict(Dm=128, H=2, I=512, E=8, K=2, B=4, L=512, seed=21)
    sd = O.make_layer_params(spec["Dm"], spec["H"], spec["I"], spec["E"], seed=spec["seed"])
    _, moe_sd, _ = O.split_layer_params(sd)
    x, noise = O.make_inputs(spec["B"], spec["L"], spec["Dm"], spec["E"], seed=spec["seed"])
    outs = {}
    for p in (0.0, 0.3):
        m = AdaptiveExpertSystem(BlockConfig(hidden_size=spec["Dm"], num_attention_heads=spec["H"], intermediate_size=spec["I"],
                                             hidden_dropout_prob=p))
        m.load_state_dict(moe_sd, strict=True)
        m = m.to(dev()).train()
        m._draw_noise = lambda S, E, device: noise.to(device)
        xg = x.to(dev()).requires_grad_(True)
        torch.manual_seed(5)
        o1, _, _ = m(xg)
        o1.pow(2).mean().backward()
        assert torch.isfinite(xg.grad).all() and xg.grad.abs().max() > 0
        torch.manual_seed(5)
        o2, _, _ = m(xg)
        assert torch.equal(o1, o2)
        m.eval()
        oe, _, _ = m(xg)
        outs[p] = (o1.detach(), oe.detach())
    assert torch.equal(outs[0.0][1], outs[0.3][1])                     # eval ignores dropout
    a, b = outs[0.3][0], outs[0.0][0]
    assert not torch.equal(a, b)
    # unbiased: the mean difference over ~260k outputs is far below the per-element noise
    diff = (a - b)
    assert diff.mean().abs().item() < 0.05 * diff.std().item() + 1e-6
    assert rel_err(a, b) < 1.0


@pytest.mark.parametrize("Dm", [128, 256])
def test_cuda_graph_replay_matches_eager(Dm):
    """The whole step (forward, loss, backward) captured as a CUDA graph and replayed gives the eager results: nothing in
    the path synchronises with the host or bakes per-launch host state into the graph.  Dm 128 (d_inner 32): the
    one-tile-per-CTA scan switches to its two-pass schedule under capture (it differs from the single pass only in the
    association of the cross-tile products); Dm 256 (d_inner 64): the pipelined scan, whose launch epoch lives in the
    workspace, is captured as it is."""
    spec = dict(Dm=Dm, H=4, I=256, E=4, K=2, B=2, L=640, seed=5)
    layer, _ = build_layer(spec)
    x, noise = O.make_inputs(spec["B"], spec["L"], spec["Dm"], spec["E"], seed=spec["seed"])
    layer.train()
    noise_d = noise.to(dev())                # resident before the capture: no host-to-device copy inside the graph
    layer.feed_forward.ffn._draw_noise = lambda S, E, device: noise_d
    xs = x.to(dev()).requires_grad_(True)

    def step():
        for p in layer.parameters():
            p.grad = None
        xs.grad = None
        with torch.autocast("cuda", dtype=torch.bfloat16):
            out, _, _, lb, rz = layer(xs)
        O.block_loss(out, lb, rz).backward()
        return out

    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for _ in range(2):
            step()
    torch.cuda.current_stream().wait_stream(side)
    eager_out = step().detach().clone()
    eager_dx = xs.grad.clone()
    eager_g = {k: v.clone() for k, v in named_grads(layer).items()}
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        g_out = step()
    for _ in range(2):                     # replays are repeatable
        graph.replay()
        torch.cuda.synchronize()
        assert rel_err(g_out.float(), eager_out.float()) < 1e-2
        assert rel_err(xs.grad, eager_dx) < 1e-2
        for k, v in named_grads(layer).items():
            assert rel_err(v, eager_g[k]) < 1e-2, k


# the unmodified reference's own bf16-autocast deviation at C4 dims on a B200 reached 4.7 % on the router-path gradients
# (DESIGN.md section 2); no bf16 bound below may be wider than twice that
REFERENCE_BF16_FLOOR_MAX = 0.047


def reference_bf16_floor(spec, sd, x, noise, want):
    """The error a bf16-autocast run of the reference's algorithm makes on this GPU, on the same weights, inputs and routing
    noise, against the fp32 gradients `want` (metric: tests.util.rel_err per tensor): the noise floor of a bf16 run of this
    shape, where near-tied tokens re-route and sums over tokens cancel.  The layer run is the oracle (the reference layer's
    op sequence, pinned to the reference in fp32 by tests/test_oracle_golden.py).  Its bf16 deviation is not the
    reference's: at C4 dims it runs up to 10 % on the router-path gradients where the reference's stayed within 4.7 %, so
    the caller caps it at REFERENCE_BF16_FLOOR_MAX."""
    sdg = {k: v.to(dev()).requires_grad_(True) for k, v in sd.items()}
    with torch.autocast("cuda", dtype=torch.bfloat16):
        out, lb, rz = O.block_forward(sdg, x.to(dev()), num_heads=spec["H"], E=spec["E"], K=spec["K"], training=True,
                                      noise=noise.to(dev()), act=spec.get("act", "gelu"))
    O.block_loss(out.float(), lb.float(), rz.float()).backward()
    torch.cuda.synchronize()
    floor = {k: rel_err(p.grad, want[k]) for k, p in sdg.items() if p.grad is not None and k in want}
    del sdg, out
    torch.cuda.empty_cache()
    return floor


@pytest.mark.parametrize("name,Dm,H,I,B,L,autocast", [
    ("c2_full_fp32", 704, 11, 2816, 8, 4096, False),        # BASELINE.json configs[1] at the size bench.py times
    ("c2_full_bf16", 704, 11, 2816, 8, 4096, True),
    ("c3_multimodal_len", 704, 11, 2816, 1, 4673, False),   # configs[2]: 4096 text + 577 image tokens (odd, not a tile multiple)
    ("c4_7b_dims", 1600, 25, 6400, 1, 4096, False),         # configs[3]: d_inner 400 (6 slabs + 16 channels), I 6400
    ("c4_7b_dims_bf16", 1600, 25, 6400, 2, 4096, True),
])
def test_block_baseline_configs_vs_oracle(name, Dm, H, I, B, L, autocast):
    """The block at the BASELINE.json shapes against the CPU oracle on the same seeded inputs and weights: output, both
    aux losses, the post-capacity expert counts (bit-exact), the input gradient and every parameter gradient."""
    spec = dict(Dm=Dm, H=H, I=I, E=8, K=2, B=B, L=L, seed=29)
    S = B * L
    layer, sd = build_layer(spec)
    x, noise = O.make_inputs(B, L, Dm, 8, seed=29)
    layer.train()
    set_rng_hooks(layer, spec, noise)
    sdr = {k: v.clone().requires_grad_(True) for k, v in sd.items()}
    xr = x.clone().requires_grad_(True)
    # O.block_forward spelled out so that the routing artefacts of the oracle are at hand
    ssm, moe, norms = O.split_layer_params(sdr)
    F = torch.nn.functional
    n1 = F.layer_norm(xr, (Dm,), norms["attention.pre_norm.weight"], norms["attention.pre_norm.bias"], 1e-12)
    a_r, _, _ = O.ssm_forward(ssm, n1, num_heads=H, training=True)
    h_r = a_r + xr
    n2 = F.layer_norm(h_r, (Dm,), norms["feed_forward.pre_norm.weight"], norms["feed_forward.pre_norm.bias"], 1e-12)
    m_r, lb_r, rz_r, parts = O.moe_forward(moe, n2, E=8, K=2, training=True, noise=noise, return_parts=True)
    out_r = m_r + h_r
    O.block_loss(out_r, lb_r, rz_r).backward()
    xg = x.to(dev()).requires_grad_(True)
    with torch.autocast("cuda", dtype=torch.bfloat16, enabled=autocast):
        out, _, _, lb, rz = layer(xg)
    O.block_loss(out, lb, rz).backward()
    torch.cuda.synchronize()
    tol = 2e-2 if autocast else 1e-4
    idx_g, row_of = (t.cpu().numpy() for t in layer.feed_forward.ffn.last_routing)
    idx_o, kept_o = parts["idx"].numpy(), parts["kept"]
    same = (idx_g == idx_o).all(1) & ((row_of >= 0) == kept_o).all(1)       # tokens routed and kept exactly as by the oracle
    if not autocast:
        assert same.all(), "fp32: router indices and kept (token, slot) sets are the oracle's, bit for bit"
        assert rel_err(out.float(), out_r.detach()) < tol, "out"
    else:
        # bf16 activations move a few near-tied logits of the 10^4..10^5 tokens across a top-k / capacity boundary (the
        # reference under autocast does the same against its own fp32 run); such a token's output changes by O(1), so the
        # element-wise bound is asserted on the tokens routed identically and the flipped fraction is bounded separately
        assert same.mean() > 0.97, f"routing agreement {same.mean():.4f}"
        same_t = torch.from_numpy(same)
        o, o_r = out.float().reshape(S, Dm).cpu(), out_r.detach().reshape(S, Dm)
        assert rel_err(o[same_t], o_r[same_t]) < tol, "out (identically routed tokens)"
    assert abs(float(lb) - float(lb_r)) < max(tol, 1e-4) * max(abs(float(lb_r)), 1e-3)
    assert abs(float(rz) - float(rz_r)) < max(tol, 1e-4) * max(abs(float(rz_r)), 1e-3)
    counts = layer.feed_forward.ffn.last_counts.cpu().numpy()
    if not autocast:        # fp32: same logits to ~1e-6, so the post-capacity counts are the oracle's, bit for bit
        assert np.array_equal(counts, parts["counts"].astype(np.int32)), "expert_token_counts_post_capacity"
    else:
        assert int(counts.max()) <= parts["cap"] and abs(int(counts.sum()) - int(parts["counts"].sum())) <= 8
    if not autocast:
        assert rel_err(xg.grad, xr.grad) < tol, "dx"
    else:
        # a re-routed token also perturbs its neighbours' input gradients through the scan: bound the error in the L2 sense
        dg, dr = xg.grad.reshape(S, Dm).cpu().double(), xr.grad.reshape(S, Dm).double()
        assert float((dg - dr).norm() / dr.norm()) < 2e-2, "dx"
    # bf16: parameter gradients are sums over all tokens in which re-routed tokens and cancellation show; the bound is 5e-2
    # or twice what a bf16-autocast run of the reference's algorithm on this GPU deviates from the same fp32 gradients,
    # that deviation capped at the largest one recorded for the unmodified reference
    floor = reference_bf16_floor(spec, sd, x, noise, {k: v.grad for k, v in sdr.items()}) if autocast else {}
    bad = []
    for k, gr in named_grads(layer).items():
        e = rel_err(gr, sdr[k].grad)
        bound = tol if not autocast else max(5e-2, 2.0 * min(floor.get(k, 0.0), REFERENCE_BF16_FLOOR_MAX))
        if not e < bound:
            bad.append((k, round(e, 4), floor.get(k)))
    assert not bad, "(tensor, error, reference bf16 floor): " + "; ".join(map(str, bad))
