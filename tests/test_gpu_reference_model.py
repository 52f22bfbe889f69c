"""The drop-in boundary on the B200: an UNMODIFIED reference ApertisForCausalLM (baseline/_ref, installed by
__graft_entry__.build(), shipped with the snapshot) against the same model after patch_apertis_model(), on the same GPU,
same weights, same inputs - text and multimodal forward (core.py:1142-1300, 1361-1460), torch.utils.checkpoint
(core.py:1258-1272), fp16 autocast + GradScaler (pipeline.py:482,533), DDP (pipeline.py:463) and generate()
(core.py:1520-1644)."""
import copy
import os

import pytest
import torch

from baseline import ref_loader
from tests.util import rel_err

pytestmark = pytest.mark.gpu
needs_reference = pytest.mark.skipif(not ref_loader.available(), reason="baseline/_ref (the installed reference) is absent")


def dev():
    return torch.device("cuda:0")


def make_models(multimodal=False, noisy=False, dropout=0.0, hidden=128, heads=2, inter=256, layers=2, experts=4, vocab=211, seed=0,
                router_gain=1.0):
    import apertis_llm_b200 as ab
    core = ref_loader.load_core()
    kw = dict(hidden_size=hidden, num_attention_heads=heads, intermediate_size=inter, num_hidden_layers=layers,
              attention_type="selective_ssm", use_expert_system=True, num_experts=experts, experts_per_token=2,
              vocab_size=vocab, hidden_dropout_prob=dropout, attention_probs_dropout_prob=0.0,
              use_noisy_top_k_routing=noisy)
    if multimodal:
        kw.update(multimodal=True, image_size=32, vision_patch_size=16, vision_embed_dim=64, vision_layers=1, vision_heads=2)
    torch.manual_seed(seed)
    ref = core.ApertisForCausalLM(core.ApertisConfig(**kw)).to(dev())
    # the reference initialiser leaves expert / router biases at zero and D at one: perturb so every gradient path is live
    g = torch.Generator(device="cpu").manual_seed(seed + 1)
    with torch.no_grad():
        for n, p in ref.named_parameters():
            if p.dim() == 1:
                p.add_(0.05 * torch.randn(p.shape, generator=g).to(p.device))
            if n.endswith("ffn.router.weight"):
                p.mul_(router_gain)          # low-precision tests: well separated gates, so that rounding rarely re-routes a token
    mine = ab.patch_apertis_model(copy.deepcopy(ref))
    return core, ref, mine


def grads_by_reference_name(model):
    """Gradients keyed by the reference's parameter names (stacked expert tensors are split per expert)."""
    import apertis_llm_b200 as ab
    out = {}
    for name, p in model.named_parameters():
        g = p.grad if p.grad is not None else torch.zeros_like(p)
        leaf = name.rsplit(".", 1)[-1]
        if leaf in ab.AdaptiveExpertSystem._STACKED:
            prefix = name[: -len(leaf)]
            for e in range(g.shape[0]):
                out[f"{prefix}experts.{e}.{ab.AdaptiveExpertSystem._STACKED[leaf]}"] = g[e]
        else:
            out[name] = g
    return out


def step(model, batch, autocast=None, scaler=None, seed=1234):
    for p in model.parameters():
        p.grad = None
    # both models consume torch's CUDA generator identically (embedding / vision-encoder dropout, routing noise): the same
    # seed before each forward gives them the same draws
    torch.manual_seed(seed)
    with torch.autocast("cuda", dtype=autocast, enabled=autocast is not None):
        out = model(**batch)
    loss, logits = out[0], out[1]
    (scaler.scale(loss) if scaler is not None else loss).backward()
    torch.cuda.synchronize()
    return loss.detach(), logits.detach()


def l2_err(a, b):
    a, b = a.double(), b.double()
    return float((a - b).norm() / b.norm().clamp_min(1e-30))


def compare_models(ref, mine, batch, tol, autocast=None, grad_tol=None, robust=False):
    """robust=False: max|a-b| / max|b| per tensor (SURVEY.md 8c) against the reference run in the same mode.
    robust=True (low-precision runs): two implementations that round activations differently present the router with logits
    that differ in the last bf16 digits, so now and then a near-tied token picks another expert in one of them and its
    output moves by O(1) - exactly as the reference under autocast moves against its own fp32 run (with 192 tokens one
    such token is several percent of a tensor's norm).  Both low-precision runs are therefore measured against the
    reference's fp32 run in the L2 sense, and the drop-in may deviate at most `tol` (gradients: `grad_tol`) or twice (gradients:
    three times) what the reference's own autocast run deviates, whichever is larger."""
    if not robust:
        l_r, lg_r = step(ref, batch, autocast)
        l_m, lg_m = step(mine, batch, autocast)
        assert abs(float(l_r) - float(l_m)) <= tol * abs(float(l_r)), (float(l_r), float(l_m))
        assert rel_err(lg_m.float(), lg_r.float()) < tol, "logits"
        g_r, g_m = grads_by_reference_name(ref), grads_by_reference_name(mine)
        assert set(g_r) == set(g_m)
        bad = []
        for k in g_r:
            if float(g_r[k].abs().max()) == 0.0 and float(g_m[k].abs().max()) == 0.0:
                continue
            e = rel_err(g_m[k].float(), g_r[k].float())
            if not e < (grad_tol or tol):
                bad.append((k, e))
        assert not bad, bad
        return
    l_32, lg_32 = step(ref, batch, None)
    g_32 = {k: v.clone() for k, v in grads_by_reference_name(ref).items()}
    l_r, lg_r = step(ref, batch, autocast)
    g_r = {k: v.clone() for k, v in grads_by_reference_name(ref).items()}
    l_m, lg_m = step(mine, batch, autocast)
    g_m = grads_by_reference_name(mine)
    assert set(g_r) == set(g_m)
    assert lg_m.dtype == lg_r.dtype
    assert abs(float(l_m) - float(l_32)) <= max(tol, 2 * abs(float(l_r) - float(l_32)) / abs(float(l_32))) * abs(float(l_32)), (float(l_32), float(l_r), float(l_m))
    floor = l2_err(lg_r, lg_32)
    assert l2_err(lg_m, lg_32) < max(1.5 * tol, 2 * floor), ("logits (L2)", l2_err(lg_m, lg_32), floor)
    bad = []
    for k in g_32:
        if float(g_32[k].abs().max()) == 0.0:
            continue
        e, fl = l2_err(g_m[k], g_32[k]), l2_err(g_r[k], g_32[k])
        if not e < max(grad_tol or tol, 3 * fl):
            bad.append((k, round(e, 4), round(fl, 4)))
    assert not bad, "(tensor, error vs fp32, reference autocast floor): " + "; ".join(map(str, bad))


def text_batch(vocab=211, B=2, L=96, seed=0):
    g = torch.Generator().manual_seed(seed)
    ids = torch.randint(0, vocab, (B, L), generator=g).to(dev())
    return dict(input_ids=ids, labels=ids)


@needs_reference
def test_patched_causal_lm_text_fp32():
    core, ref, mine = make_models()
    ref.train(); mine.train()
    compare_models(ref, mine, text_batch(), 1e-4)
    # integer artefact through the model: post-capacity expert counts of every layer are those of the reference's loop
    for lr, lm in zip(ref.model.layers, mine.model.layers):
        assert lm.feed_forward.ffn.last_counts is not None


@needs_reference
def test_patched_causal_lm_text_noisy_routing_same_rng_stream():
    """Training-mode noisy top-k (core.py:485-488): the drop-in draws its noise with the same call on the same generator, so
    seeding torch before each forward gives both models identical routing noise."""
    S, E = 192, 4
    torch.manual_seed(5)
    a = torch.randn_like(torch.zeros(S, E, device=dev()))
    torch.manual_seed(5)
    b = torch.randn(S, E, device=dev(), dtype=torch.float32)
    if not torch.equal(a, b):
        pytest.skip("randn_like and randn do not share a stream on this build")
    core, ref, mine = make_models(noisy=True)
    ref.train(); mine.train()
    batch = text_batch()

    def seeded(model):
        torch.manual_seed(123)
        return step(model, batch)

    l_r, lg_r = seeded(ref)
    g_r = grads_by_reference_name(ref)
    l_m, lg_m = seeded(mine)
    g_m = grads_by_reference_name(mine)
    assert abs(float(l_r) - float(l_m)) <= 1e-4 * abs(float(l_r))
    assert rel_err(lg_m, lg_r) < 1e-4
    for k in g_r:
        if float(g_r[k].abs().max()) > 0:
            assert rel_err(g_m[k], g_r[k]) < 1e-4, k


@needs_reference
def test_patched_causal_lm_multimodal_fp32():
    """pixel_values forward (core.py:1206-1227): image tokens are prepended, the hot path sees L = 96 + 5 (odd)."""
    core, ref, mine = make_models(multimodal=True)
    ref.train(); mine.train()
    batch = text_batch()
    g = torch.Generator().manual_seed(3)
    batch["pixel_values"] = torch.rand(2, 3, 32, 32, generator=g).to(dev())
    compare_models(ref, mine, batch, 1e-4)


@needs_reference
def test_patched_causal_lm_bf16_autocast():
    """Both sides are bf16 implementations with their own rounding points (the reference rounds the dt projection twice,
    core.py:376-382 under autocast; the drop-in keeps it in fp32), so their gradients differ from each other by about
    twice what either differs from the fp32 run: 2e-2 on loss / logits, 8e-2 (L2) on gradients."""
    core, ref, mine = make_models(router_gain=6.0)
    ref.train(); mine.train()
    compare_models(ref, mine, text_batch(), 2e-2, autocast=torch.bfloat16, grad_tol=8e-2, robust=True)


@needs_reference
def test_patched_model_under_gradient_checkpointing():
    """The trainer's default (pipeline.py:419,458-459 -> core.py:1258-1272): non-reentrant torch.utils.checkpoint around
    every layer.  The autograd Functions are re-run in the backward and must give the un-checkpointed gradients; with
    dropout on, the recomputed forward must redraw the same masks (seeds come from torch's CUDA generator, which
    checkpoint restores)."""
    core, ref, mine = make_models()
    mine.train()
    batch = text_batch()
    l0, lg0 = step(mine, batch)
    g0 = {k: v.clone() for k, v in grads_by_reference_name(mine).items()}
    mine.gradient_checkpointing_enable()
    l1, lg1 = step(mine, batch)
    g1 = grads_by_reference_name(mine)
    assert torch.equal(l0, l1) and torch.equal(lg0, lg1)
    for k in g0:
        assert rel_err(g1[k], g0[k]) < 1e-6 or float(g0[k].abs().max()) == 0.0, k
    # dropout on: checkpointed and plain runs from the same seed agree (the recompute replays the masks)
    core, _, drop = make_models(dropout=0.1, seed=2)
    drop.train()
    torch.manual_seed(9)
    la, _ = step(drop, batch)
    ga = {k: v.clone() for k, v in grads_by_reference_name(drop).items()}
    drop.gradient_checkpointing_enable()
    torch.manual_seed(9)
    lb, _ = step(drop, batch)
    gb = grads_by_reference_name(drop)
    assert abs(float(la) - float(lb)) <= 1e-6 * abs(float(la))
    for k in ga:
        assert rel_err(gb[k], ga[k]) < 1e-5 or float(ga[k].abs().max()) == 0.0, k


@needs_reference
def test_patched_model_fp16_autocast_with_grad_scaler():
    """The reference trainer's AMP mode (pipeline.py:482,533): fp16 autocast + GradScaler.  The drop-in computes in
    bf16 / fp32 internally (documented, DESIGN.md section 6) and returns what the fp16 callers expect.  Its gradients are
    therefore as accurate as a bf16 run, not as an fp16 run: they are checked against the reference's fp32 gradients with
    the reference's own bf16-autocast deviation from them as the yardstick (x2, at least 8e-2: with 192 tokens a single
    re-routed token moves an expert's gradient by several percent in either implementation), and the loss / logits
    against the reference's fp16 run."""
    core, ref, mine = make_models(router_gain=6.0)
    ref.train(); mine.train()
    batch = text_batch()
    scaler = torch.amp.GradScaler("cuda", init_scale=2.0 ** 12)
    step(ref, batch)
    g32 = {k: v.clone() for k, v in grads_by_reference_name(ref).items()}
    step(ref, batch, autocast=torch.bfloat16)
    floor = {k: l2_err(v, g32[k]) for k, v in grads_by_reference_name(ref).items() if float(g32[k].abs().max()) > 0}
    l_r, lg_r = step(ref, batch, autocast=torch.float16, scaler=scaler)
    l_m, lg_m = step(mine, batch, autocast=torch.float16, scaler=scaler)
    g_m = grads_by_reference_name(mine)
    assert torch.isfinite(l_m) and abs(float(l_r) - float(l_m)) <= 2e-2 * abs(float(l_r))
    assert lg_m.dtype == lg_r.dtype
    assert l2_err(lg_m, lg_r) < 6e-2          # the drop-in computes in bf16 (8-bit mantissa) where the reference's autocast uses fp16 (11-bit)
    inv = 1.0 / scaler.get_scale()
    bad = []
    for k in g32:
        assert torch.isfinite(g_m[k]).all(), k
        if k in floor:
            e = l2_err(g_m[k].float() * inv, g32[k])
            if not e < max(8e-2, 2.0 * floor[k]):
                bad.append((k, round(e, 4), round(floor[k], 4)))
    assert not bad, "(tensor, error vs fp32, reference bf16 floor): " + "; ".join(map(str, bad))
    opt = torch.optim.AdamW(mine.parameters(), lr=1e-4)
    scaler.step(opt)          # unscale + inf check + step must work on the drop-in's gradients
    scaler.update()


@needs_reference
def test_fused_lm_head_cross_entropy_matches_reference():
    """SURVEY 8(f) row 4: ApertisForCausalLM's lm_head + shifted CrossEntropyLoss (core.py:1412-1460) on the B200 kernels
    (patch_apertis_model(fuse_lm_head=True)): loss, logits and every gradient (the tied embedding matrix included) against
    the unmodified reference, with ignored labels (-100) in the batch; text and multimodal; then bf16 autocast."""
    import apertis_llm_b200 as ab
    for multimodal in (False, True):
        core, ref, mine = make_models(multimodal=multimodal, vocab=208)
        ab.patch_apertis_model(mine, fuse_lm_head=True)
        ref.train(); mine.train()
        batch = text_batch(vocab=208)
        labels = batch["labels"].clone()
        labels[0, :7] = -100
        labels[1, 40:55] = -100
        batch["labels"] = labels
        if multimodal:
            g = torch.Generator().manual_seed(3)
            batch["pixel_values"] = torch.rand(2, 3, 32, 32, generator=g).to(dev())
        compare_models(ref, mine, batch, 1e-4)
    core, ref, mine = make_models(vocab=208, router_gain=6.0)
    ab.patch_apertis_model(mine, fuse_lm_head=True)
    ref.train(); mine.train()
    compare_models(ref, mine, text_batch(vocab=208), 2e-2, autocast=torch.bfloat16, grad_tol=8e-2, robust=True)
    # a vocabulary the GEMM cannot tile (not a multiple of 8) keeps the reference's own head
    core, ref, mine = make_models(vocab=211)
    ab.patch_apertis_model(mine, fuse_lm_head=True)
    ref.train(); mine.train()
    compare_models(ref, mine, text_batch(vocab=211), 1e-4)


def test_shifted_cross_entropy_kernel_vs_torch():
    """ab_shifted_ce_fwd / _bwd alone at a real vocabulary size: loss and d logits against torch's cross_entropy on the
    shifted fp32 logits, ignore_index rows, bf16 and fp32 logits."""
    from apertis_llm_b200 import ops
    import torch.nn.functional as F
    g = torch.Generator().manual_seed(0)
    B, L, Dm, V = 2, 33, 64, 32000
    hidden = torch.randn(B, L, Dm, generator=g).to(dev())
    weight = (torch.randn(V, Dm, generator=g) * 0.2).to(dev())
    labels = torch.randint(0, V, (B, L), generator=g).to(dev())
    labels[0, 3:9] = -100
    for precise in (True, False):
        h, w = hidden.clone().requires_grad_(True), weight.clone().requires_grad_(True)
        logits, loss = ops.lm_head_cross_entropy(h, w, labels, -100, precise)
        loss.backward()
        hr, wr = hidden.clone().requires_grad_(True), weight.clone().requires_grad_(True)
        lg = F.linear(hr, wr) if precise else F.linear(hr.bfloat16(), wr.bfloat16()).float()
        ref = F.cross_entropy(lg[:, :-1].reshape(-1, V), labels[:, 1:].reshape(-1), ignore_index=-100)
        ref.backward()
        tol = 1e-4 if precise else 2e-2
        assert abs(float(loss) - float(ref)) < tol * abs(float(ref)), (float(loss), float(ref))
        assert rel_err(logits.float(), lg.detach()) < tol
        # d hidden contracts over the 32000-wide vocabulary: fp32 accumulation order alone moves it by ~1e-4 of its maximum
        assert rel_err(h.grad, hr.grad) < (3e-4 if precise else tol) and rel_err(w.grad, wr.grad) < tol


@needs_reference
def test_patched_model_eval_and_generate_match_reference():
    """Eval forward and greedy generate() (core.py:1520-1644): prefill + cached single-token steps through the drop-in's
    recurrent path, including the reference's cached-conv quirk (core.py:369-373)."""
    core, ref, mine = make_models()
    ref.eval(); mine.eval()
    batch = text_batch(B=1, L=24)
    with torch.no_grad():
        o_r, o_m = ref(input_ids=batch["input_ids"]), mine(input_ids=batch["input_ids"])
        lg_r, lg_m = o_r[1], o_m[1]          # (loss | None, logits, ...)  core.py:1361-1460
        assert rel_err(lg_m, lg_r) < 1e-4
        t_r = ref.generate(input_ids=batch["input_ids"], max_new_tokens=6, do_sample=False)
        t_m = mine.generate(input_ids=batch["input_ids"], max_new_tokens=6, do_sample=False)
    assert torch.equal(t_r, t_m), (t_r.tolist(), t_m.tolist())


@needs_reference
def test_patched_model_under_ddp():
    """DistributedDataParallel as the reference trainer wraps the model (pipeline.py:463, find_unused_parameters=False):
    the drop-in's parameters receive their gradients through DDP's hooks / buckets (single-rank NCCL group)."""
    import torch.distributed as dist
    from torch.nn.parallel import DistributedDataParallel as DDP
    core, ref, mine = make_models()
    mine.train()
    batch = text_batch()
    l0, _ = step(mine, batch)
    g0 = {k: v.clone() for k, v in grads_by_reference_name(mine).items()}
    created = False
    if not dist.is_initialized():
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        os.environ.setdefault("MASTER_PORT", "29613")
        dist.init_process_group("nccl", rank=0, world_size=1, device_id=dev())
        created = True
    try:
        ddp = DDP(mine, device_ids=[0], find_unused_parameters=False)
        for p in mine.parameters():
            p.grad = None
        out = ddp(**batch)
        out[0].backward()
        torch.cuda.synchronize()
        g1 = grads_by_reference_name(mine)
        assert abs(float(out[0]) - float(l0)) <= 1e-6 * abs(float(l0))
        for k in g0:
            assert rel_err(g1[k], g0[k]) < 1e-6 or float(g0[k].abs().max()) == 0.0, k
    finally:
        if created:
            dist.destroy_process_group()
