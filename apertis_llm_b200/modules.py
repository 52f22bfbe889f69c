"""Drop-in nn.Modules for the Apertis block hot path.

``SelectiveLinearAttention`` and ``AdaptiveExpertSystem`` keep the reference's class names, constructor
arguments, ``forward()`` signatures, return tuples and ``state_dict`` keys (core.py:295-401, 403-607), so
``ApertisAttention`` / ``ApertisFeedForward`` (core.py:650, 861-865, 699-704, 894) can hold them unchanged.
``patch_apertis_model`` swaps them into an existing reference ``ApertisModel`` in place.

All arithmetic of the two layers runs in the sm_100a kernels behind the C ABI, the SSM projections
(core.py:366-367, 376-383, 397) included: they run on the library's tcgen05 GEMM kernel, in_proj_x | in_proj_z as
one GEMM and x_param_proj with dt_proj_head folded in as one GEMM.  There is no CPU / other-GPU fallback: calling
these modules on a non-sm_100 device raises.
"""
from __future__ import annotations

import math
from dataclasses import dataclass
from typing import Any, Optional, Tuple

import torch
import torch.nn as nn
import torch.nn.functional as F

from . import _lib, ops


@dataclass
class BlockConfig:
    """The subset of ApertisConfig (core.py:67-204) the hot path reads, with the reference's defaults."""
    hidden_size: int = 768
    num_attention_heads: int = 12
    intermediate_size: int = 3072
    hidden_act: str = "gelu"
    hidden_dropout_prob: float = 0.1
    layer_norm_eps: float = 1e-12
    ssm_d_state: int = 16
    ssm_dt_rank: Any = "auto"
    ssm_conv_kernel: int = 4
    num_experts: int = 8
    experts_per_token: int = 2
    load_balancing_loss_coef: float = 0.01
    expert_capacity_factor: float = 1.25
    noisy_routing_alpha: float = 0.1
    expert_dropout_prob: float = 0.1
    router_z_loss_coef: float = 0.001
    use_noisy_top_k_routing: bool = True
    use_expert_capacity_limit: bool = True
    use_expert_dropout: bool = True
    use_router_z_loss: bool = True
    use_load_balancing_loss: bool = True
    attention_type: str = "selective_ssm"
    use_expert_system: bool = True
    use_rmsnorm: bool = False

    def __post_init__(self):
        if self.ssm_dt_rank == "auto":
            self.ssm_dt_rank = math.ceil(self.hidden_size / 16)      # core.py:163-164
        self.ssm_d_inner = self.num_attention_heads * self.ssm_d_state  # core.py:154
        self.experts_per_token = min(self.num_experts, self.experts_per_token)


def _autocast_dtype(device_type: str = "cuda") -> Optional[torch.dtype]:
    """The active autocast dtype, or None.  torch.float16 is what the reference trainer asks for (pipeline.py:482,533:
    ``torch.amp.autocast('cuda')`` + ``GradScaler``); the kernels then compute in bf16 / fp32 (same exponent range as fp32,
    so the scaler's 2^16 loss scale cannot overflow inside the layer) and only the tensors the reference would return
    as fp16 are cast on the way out."""
    if not torch.is_autocast_enabled(device_type):
        return None
    return torch.get_autocast_dtype(device_type)


def _compute_dtype(ac: Optional[torch.dtype]) -> Optional[torch.dtype]:
    """Kernel activation dtype for an autocast dtype: fp16 requests run in bf16."""
    return torch.bfloat16 if ac == torch.float16 else ac


# ================================================================================================
# SSM layer
# ================================================================================================
SSM_D_STATES = (16, 32, 64)              # ssm_d_state values the selective-scan kernels take (csrc/ssm_scan_rounds.cu)
SSM_CONV_KERNELS = tuple(range(2, 9))    # ssm_conv_kernel values the causal-conv kernels take (csrc/ssm_conv.cu)


class SelectiveLinearAttention(nn.Module):
    """B200-native SelectiveLinearAttention (core.py:295-401): same parameters, same forward contract."""

    def __init__(self, config):
        super().__init__()
        self.hidden_size = config.hidden_size
        self.num_heads = config.num_attention_heads
        self.d_state = config.ssm_d_state
        self.d_inner = self.num_heads * self.d_state
        self.dt_rank = config.ssm_dt_rank
        self.conv_kernel_size = config.ssm_conv_kernel
        # limits of the kernels: a 64-channel slab of the scan holds whole heads; the conv keeps its window in registers.
        # ssm_conv_kernel 1 stays out: the reference's conv state x_seq[:, :, -(Kc-1):] (core.py:372) is then the whole sequence
        if self.d_state not in SSM_D_STATES:
            raise NotImplementedError(f"the selective-scan kernels support ssm_d_state in {SSM_D_STATES} (got {self.d_state})")
        if not SSM_CONV_KERNELS[0] <= self.conv_kernel_size <= SSM_CONV_KERNELS[-1]:
            raise NotImplementedError(f"the causal-conv kernels support ssm_conv_kernel in {SSM_CONV_KERNELS[0]}..{SSM_CONV_KERNELS[-1]} "
                                      f"(got {self.conv_kernel_size})")
        self.in_proj_x = nn.Linear(self.hidden_size, self.d_inner, bias=False)
        self.in_proj_z = nn.Linear(self.hidden_size, self.d_inner, bias=False)
        self.conv1d = nn.Conv1d(self.d_inner, self.d_inner, kernel_size=self.conv_kernel_size, groups=self.d_inner,
                                padding=self.conv_kernel_size - 1)
        self.x_param_proj = nn.Linear(self.d_inner, self.dt_rank + 2 * self.d_inner, bias=False)
        self.dt_proj_head = nn.Linear(self.dt_rank, self.num_heads, bias=True)
        nn.init.uniform_(self.dt_proj_head.bias, a=math.log(1e-3), b=math.log(1e-2))          # core.py:315
        self.A_log = nn.Parameter(torch.empty(self.num_heads, self.d_state))
        nn.init.uniform_(self.A_log, a=math.log(0.5), b=math.log(0.99))                       # core.py:316-317
        self.D = nn.Parameter(torch.ones(self.d_inner))
        self.out_proj = nn.Linear(self.d_inner, self.hidden_size, bias=False)
        self.use_cache = False
        self.scan_mode: Optional[int] = None      # None = library default (the "rounds" schedule); 0 / 1 / 2 select the older ones

    def forward(self, hidden_states: torch.Tensor, attention_mask: Optional[torch.Tensor] = None,
                position_ids: Optional[torch.Tensor] = None,
                past_key_value: Optional[Tuple[torch.Tensor, torch.Tensor]] = None,
                output_attentions: bool = False, use_cache: bool = False):
        # attention_mask / position_ids are accepted and ignored, exactly like the reference (core.py:355-401)
        _lib.ensure_device(hidden_states.device)
        ac = _autocast_dtype()
        if ac == torch.float16:
            # the reference trainer's AMP mode (pipeline.py:482,533): run the layer in bf16 and hand back what the reference
            # would (fp16 out_proj output, fp16 y_ssm / states), so GradScaler and the fp16 callers keep working
            with torch.autocast("cuda", dtype=torch.bfloat16):
                out, y_ssm, cache = self.forward(hidden_states, attention_mask, position_ids, past_key_value, output_attentions, use_cache)
            h16 = lambda t: t.to(torch.float16) if (t is not None and t.dtype == torch.bfloat16) else t
            return h16(out), h16(y_ssm), (tuple(h16(c) for c in cache) if cache is not None else None)
        self.use_cache = use_cache
        if hidden_states.dtype == torch.float16:
            hidden_states = hidden_states.to(torch.bfloat16 if ac is not None else torch.float32)
        B, L, _ = hidden_states.shape
        Di, R, Kc, H = self.d_inner, self.dt_rank, self.conv_kernel_size, self.num_heads
        # fp32 activations without autocast: fp32-accurate GEMMs (3-product bf16 split); everything else runs the bf16 kernels
        precise = hidden_states.dtype == torch.float32 and ac is None
        conv_prev, h_prev = (past_key_value if past_key_value is not None else (None, None))
        cached = conv_prev is not None and use_cache and conv_prev.shape[1] == Di and conv_prev.shape[2] == Kc - 1
        recurrent = not (self.training and not use_cache)                     # :388-393
        # in_proj_x | in_proj_z as one GEMM: [xp | z] rows                     # :366-367
        xz = ops.linear(hidden_states, [self.in_proj_x.weight, self.in_proj_z.weight], precise=precise)
        if not (cached or use_cache or output_attentions) and self.scan_mode in (None, _lib.SCAN_ROUNDS):
            # the hot path (training, plain evaluation): conv + SiLU, fused parameter projection and scan as one autograd node
            y = ops.ssm_core(xz, self.conv1d.weight, self.conv1d.bias, self.x_param_proj.weight, self.dt_proj_head.weight,
                             self.dt_proj_head.bias, self.A_log, self.D, precise)
            return ops.linear(y, self.out_proj.weight, precise=precise), None, None       # :397
        # general path: cached decoding (:369-373, :391-393, :398-400), output_attentions, explicit scan schedules
        xp, z = xz[..., :Di], xz[..., Di:]
        x_seq = xp
        if cached:
            x_seq = torch.cat([conv_prev.transpose(1, 2).to(xp.dtype), xp], dim=1)      # :369-371 (state goes in FRONT)
        conv_state = x_seq[:, -(Kc - 1):, :].transpose(1, 2).detach() if use_cache else None   # :372
        # the reference convolves the (possibly state-prefixed) sequence and keeps the FIRST L outputs (:373)
        xa = ops.causal_conv1d_silu(x_seq, self.conv1d.weight, self.conv1d.bias)
        if x_seq.shape[1] != L:
            xa = xa[:, :L].contiguous()
        h0 = h_prev if (recurrent and use_cache and h_prev is not None) else None
        # x_param_proj with dt_proj_head folded in: one GEMM writes [dt (no bias) | pad | B | C] rows  (:376-383)
        wcat = ops.dt_compose(self.x_param_proj.weight, self.dt_proj_head.weight, precise)
        prm = ops.linear(xa, wcat, precise=precise)
        if self.scan_mode in (None, _lib.SCAN_ROUNDS):
            y, y_ssm, h_last = ops.selective_scan_fused(xa, prm, self.dt_proj_head.bias, z, self.A_log, self.D, H, h0=h0,
                                                        want_yssm=output_attentions, want_hlast=use_cache)
        else:           # the older schedules take separate, contiguous dt and [B | C] tensors
            Hp = prm.shape[-1] - 2 * Di
            dlog = (prm[..., :H] + self.dt_proj_head.bias.to(prm.dtype)).contiguous()
            y, y_ssm, h_last = ops.selective_scan(xa, dlog, prm[..., Hp:].contiguous(), z.contiguous(), self.A_log, self.D, h0=h0,
                                                  want_yssm=output_attentions, want_hlast=use_cache, mode=self.scan_mode)
        out = ops.linear(y, self.out_proj.weight, precise=precise)            # :397
        cache = None
        if use_cache:
            cache = (conv_state, h_last.view(B, self.num_heads, self.d_state).to(xa.dtype))      # :398-400
        return out, (y_ssm if output_attentions else None), cache


# ================================================================================================
# MoE layer
# ================================================================================================
# The router forward (csrc/moe_router.cu, ab_moe_router_fwd) keeps the router weight, its bias, the per-warp aux sums of
# its 8 warps and the LayerNorm affine in dynamic shared memory, all fp32.  An sm_100 block can opt in to at most 227 KB.
ROUTER_SMEM_LIMIT = 232448


def router_smem_bytes(E: int, Dm: int) -> int:
    """Dynamic shared memory of the router forward: (E*Dm + 32 + 8*(2E+1) + 2*Dm) floats."""
    return (E * Dm + 32 + 8 * (2 * E + 1) + 2 * Dm) * 4


def router_max_hidden(E: int) -> int:
    """Largest hidden size (a multiple of 8) whose router forward fits in ROUTER_SMEM_LIMIT for E experts."""
    return (ROUTER_SMEM_LIMIT // 4 - 32 - 8 * (2 * E + 1)) // (E + 2) // 8 * 8


class AdaptiveExpertSystem(nn.Module):
    """B200-native AdaptiveExpertSystem (core.py:403-607).

    Expert parameters are stored stacked ([E, ...]) so that the grouped GEMM reads them in place; the
    ``state_dict`` is translated to / from the reference's per-expert keys (``experts.{e}.0.weight`` ...
    ``experts.{e}.4.bias``) so reference checkpoints load with ``strict=True`` and vice versa.
    With ``ep_group`` (a torch.distributed process group) experts are sharded across ranks; see ep.py."""

    _STACKED = {"expert_ln_weight": "0.weight", "expert_ln_bias": "0.bias", "expert_w1": "1.weight",
                "expert_b1": "1.bias", "expert_w2": "4.weight", "expert_b2": "4.bias"}

    def __init__(self, config, activation_function_override: Optional[str] = None, ep_group=None):
        super().__init__()
        self.config = config
        self.hidden_size = config.hidden_size
        self.intermediate_size = config.intermediate_size
        self.num_experts = config.num_experts
        self.experts_per_token = config.experts_per_token
        self.ep_group = ep_group
        self.router = None
        self.w_noise = None
        g = lambda k, d: getattr(config, k, d)
        if self.num_experts <= 0:                                             # core.py:412-427 passthrough
            self.use_noisy_top_k_routing = self.use_expert_capacity_limit = self.use_expert_dropout = False
            self.use_router_z_loss = self.use_load_balancing_loss = False
            self.load_balancing_loss_coef = self.router_z_loss_coef = self.expert_dropout_prob = self.noisy_routing_alpha = 0.0
            return
        E, Dm, I = self.num_experts, self.hidden_size, self.intermediate_size
        # limits of the kernels (the reference has none): say so here, not at the first forward
        if E > 32 or self.experts_per_token > 8:
            raise ValueError(f"the B200 MoE kernels support num_experts <= 32 and experts_per_token <= 8 (got {E}, {self.experts_per_token})")
        if Dm % 8 or I % 8:
            raise ValueError(f"hidden_size ({Dm}) and intermediate_size ({I}) must be multiples of 8 (16-byte rows for TMA)")
        if router_smem_bytes(E, Dm) > ROUTER_SMEM_LIMIT:
            raise ValueError(f"the B200 router kernels stage the {E} x {Dm} router weight in shared memory: "
                             f"{router_smem_bytes(E, Dm)} bytes exceed the {ROUTER_SMEM_LIMIT} a block can hold, so with "
                             f"{E} experts hidden_size must be <= {router_max_hidden(E)}")
        if not 0.0 <= float(g("hidden_dropout_prob", 0.0)) < 1.0:
            raise ValueError("hidden_dropout_prob must be in [0, 1)")
        self.eps = config.layer_norm_eps
        self.router_norm = nn.LayerNorm(Dm, eps=self.eps)
        self.router = nn.Linear(Dm, E)
        act = activation_function_override if activation_function_override is not None else g("hidden_act", "gelu")
        self.act_name = act if act in _lib.ACT else "gelu"                    # core.py:463-468 (unknown -> GELU)
        self.hidden_dropout_prob = float(g("hidden_dropout_prob", 0.0))
        self.ep_world = ep_group.size() if ep_group is not None else 1
        self.ep_rank = ep_group.rank() if ep_group is not None else 0
        if E % self.ep_world:
            raise ValueError(f"num_experts ({E}) must be divisible by the expert-parallel world size ({self.ep_world})")
        El = E // self.ep_world
        self.local_experts = El
        self.expert_ln_weight = nn.Parameter(torch.ones(El, Dm))
        self.expert_ln_bias = nn.Parameter(torch.zeros(El, Dm))
        self.expert_w1 = nn.Parameter(torch.empty(El, I, Dm))
        self.expert_b1 = nn.Parameter(torch.empty(El, I))
        self.expert_w2 = nn.Parameter(torch.empty(El, Dm, I))
        self.expert_b2 = nn.Parameter(torch.empty(El, Dm))
        for e in range(El):                                                   # nn.Linear default init per expert
            nn.init.kaiming_uniform_(self.expert_w1[e], a=math.sqrt(5))
            nn.init.uniform_(self.expert_b1[e], -1 / math.sqrt(Dm), 1 / math.sqrt(Dm))
            nn.init.kaiming_uniform_(self.expert_w2[e], a=math.sqrt(5))
            nn.init.uniform_(self.expert_b2[e], -1 / math.sqrt(I), 1 / math.sqrt(I))
        if g("use_noisy_top_k_routing", True):
            self.w_noise = nn.Parameter(torch.zeros(E))
        self.load_balancing_loss_coef = g("load_balancing_loss_coef", 0.01)
        self.expert_capacity_factor = g("expert_capacity_factor", 1.25)
        self.router_z_loss_coef = g("router_z_loss_coef", 0.001)
        self.noisy_routing_alpha = g("noisy_routing_alpha", 0.1)
        self.expert_dropout_prob = g("expert_dropout_prob", 0.1)
        self.use_noisy_top_k_routing = g("use_noisy_top_k_routing", True)
        self.use_expert_capacity_limit = g("use_expert_capacity_limit", True)
        self.use_expert_dropout = g("use_expert_dropout", True)
        self.use_router_z_loss = g("use_router_z_loss", True)
        self.use_load_balancing_loss = g("use_load_balancing_loss", True)
        self.last_counts: Optional[torch.Tensor] = None       # expert_token_counts_post_capacity of the last call (int32 [E])
        self.last_routing = None
        # Under torch.autocast the reference's router Linear runs in the autocast dtype (core.py:482), so its top-k sees
        # logits rounded to bf16 / fp16.  True (default): round the same way, i.e. pick the experts the reference picks in
        # that mode; False: route on fp32 logits whatever the autocast state (what the fp32 oracle does).
        self.router_autocast_rounding = True
        self._register_state_dict_hook(self._to_reference_keys)
        self._register_load_state_dict_pre_hook(self._from_reference_keys)

    # ---- state_dict translation (reference keys: experts.{e}.{0,1,4}.{weight,bias}) ----
    @staticmethod
    def _to_reference_keys(module, state_dict, prefix, local_metadata):
        if module.num_experts <= 0:
            return state_dict
        base = module.ep_rank * module.local_experts
        stacked = {suffix: state_dict.pop(prefix + name) for name, suffix in module._STACKED.items()}
        for e in range(module.local_experts):                 # expert-major, like the reference's ModuleList
            for suffix, t in stacked.items():
                state_dict[f"{prefix}experts.{base + e}.{suffix}"] = t[e]
        return state_dict

    def _from_reference_keys(self, state_dict, prefix, local_metadata, strict, missing_keys, unexpected_keys, error_msgs):
        if self.num_experts <= 0:
            return
        base = self.ep_rank * self.local_experts
        for name, suffix in self._STACKED.items():
            if prefix + name in state_dict:
                continue
            keys = [f"{prefix}experts.{base + e}.{suffix}" for e in range(self.local_experts)]
            if all(k in state_dict for k in keys):
                state_dict[prefix + name] = torch.stack([state_dict[k] for k in keys])
        # the per-expert keys have been folded into the stacked tensors (or belong to other ranks' experts under EP): remove
        # exactly those - a well-formed key of an expert in [0, num_experts) - and leave anything else under "experts." in
        # place, so that malformed or out-of-range keys still surface as unexpected keys with strict=True
        known = set(self._STACKED.values())
        for k in [k for k in state_dict if k.startswith(prefix + "experts.")]:
            parts = k[len(prefix) + len("experts."):].split(".", 1)
            if len(parts) == 2 and parts[0].isdigit() and int(parts[0]) < self.num_experts and parts[1] in known:
                del state_dict[k]

    # ---- hooks the parity tests use to feed both sides the same random numbers ----
    def _draw_noise(self, S: int, E: int, device) -> torch.Tensor:
        """The standard-normal draw of core.py:487 (torch.randn_like on the fp32 logits)."""
        return torch.randn(S, E, device=device, dtype=torch.float32)

    def _draw_active_mask(self, device) -> Optional[torch.Tensor]:
        """Whole-expert dropout mask of core.py:514-521 (None = all experts active)."""
        E = self.num_experts
        if not (self.use_expert_dropout and self.training and self.expert_dropout_prob > 0):
            return None
        ndrop = math.floor(E * self.expert_dropout_prob)
        if ndrop >= E:
            ndrop = E - 1
        if ndrop <= 0:
            return None
        perm = torch.randperm(E, device=device)
        active = torch.ones(E, dtype=torch.int32, device=device)
        active[perm[:ndrop]] = 0
        return active

    def forward(self, hidden_states: torch.Tensor, residual: Optional[torch.Tensor] = None, output_dropout_p: float = 0.0):
        """forward(hidden_states) is the reference's contract (core.py:470).  The two optional arguments let a caller hand
        in its residual and output-dropout probability (core.py:918-919): the result is then
        residual + Dropout(p)(moe(hidden_states)), computed inside the combine kernel instead of by two more passes."""
        zero = lambda: torch.tensor(0.0, device=hidden_states.device, dtype=hidden_states.dtype)
        if self.num_experts <= 0 or self.router is None:
            out = hidden_states
            if residual is not None:
                out = residual + F.dropout(out, output_dropout_p, self.training)
            return out, zero(), zero()                                        # core.py:474-475
        _lib.ensure_device(hidden_states.device)
        ac = _autocast_dtype()
        B, L, Dm = hidden_states.shape
        S, E, K = B * L, self.num_experts, self.experts_per_token
        x2 = hidden_states.reshape(S, Dm)
        training = self.training
        noise = noise_scale = None
        if self.use_noisy_top_k_routing and training and self.w_noise is not None:          # core.py:485-488
            noise_scale = F.softplus(self.w_noise.float()) * self.noisy_routing_alpha
            noise = self._draw_noise(S, E, x2.device)
        cap = ops.moe_capacity(S, E, self.expert_capacity_factor, training, self.use_expert_capacity_limit)
        cfg = dict(K=K, eps=self.eps, act=_lib.ACT[self.act_name], training=training, cap=cap,
                   lb_coef=self.load_balancing_loss_coef if self.use_load_balancing_loss else 0.0,
                   rz_coef=self.router_z_loss_coef if self.use_router_z_loss else 0.0,
                   active=self._draw_active_mask(x2.device), drop_p=self.hidden_dropout_prob,
                   precise=(x2.dtype == torch.float32 and ac is None),
                   # the reference's router Linear runs in the autocast dtype (core.py:482): pick the experts it picks
                   quant={torch.bfloat16: _lib.ROUTER_BF16, torch.float16: _lib.ROUTER_FP16}.get(ac, _lib.ROUTER_EXACT)
                   if self.router_autocast_rounding else _lib.ROUTER_EXACT)
        if self.ep_world > 1:
            from . import ep
            cfg["out_drop_p"] = float(output_dropout_p)
            out, lb, rz, counts = ep.moe_experts_ep(self, x2, noise, noise_scale, cfg, res=residual.reshape(S, Dm) if residual is not None else None)
        else:
            cfg["out_drop_p"] = float(output_dropout_p)
            out, lb, rz, counts = ops.moe_experts(x2, self.router_norm.weight, self.router_norm.bias, self.router.weight,
                                                  self.router.bias, noise, noise_scale, self.expert_ln_weight,
                                                  self.expert_ln_bias, self.expert_w1, self.expert_b1, self.expert_w2,
                                                  self.expert_b2, cfg, res=residual.reshape(S, Dm) if residual is not None else None)
        self.last_counts = counts
        self.last_routing = cfg.get("_routing")          # (idx int32 [S,K], row_of int32 [S,K], -1 = dropped by the capacity limit)
        return out.reshape(B, L, Dm), lb, rz


# ================================================================================================
# the callers (boundary; kept as plain PyTorch like the reference's ApertisAttention / ApertisFeedForward)
# ================================================================================================
def _require_layernorm(config):
    """The fused wrappers implement the reference's default pre-norm (nn.LayerNorm, core.py:668-669, 846-847).  With
    use_rmsnorm=True the reference builds RMSNorm (core.py:666-667, 844-845): refuse instead of silently normalising
    differently; patch_apertis_model() keeps the reference's own wrappers (and therefore its RMSNorm) and still works."""
    if getattr(config, "use_rmsnorm", False):
        raise NotImplementedError("ApertisLayerB200 implements the LayerNorm pre-norm only; for use_rmsnorm=True keep the reference "
                                  "wrappers and swap the hot-path modules with patch_apertis_model()")


class _AttentionWrapper(nn.Module):
    """ApertisAttention for attention_type == 'selective_ssm' (core.py:639-704, 836-838)."""

    def __init__(self, config):
        super().__init__()
        _require_layernorm(config)
        self.config = config
        self.attention_mechanism_impl = SelectiveLinearAttention(config)
        self.pre_norm = nn.LayerNorm(config.hidden_size, eps=config.layer_norm_eps)
        self.output_dropout = nn.Dropout(config.hidden_dropout_prob)

    def forward(self, hidden_s, att_mask=None, pos_ids=None, past_kv=None, output_att=False, use_c=False):
        # under autocast the projections consume bf16: emit the normalised rows in that type directly (same rounding
        # point as the reference's fp32 LayerNorm followed by the autocast cast inside nn.Linear)
        ac = _compute_dtype(_autocast_dtype())
        normed, skip = ops.layer_norm_skip(hidden_s, self.pre_norm.weight, self.pre_norm.bias, self.pre_norm.eps,
                                           out_dtype=ac if (ac is not None and hidden_s.dtype == torch.float32) else None)
        out, proxy, cache = self.attention_mechanism_impl(normed, attention_mask=att_mask, position_ids=pos_ids,
                                                          past_key_value=past_kv, output_attentions=output_att, use_cache=use_c)
        return ops.dropout_add(out, skip, self.output_dropout.p, self.training), proxy, cache


class _FeedForwardWrapper(nn.Module):
    """ApertisFeedForward with the expert system (core.py:840-923)."""

    def __init__(self, config, ep_group=None):
        super().__init__()
        _require_layernorm(config)
        self.config = config
        self.pre_norm = nn.LayerNorm(config.hidden_size, eps=config.layer_norm_eps)
        self.ffn = AdaptiveExpertSystem(config, activation_function_override=config.hidden_act, ep_group=ep_group)
        self.is_expert_system = True
        self.output_dropout = nn.Dropout(config.hidden_dropout_prob)

    def forward(self, hidden_s):
        normed, skip = ops.layer_norm_skip(hidden_s, self.pre_norm.weight, self.pre_norm.bias, self.pre_norm.eps)
        # output dropout + residual add (core.py:918-919) happen inside the MoE's combine kernel
        return self.ffn(normed, residual=skip, output_dropout_p=self.output_dropout.p)


class ApertisLayerB200(nn.Module):
    """ApertisLayer (core.py:995-1018) built from the B200 modules; state_dict keys equal the reference layer's."""

    def __init__(self, config, ep_group=None):
        super().__init__()
        self.config = config
        self.attention = _AttentionWrapper(config)
        self.feed_forward = _FeedForwardWrapper(config, ep_group=ep_group)

    def forward(self, hidden_s, att_mask=None, pos_ids=None, past_kv=None, output_att=False, use_c=False):
        att_out, att_w, cache = self.attention(hidden_s, att_mask, pos_ids, past_kv, output_att, use_c)
        out, lb, rz = self.feed_forward(att_out)
        return out, att_w, cache, lb, rz


def _causal_lm_forward(self, input_ids=None, attention_mask=None, position_ids=None, past_key_values=None, inputs_embeds=None,
                       pixel_values=None, labels=None, use_cache=None, output_attentions=None, output_hidden_states=None):
    """ApertisForCausalLM.forward (core.py:1361-1473) with the language-model head and the shifted cross-entropy on the
    B200 kernels (SURVEY.md 8(f) row 4): same arguments, same return tuple.  Installed on a model instance by
    patch_apertis_model(fuse_lm_head=True); shapes the fused path does not cover (no labels, a vocabulary that is not a
    multiple of 8, label / logit lengths that differ, sequences of one token) go through the reference's own forward."""
    ref_forward = type(self).forward
    kw = dict(input_ids=input_ids, attention_mask=attention_mask, position_ids=position_ids, past_key_values=past_key_values,
              inputs_embeds=inputs_embeds, pixel_values=pixel_values, labels=labels, use_cache=use_cache,
              output_attentions=output_attentions, output_hidden_states=output_hidden_states)
    V = self.lm_head.weight.shape[0]
    if labels is None or V % 8 or getattr(self.lm_head, "bias", None) is not None:
        return ref_forward(self, **kw)
    model_outputs = self.model(**{k: v for k, v in kw.items() if k != "labels"})
    hidden = model_outputs[0]
    text_hidden = hidden
    if self.config.multimodal and pixel_values is not None and past_key_values is None and input_ids is not None:   # core.py:1398-1405
        start = hidden.shape[1] - input_ids.shape[1]
        if start >= 0:
            text_hidden = hidden[:, start:, :]
    if text_hidden.shape[1] != labels.shape[1] or text_hidden.shape[1] < 2 or not text_hidden.is_cuda:
        return ref_forward(self, **kw)
    ac = _autocast_dtype()
    precise = text_hidden.dtype == torch.float32 and ac is None
    logits, loss = ops.lm_head_cross_entropy(text_hidden.contiguous(), self.lm_head.weight, labels, -100, precise)
    if ac == torch.float16:
        logits = logits.to(torch.float16)
    if model_outputs[4] is not None:                                # core.py:1449-1456: aux losses of the expert layers
        loss = loss + model_outputs[4]
    if model_outputs[5] is not None:
        loss = loss + model_outputs[5]
    return (loss, logits) + tuple(model_outputs[1:])


def patch_apertis_model(model: nn.Module, ep_group=None, fuse_lm_head: bool = False) -> nn.Module:
    """Swaps the B200 modules into a reference ApertisModel / ApertisForCausalLM in place.

    fuse_lm_head=True additionally routes ApertisForCausalLM's language-model head and shifted cross-entropy
    (core.py:1412-1460) through the B200 kernels (_causal_lm_forward): the tied embedding matrix is used as it is.

    For every layer: ``attention.attention_mechanism_impl`` (core.py:650) is replaced by a
    SelectiveLinearAttention that adopts the SAME Parameter objects, and ``feed_forward.ffn`` (core.py:861)
    by an AdaptiveExpertSystem whose stacked parameters are filled from the per-expert modules (new Parameter
    objects, in the device and dtype of the old ones): patch BEFORE building the optimizer or wrapping in DDP."""
    layers = model.model.layers if hasattr(model, "model") and hasattr(model.model, "layers") else model.layers
    for layer in layers:
        att = layer.attention
        old = getattr(att, "attention_mechanism_impl", None)
        if old is not None and type(old).__name__ == "SelectiveLinearAttention" and not isinstance(old, SelectiveLinearAttention):
            new = SelectiveLinearAttention(att.config)
            for name, prm in old.named_parameters():
                mod, _, leaf = name.rpartition(".")
                setattr(new.get_submodule(mod) if mod else new, leaf, prm)
            new.train(old.training)
            att.attention_mechanism_impl = new
        ff = layer.feed_forward
        oldf = getattr(ff, "ffn", None)
        if getattr(ff, "is_expert_system", False) and type(oldf).__name__ == "AdaptiveExpertSystem" \
                and not isinstance(oldf, AdaptiveExpertSystem):
            newf = AdaptiveExpertSystem(ff.config, activation_function_override=ff.config.hidden_act, ep_group=ep_group)
            ref_p = next(oldf.parameters())
            newf.to(device=ref_p.device, dtype=ref_p.dtype)
            newf.load_state_dict(oldf.state_dict(), strict=True)
            newf.train(oldf.training)
            ff.ffn = newf
    if fuse_lm_head and hasattr(model, "lm_head") and hasattr(model, "model"):
        import types
        model.forward = types.MethodType(_causal_lm_forward, model)
    return model
