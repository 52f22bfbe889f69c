"""patch_apertis_model against the UNMODIFIED reference model (baseline/_ref, installed by __graft_entry__.build() where a
reference checkout is at hand; the file skips without it).  CPU-only: checks the module swap, parameter adoption and
state_dict compatibility; the numerical parity of the swapped modules is what tests/test_gpu_modules.py covers through
the golden vectors."""
import pytest
import torch

from baseline import ref_loader

pytestmark = pytest.mark.skipif(not ref_loader.available(), reason="baseline/_ref (the installed reference) is absent")


def _ref_model():
    core = ref_loader.load_core()
    cfg = core.ApertisConfig(hidden_size=64, num_attention_heads=4, intermediate_size=128, num_hidden_layers=2,
                             attention_type="selective_ssm", use_expert_system=True, num_experts=4, experts_per_token=2,
                             vocab_size=97, hidden_dropout_prob=0.0, attention_probs_dropout_prob=0.0)
    torch.manual_seed(0)
    return core.ApertisForCausalLM(cfg)


def test_patch_swaps_modules_and_keeps_state_dict():
    import apertis_llm_b200 as ab
    model = _ref_model()
    before = {k: v.clone() for k, v in model.state_dict().items()}
    ssm_params = {n: p for n, p in model.named_parameters() if "attention_mechanism_impl" in n}
    ab.patch_apertis_model(model)
    for layer in model.model.layers:
        assert isinstance(layer.attention.attention_mechanism_impl, ab.SelectiveLinearAttention)
        assert isinstance(layer.feed_forward.ffn, ab.AdaptiveExpertSystem)
    # the SSM adopts the very same Parameter objects (optimizer state and tied references stay valid)
    after_params = dict(model.named_parameters())
    for n, p in ssm_params.items():
        assert after_params[n] is p, n
    # checkpoints are interchangeable: same keys, same shapes, same values
    after = model.state_dict()
    assert list(after.keys()) == list(before.keys())
    for k, v in before.items():
        assert after[k].shape == v.shape and torch.equal(after[k], v), k
    # and a reference checkpoint loads into the patched model (strict)
    model.load_state_dict(before, strict=True)
    # patching twice is a no-op
    ab.patch_apertis_model(model)
    assert list(model.state_dict().keys()) == list(before.keys())


def test_patched_model_refuses_to_run_on_cpu():
    import apertis_llm_b200 as ab
    model = ab.patch_apertis_model(_ref_model())
    with pytest.raises(RuntimeError, match="no CPU fallback|CUDA"):
        model(input_ids=torch.randint(0, 97, (1, 8)))


def test_fuse_lm_head_installs_the_reference_shaped_forward():
    """patch_apertis_model(fuse_lm_head=True) binds a forward with the reference's argument list on the instance; the state
    dict (tied embeddings included) is untouched, and on a CPU model the fused path still refuses to run."""
    import inspect
    import apertis_llm_b200 as ab
    from apertis_llm_b200 import modules
    model = _ref_model()
    keys = list(model.state_dict().keys())
    ref_params = list(inspect.signature(type(model).forward).parameters)[1:]
    ab.patch_apertis_model(model, fuse_lm_head=True)
    assert model.forward.__func__ is modules._causal_lm_forward
    assert list(inspect.signature(model.forward).parameters) == ref_params
    assert list(model.state_dict().keys()) == keys
    assert model.lm_head.weight is model.model.token_embeddings.weight        # still tied
    with pytest.raises(RuntimeError, match="no CPU fallback|CUDA"):
        ids = torch.randint(0, 97, (1, 8))
        model(input_ids=ids, labels=ids)
