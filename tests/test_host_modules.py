"""CPU: the host-side mirror of the reference's quant package -- names, constructor, buffers,
state_dict layout, module surgery, exceptions.  No kernel is launched."""
import math

import numpy as np
import pytest
import torch
import torch.nn as nn

import quant
import utils


def test_public_names_match_reference_init():
    # quant/__init__.py:1-5 of the reference, plus the older make_quant alias
    for name in ('Quantizer', 'QuantLlamaAttention', 'make_quant_attn', 'QuantLlamaMLP', 'make_fused_mlp', 'autotune_warmup_fused', 'QuantLinear',
                 'make_quant_linear', 'autotune_warmup_linear', 'TritonLlamaRMSNorm', 'make_quant_norm', 'make_quant'):
        assert hasattr(quant, name), name
    assert quant.make_quant is quant.make_quant_linear
    assert utils.DEV == torch.device('cuda:0')


@pytest.mark.parametrize('bits', [2, 3, 4, 8])
@pytest.mark.parametrize('groupsize', [-1, 32, 128])
def test_quantlinear_buffers(bits, groupsize):
    K, N = 256, 96
    ql = quant.QuantLinear(bits, groupsize, K, N, True)
    gs = K if groupsize == -1 else groupsize
    G = math.ceil(K / gs)
    sd = ql.state_dict()
    assert set(sd) == {'qweight', 'qzeros', 'scales', 'g_idx', 'bias'}
    assert sd['qweight'].shape == (K // 32 * bits, N) and sd['qweight'].dtype == torch.int32
    assert sd['qzeros'].shape == (G, N // 32 * bits) and sd['qzeros'].dtype == torch.int32
    assert sd['scales'].shape == (G, N) and sd['scales'].dtype == torch.float16
    assert sd['g_idx'].dtype == torch.int32 and torch.equal(sd['g_idx'], (torch.arange(K) // gs).int())
    assert sd['bias'].shape == (N, ) and sd['bias'].dtype == torch.float16
    assert (ql.maxq, ql.groupsize, ql.infeatures, ql.outfeatures) == (2**bits - 1, gs, K, N)
    assert not list(ql.parameters())  # buffers, not Parameters (quant_linear.py:316-321)
    assert quant.QuantLinear(bits, groupsize, K, N, False).bias is None


@pytest.mark.parametrize('bits', [1, 5, 6, 16])
def test_unsupported_bits_raise_not_implemented(bits):
    with pytest.raises(NotImplementedError):
        quant.QuantLinear(bits, 128, 128, 32, False)


def test_forward_on_cpu_fails_loudly():
    ql = quant.QuantLinear(4, 128, 128, 32, False)
    with pytest.raises(ValueError, match='cuda'):
        ql(torch.zeros(1, 128, dtype=torch.float16))


def test_golden_checkpoint_loads_into_quantlinear(golden_cases):
    d = golden_cases['b4_g32_bias']
    ql = quant.QuantLinear(4, 32, int(d['K']), int(d['N']), True)
    sd = {k: torch.from_numpy(d[s]) for k, s in (('qweight', 'qweight'), ('qzeros', 'qzeros'), ('scales', 'scales_h'), ('g_idx', 'g_idx'), ('bias', 'bias_h'))}
    ql.load_state_dict(sd, strict=True)
    assert torch.equal(ql.qweight, sd['qweight'])


class _Toy(nn.Module):

    def __init__(self):
        super().__init__()
        self.a = nn.Linear(64, 32, bias=False)
        self.blk = nn.Sequential(nn.Linear(32, 64, bias=True), nn.ReLU(), nn.Linear(64, 32))
        self.head = nn.Linear(32, 8)


def test_find_layers_and_make_quant_linear():
    m = _Toy()
    layers = utils.find_layers(m)
    assert set(layers) == {'a', 'blk.0', 'blk.2', 'head'}
    del layers['head']
    quant.make_quant_linear(m, layers, 4, 32)
    assert isinstance(m.a, quant.QuantLinear) and m.a.bias is None
    assert isinstance(m.blk[0], quant.QuantLinear) and m.blk[0].bias is not None
    assert isinstance(m.head, nn.Linear)
    assert (m.blk[2].infeatures, m.blk[2].outfeatures) == (64, 32)
    quant.make_quant_linear(m, layers, 4, 32)  # idempotent


def _tiny_llama():
    from transformers import LlamaConfig, LlamaForCausalLM
    cfg = LlamaConfig(hidden_size=64, intermediate_size=96, num_hidden_layers=2, num_attention_heads=2, num_key_value_heads=2, vocab_size=128,
                      max_position_embeddings=64)
    torch.manual_seed(0)
    return LlamaForCausalLM(cfg).half().eval()


def test_load_quant_style_surgery_on_hf_llama():
    """The sequence of quant.* calls made by the reference's load_quant (llama_inference.py:45-68)."""
    model = _tiny_llama()
    layers = utils.find_layers(model)
    layers.pop('lm_head')
    quant.make_quant_linear(model, layers, 4, 32)
    sd_keys = set(model.state_dict())
    assert 'model.layers.0.self_attn.q_proj.qweight' in sd_keys and 'model.layers.1.mlp.down_proj.g_idx' in sd_keys
    assert 'lm_head.weight' in sd_keys
    quant.make_quant_attn(model)
    quant.make_quant_norm(model)
    quant.make_fused_mlp(model)
    l0 = model.model.layers[0]
    assert isinstance(l0.self_attn, quant.QuantLlamaAttention)
    assert l0.self_attn.qkv_proj.qweight.shape == (64 // 8, 3 * 64)
    assert l0.self_attn.qkv_proj.qzeros.shape == (2, 3 * 64 // 8)
    assert l0.self_attn.qkv_proj.g_idx.shape == (64, )
    assert (l0.self_attn.num_heads, l0.self_attn.head_dim, l0.self_attn.layer_idx) == (2, 32, 0)
    assert isinstance(l0.mlp, quant.QuantLlamaMLP) and l0.mlp.intermediate_size == 96
    assert l0.mlp.gate_proj_qweight.shape == (8, 96) and isinstance(l0.mlp.down_proj, quant.QuantLinear)
    assert isinstance(l0.input_layernorm, quant.TritonLlamaRMSNorm) and isinstance(model.model.norm, quant.TritonLlamaRMSNorm)
    assert quant.autotune_warmup_linear(model) == 0 and quant.autotune_warmup_fused(model) == 0  # nothing on the GPU yet


def test_load_quant_recipe_routes_checkpoint_tensors(tmp_path):
    """A GPTQ checkpoint saved from a make_quant_linear model and loaded the way llama_inference.load_quant loads one (fresh fp16 model,
    make_quant_linear without lm_head, non-strict load, then attention / norm / MLP fusion and warm-up): every tensor arrives where the
    kernels read it."""
    from transformers import LlamaConfig, LlamaForCausalLM
    cfg = LlamaConfig(hidden_size=256, intermediate_size=768, num_hidden_layers=2, num_attention_heads=2, num_key_value_heads=2, vocab_size=320,
                      max_position_embeddings=64, rms_norm_eps=1e-6)

    def quant_model():
        torch.set_default_dtype(torch.half)
        try:
            m = LlamaForCausalLM(cfg).eval()
        finally:
            torch.set_default_dtype(torch.float)
        layers = utils.find_layers(m)
        del layers['lm_head']
        quant.make_quant_linear(m, layers, 4, 128)
        return m

    src = quant_model()
    g = torch.Generator().manual_seed(0)
    for m in src.modules():
        if isinstance(m, quant.QuantLinear):
            m.qweight.copy_(torch.randint(-2**31, 2**31 - 1, m.qweight.shape, generator=g, dtype=torch.int64).to(torch.int32))
            m.qzeros.copy_(torch.randint(-2**31, 2**31 - 1, m.qzeros.shape, generator=g, dtype=torch.int64).to(torch.int32))
            m.scales.copy_((torch.rand(m.scales.shape, generator=g) * 1e-2 + 1e-3).half())
    sd = src.state_dict()
    assert sd['model.layers.0.self_attn.q_proj.qweight'].shape == (256 // 8, 256) and sd['model.layers.0.mlp.down_proj.qzeros'].dtype == torch.int32
    ckpt = tmp_path / 'tiny-4bit-128g.pt'
    torch.save(sd, ckpt)

    model = quant_model()
    model.load_state_dict(torch.load(ckpt), strict=False)
    quant.make_quant_attn(model)
    quant.make_quant_norm(model)
    quant.make_fused_mlp(model)
    quant.autotune_warmup_linear(model, transpose=False)
    quant.autotune_warmup_fused(model)
    layer = model.model.layers[0]
    assert isinstance(layer.self_attn, quant.QuantLlamaAttention) and isinstance(layer.mlp, quant.QuantLlamaMLP)
    assert isinstance(layer.input_layernorm, quant.TritonLlamaRMSNorm) and isinstance(model.model.norm, quant.TritonLlamaRMSNorm)
    # fused q|k|v along N, gate/up buffers of the fused MLP, down_proj untouched, lm_head never quantized
    q, k, v = (sd[f'model.layers.0.self_attn.{n}_proj.qweight'] for n in 'qkv')
    assert torch.equal(layer.self_attn.qkv_proj.qweight, torch.cat([q, k, v], dim=1))
    assert torch.equal(layer.mlp.gate_proj_qweight, sd['model.layers.0.mlp.gate_proj.qweight'])
    assert torch.equal(layer.mlp.up_proj_scales, sd['model.layers.0.mlp.up_proj.scales'])
    assert torch.equal(layer.mlp.down_proj.qzeros, sd['model.layers.0.mlp.down_proj.qzeros'])
    assert torch.equal(model.lm_head.weight, sd['lm_head.weight'])


def test_fuse_qkv_rejects_mismatched_act_order():
    from quant.fused_attn import fuse_qkv
    q, k, v = (quant.QuantLinear(4, 32, 64, 64, False) for _ in range(3))
    k.g_idx = k.g_idx.flip(0).contiguous()
    with pytest.raises(ValueError):
        fuse_qkv(q, k, v)


def test_attention_head_split_error():
    with pytest.raises(ValueError):
        quant.QuantLlamaAttention(100, 3, None, None)


def test_rmsnorm_width_limit():
    n = quant.TritonLlamaRMSNorm(torch.ones(40000, dtype=torch.float16))
    with pytest.raises(RuntimeError, match='64KB'):
        n(torch.zeros(1, 40000, dtype=torch.float16))


def test_quantizer_reproduces_reference_scale_zero(golden_cases):
    """Our Quantizer, configured as gptq.py:185-194, reproduces the reference Quantizer's outputs stored
    in the golden fixtures (scale, zero and the on-grid weights Q)."""
    for name, d in golden_cases.items():
        bits, K = int(d['bits']), int(d['K'])
        W, g_idx = torch.from_numpy(d['W']), torch.from_numpy(d['g_idx']).long()
        for g in range(d['scale'].shape[1]):
            cols = (g_idx == g).nonzero().flatten()
            q = quant.Quantizer()
            q.configure(bits, perchannel=True, sym=False, mse=False)
            q.find_params(W[:, cols], weight=True)
            assert np.array_equal(q.scale.flatten().numpy(), d['scale'][:, g]), name
            assert np.array_equal(q.zero.flatten().numpy(), d['zero'][:, g]), name
            assert np.array_equal(q.quantize(W[:, cols]).numpy(), d['Q'][:, cols.numpy()]), name


def test_quantizer_modes():
    x = torch.randn(8, 32, generator=torch.Generator().manual_seed(0))
    q = quant.Quantizer()
    q.configure(4, perchannel=True, sym=True, mse=True)
    q.find_params(x, weight=True)
    assert q.scale.shape == (8, 1) and q.ready() and q.enabled()
    y = q.quantize(x)
    assert (y - x).abs().max() <= q.scale.max()
    q2 = quant.Quantizer()
    q2.configure(8, perchannel=False, sym=False)
    q2.find_params(x, weight=True)
    assert q2.scale.shape == (8, 1) and torch.all(q2.scale == q2.scale[0])
