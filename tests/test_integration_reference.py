"""J1 - "AutoGPTQForCausalLM loads and runs unchanged": the B200 QuantLinear through the reference's OWN construction
path.

CPU part: replays what the reference's `modeling/_utils.py` did when it built this package's module, as recorded from the
unmodified original by tests/golden/make_golden_integration.py into tests/golden/ref_make_quant.json: the selection call
that `patch_auto_gptq()` answers, `make_quant`'s positional constructor calls (_utils.py:69-148) with `new_layer.device =
...; .to(device)`, then the name-keyed buffer fill (_base.py:1114-1121) on a tiny HF Llama; `autogptq_post_init`
(_utils.py:380-513) must not act on our QUANT_TYPE.

GPU part: the same construction sequence written out, a GPTQ checkpoint written with
`QuantLinear.pack` to safetensors and read back (also through `autogptq_b200.checkpoint`), logits and greedy decode
(reference tests/test_q4.py:1165-1222 compares generated text) against the same model holding the dequantised fp16
weights in plain nn.Linear."""
import json
import os
import sys
import types

import numpy as np
import pytest
import torch
import torch.nn as nn

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
LINEAR_NAMES = ("q_proj", "k_proj", "v_proj", "o_proj", "gate_proj", "up_proj", "down_proj")


def _tiny_llama(seed=0, hidden=256, inter=512, layers=2, heads=4, vocab=128):
    from transformers import LlamaConfig, LlamaForCausalLM

    torch.manual_seed(seed)
    cfg = LlamaConfig(vocab_size=vocab, hidden_size=hidden, intermediate_size=inter, num_hidden_layers=layers,
                      num_attention_heads=heads, num_key_value_heads=heads, max_position_embeddings=64,
                      tie_word_embeddings=False)
    return LlamaForCausalLM(cfg).eval()


def _quant_names(model):
    return [n for n, m in model.named_modules() if isinstance(m, nn.Linear) and n.split(".")[-1] in LINEAR_NAMES]


def _rtn_pack(model, group_size=128):
    """Round-to-nearest 4-bit quantisation of every decoder Linear, packed with QuantLinear.pack (the reference contract,
    qlinear_cuda_old.py:110-200).  Returns {name: packed module (CPU)} and {name: dequantised fp16 weight [N, K]}."""
    from autogptq_b200 import QuantLinear
    from oracle import w4a16_oracle as O

    packed, deq = {}, {}
    for name in _quant_names(model):
        lin = dict(model.named_modules())[name]
        W = lin.weight.data.float()                                  # [N, K]
        N, K = W.shape
        G = K // group_size
        Wg = W.reshape(N, G, group_size)
        wmax, wmin = Wg.amax(-1), Wg.amin(-1)
        scales = ((wmax - wmin).clamp(min=1e-5) / 15).half().float()      # [N, G], representable in fp16
        zeros = torch.round(-wmin / scales).clamp(0, 15)                  # [N, G]
        ql = QuantLinear(4, group_size, K, N, lin.bias is not None)
        half_lin = nn.Linear(K, N, bias=lin.bias is not None).half()
        half_lin.weight.data = W.half()
        ql.pack(half_lin, scales, zeros, None)
        packed[name] = ql
        deq[name] = torch.from_numpy(O.dequantize(ql.qweight.numpy(), ql.qzeros.numpy(), ql.scales.numpy(),
                                                  g_idx=ql.g_idx.numpy(), group_size=group_size, dtype=np.float16).T.copy())
    return packed, deq


def _stand_in_auto_gptq():
    """An importable `auto_gptq.modeling._utils` that binds `dynamically_import_QuantLinear` by name, as the original
    does at import time (_utils.py:17); returns it."""
    for pkg in ("auto_gptq", "auto_gptq.modeling"):
        sys.modules[pkg] = types.ModuleType(pkg)
        sys.modules[pkg].__path__ = []
    utils = types.ModuleType("auto_gptq.modeling._utils")
    utils.dynamically_import_QuantLinear = None
    sys.modules[utils.__name__] = utils
    return utils


def test_reference_make_quant_builds_and_fills_the_b200_module():
    import autogptq_b200
    from autogptq_b200 import QuantLinear

    with open(os.path.join(GOLDEN, "ref_make_quant.json")) as f:
        rec = json.load(f)
    model = _tiny_llama()
    packed, _ = _rtn_pack(model)
    names = _quant_names(model)
    assert [layer["name"] for layer in rec["layers"]] == names and len(names) == 14
    try:
        U = _stand_in_auto_gptq()
        assert "auto_gptq.modeling._utils" in autogptq_b200.patch_auto_gptq()
        # the selection make_quant made (backend flags as from_quantized passes them)
        assert rec["selections"] and all(U.dynamically_import_QuantLinear(**sel) is QuantLinear for sel in rec["selections"])
    finally:
        for name in list(sys.modules):
            if name == "auto_gptq" or name.startswith("auto_gptq."):
                del sys.modules[name]
    # make_quant's construction of every layer: positional ctor, `new_layer.device = ori_layer_device`, .to(), setattr
    for layer in rec["layers"]:
        kwargs = {k: getattr(torch, v.removeprefix("torch.")) if k == "weight_dtype" else v for k, v in layer["kwargs"].items()}
        new = QuantLinear(*layer["args"], **kwargs)
        new.device = torch.device(layer["device"])
        for args in layer["to"]:
            new = new.to(*(torch.device(a) for a in args))
        parent_name, _, child = layer["name"].rpartition(".")
        setattr(model.get_submodule(parent_name), child, new)
    mods = dict(model.named_modules())
    assert all(isinstance(mods[n], QuantLinear) for n in names)
    assert all(hasattr(mods[n], "device") for n in names)
    # name-keyed buffer fill (what accelerate.load_checkpoint_in_model does with the checkpoint keys, _base.py:1114-1121)
    sd = {f"{n}.{k}": v for n, q in packed.items() for k, v in q.state_dict().items()}
    missing, unexpected = model.load_state_dict(sd, strict=False)
    assert not unexpected and not [m for m in missing if any(x in m for x in ("qweight", "qzeros", "scales", "g_idx"))]
    for n in names:
        assert torch.equal(mods[n].qweight, packed[n].qweight) and torch.equal(mods[n].scales, packed[n].scales)
    # autogptq_post_init walks the modules by QUANT_TYPE (_utils.py:380-513): ours is none of those it handles
    assert rec["post_init_acts_on"] and QuantLinear.QUANT_TYPE not in rec["post_init_acts_on"]
    # no CPU fallback in the product: a forward without a GPU fails loudly
    with pytest.raises(RuntimeError):
        mods[names[0]](torch.zeros(1, 256, dtype=torch.float16))


@pytest.mark.gpu
def test_checkpoint_roundtrip_logits_and_greedy_decode(tmp_path):
    from safetensors.torch import save_file

    from autogptq_b200 import QuantLinear, checkpoint

    dev = torch.device("cuda", 0)
    model = _tiny_llama(seed=1)
    packed, deq = _rtn_pack(model)
    names = _quant_names(model)
    # a GPTQ checkpoint as AutoGPTQ writes it: packed buffers under the module names, everything else fp16
    sd = {k: v.half() if v.is_floating_point() else v for k, v in model.state_dict().items()
          if not any(k.startswith(n + ".") for n in names)}
    sd.update({f"{n}.{k}": v.contiguous() for n, q in packed.items() for k, v in q.state_dict().items()})
    path = os.path.join(tmp_path, "model.safetensors")
    save_file(sd, path, metadata={"format": "pt"})
    with open(os.path.join(tmp_path, "quantize_config.json"), "w") as f:
        f.write('{"bits": 4, "group_size": 128, "desc_act": false, "sym": false}')

    # (1) the reference's construction sequence (_utils.py:121-148), written out: positional ctor, .device attribute, .to()
    qmodel = _tiny_llama(seed=2).half()
    for n in names:
        sub = dict(qmodel.named_modules())[n]
        new = QuantLinear(4, 128, sub.in_features, sub.out_features, sub.bias is not None, use_cuda_fp16=True,
                          trainable=False, weight_dtype=sub.weight.dtype)
        new.device = sub.weight.device
        parent = qmodel
        parts = n.split(".")
        for p_ in parts[:-1]:
            parent = getattr(parent, p_)
        setattr(parent, parts[-1], new.to(sub.weight.device))
    from safetensors.torch import load_file

    assert not qmodel.load_state_dict(load_file(path), strict=True).missing_keys
    qmodel = qmodel.to(dev)

    # (2) the reference model: the same checkpoint with the dequantised weights in plain nn.Linear
    ref = _tiny_llama(seed=3).half()
    ref.load_state_dict({k: v for k, v in sd.items() if not any(k.startswith(n + ".") for n in names)}, strict=False)
    for n in names:
        dict(ref.named_modules())[n].weight.data = deq[n].clone()
    ref = ref.to(dev)

    ids = torch.randint(0, 128, (2, 12), device=dev)
    with torch.inference_mode():
        lq = qmodel(ids).logits.float()
        lr = ref(ids).logits.float()
    scale = lr.abs().max().item()
    assert torch.isfinite(lq).all() and (lq - lr).abs().max().item() <= 2e-2 * scale, ((lq - lr).abs().max().item(), scale)

    # greedy decode, token by token (M = batch rows: the decode kernels), as generate(do_sample=False) would
    def greedy(m, start, steps=8):
        seq = start.clone()
        with torch.inference_mode():
            for _ in range(steps):
                seq = torch.cat([seq, m(seq).logits[:, -1].argmax(-1, keepdim=True)], dim=1)
        return seq

    gq, gr = greedy(qmodel, ids[:, :4]), greedy(ref, ids[:, :4])
    # identical unless two logits are closer than the fp16 noise of the two paths
    if not torch.equal(gq, gr):
        with torch.inference_mode():
            top2 = ref(gr[:, :-1]).logits.float().topk(2, -1).values
        assert (top2[..., 0] - top2[..., 1]).min().item() < 2e-2 * scale, "greedy decode diverged with a clear margin"

    # (3) f1: the same checkpoint through autogptq_b200.checkpoint, layer by layer against the module path
    layers = checkpoint.load_quant_linears(str(tmp_path), device=dev)
    assert set(layers) == set(names)
    x = torch.randn(3, 256, dtype=torch.float16, device=dev)
    n0 = names[0]
    assert torch.equal(layers[n0](x), dict(qmodel.named_modules())[n0](x))
