"""CPU tests of the host-side mirror: configuration arithmetic, state_dict compatibility with the reference, schedules,
sharding, flat buffers, the install() patcher and the "CUDA only" contract."""
import importlib
import os
import sys
import types

import pytest
import torch

import b200asr
from oracle import asr_oracle as O
from oracle import ref_shim
from tests.helpers import GOLDEN_CASES, load_golden


def test_config_dims_follow_reference_formulae():
    assert b200asr.ASRConfig(feat_extractor="vgg_cnn").dim_input == 5120          # utils/functions.py:128-130
    assert b200asr.ASRConfig(feat_extractor="emb_cnn").dim_input == 672           # utils/functions.py:121-126
    assert b200asr.ASRConfig(feat_extractor="").dim_input == 161
    assert b200asr.ASRConfig().t_enc(800) == 200 and b200asr.ASRConfig(feat_extractor="emb_cnn").t_enc(400) == 195
    c2 = b200asr.BASELINE_CONFIGS["cfg2"]
    assert (c2["batch"], c2["t_src"], c2["cfg"].tgt_max_len, c2["cfg"].vocab) == (32, 800, 100, 4364)


@pytest.mark.parametrize("case", GOLDEN_CASES)
def test_mirror_state_dict_is_reference_compatible(case):
    """Parameter names/shapes equal the reference's (fixtures hold its state_dict), so checkpoints round-trip."""
    from tests.gpu_util import asr_cfg
    cfg, P, _, _, _ = load_golden(case)
    m = b200asr.build_model(asr_cfg(cfg))
    sd = {k: v for k, v in m.state_dict().items() if not (k.endswith("positional_encoding.pe") or "running_" in k or "num_batches" in k)}
    assert set(sd) == set(P)
    for k in P:
        assert tuple(sd[k].shape) == tuple(P[k].shape), k
    assert sum(p.numel() for p in b200asr.build_model(b200asr.ASRConfig()).parameters()) == 36776384   # SURVEY.md §8d


def test_noam_schedule_and_shard_batch():
    opt = b200asr.NoamOpt(5120, 1.0, 4000, types.SimpleNamespace(param_groups=[{"lr": 0}], step=lambda **kw: None, zero_grad=lambda: None), min_lr=1e-6)
    for s in range(1, 6):
        opt.step()
        assert opt._rate == pytest.approx(O.noam_rate(s, 5120, 1.0, 4000, 1e-6))
    src, lens, tgt = torch.arange(8).view(8, 1), torch.arange(8), torch.arange(8)
    a = b200asr.shard_batch(src, lens, tgt, 1, 4)
    assert a[0].view(-1).tolist() == [2, 3] and a[1].tolist() == [2, 3]
    with pytest.raises(ValueError):
        b200asr.shard_batch(src, lens, tgt, 0, 3)


def test_flat_params_views_alias_one_buffer():
    lin = torch.nn.Sequential(torch.nn.Linear(5, 3), torch.nn.Linear(3, 2))
    before = [p.detach().clone() for p in lin.parameters()]
    flat = b200asr.FlatParams(lin, extra=2)
    assert flat.flat_grad.numel() == flat.numel + 2 and all(o % 4 == 0 for o in flat.offsets)
    for p, b in zip(lin.parameters(), before):
        assert torch.equal(p.detach(), b)
        assert p.data_ptr() >= flat.flat.data_ptr() and p.grad.data_ptr() >= flat.flat_grad.data_ptr()
    lin(torch.randn(4, 5)).sum().backward()
    assert flat.flat_grad[:flat.numel].abs().sum() > 0            # autograd accumulated straight into the flat buffer
    lin.zero_grad(set_to_none=True)
    lin(torch.randn(4, 5)).sum().backward()
    flat.ensure_grad_views()
    assert all(p.grad.data_ptr() >= flat.flat_grad.data_ptr() for p in lin.parameters())


def test_flat_params_lay_qkv_projections_back_to_back():
    """The layout ops.AttnProjFn keys on: W_q|W_k|W_v, their biases and all their gradients adjacent in ONE storage, while
    names / shapes / values (state_dict) are untouched."""
    import importlib
    ops = importlib.import_module(b200asr.__name__ + ".ops")
    m = b200asr.build_model(b200asr.ASRConfig(num_layers=2, num_heads=2, dim_model=32, dim_key=16, dim_value=8, dim_inner=64,
                                              vocab=40, feat_extractor="", tgt_max_len=6))
    before = {k: v.clone() for k, v in m.state_dict().items()}
    flat = b200asr.FlatParams(m)
    blocks = [l.self_attn for l in m.encoder.layers] + [a for l in m.decoder.layers for a in (l.self_attn, l.encoder_attn)]
    for att in blocks:
        ws = [att.query_linear.weight, att.key_linear.weight, att.value_linear.weight]
        bs = [att.query_linear.bias, att.key_linear.bias, att.value_linear.bias]
        assert ops._adjacent(*ws) and ops._adjacent(*bs)                       # dk != dv: rows differ, widths equal
        assert ops._adjacent(*[w.grad for w in ws]) and ops._adjacent(*[b.grad for b in bs])
        stacked = ops._stacked(*ws)
        assert stacked.shape == (2 * 16 + 2 * 16 + 2 * 8, 32) and torch.equal(stacked[:32], ws[0]) and torch.equal(stacked[64:], ws[2])
    after = m.state_dict()
    assert list(after) == list(before) and all(torch.equal(after[k], before[k]) for k in before)
    assert len({id(p) for p in flat.params}) == len(list(m.parameters()))      # every parameter exactly once
    # separately allocated neighbours must not be stacked (a view cannot span two storages)
    a, b = torch.zeros(4, 8), torch.zeros(4, 8)
    assert not ops._adjacent(a, b)


def test_cpu_tensors_are_rejected_not_computed():
    m = b200asr.build_model(b200asr.ASRConfig(num_layers=1, vocab=40, feat_extractor="", tgt_max_len=6))
    with pytest.raises(RuntimeError, match="CUDA"):
        m(torch.randn(2, 1, 161, 16), torch.tensor([16, 12]), torch.randint(3, 40, (2, 5)))
    with pytest.raises(RuntimeError, match="CUDA"):
        b200asr.calculate_metrics(torch.randn(2, 3, 8), torch.ones(2, 3, dtype=torch.long))


REF = ref_shim.reference_root()


@pytest.mark.skipif(REF is None, reason="no reference checkout: neither $B200ASR_REFERENCE nor oracle/_ref (staged by build())")
def test_install_rebinds_reference_classes_and_keeps_module_tree():
    """Runs in a subprocess because the reference parses flags at import (utils/constant.py:99)."""
    import subprocess
    code = r'''
import sys, types
sys.path.insert(0, %r); sys.path.insert(0, %r)
sys.modules["Levenshtein"] = types.ModuleType("Levenshtein")
sys.argv = ["x", "--num-layers", "1", "--num-heads", "2", "--dim-model", "64", "--dim-emb", "64", "--dim-key", "32", "--dim-value", "32",
            "--dim-inner", "64", "--feat_extractor", "vgg_cnn", "--tgt-max-len", "8", "--sample-rate", "4000"]
import torch
from utils import constant
from utils.functions import init_transformer_model
import models.common_layers as cl, models.asr.transformer as tr, utils.metrics as um
import b200asr
orig = tr.Transformer.forward
labels = {i: str(i) for i in range(20)}
model = init_transformer_model(constant.args, {v: k for k, v in labels.items()}, labels)
keys = list(model.state_dict().keys())
b200asr.install()
assert tr.Transformer.forward is not orig and cl.MultiHeadAttention.forward.__module__.endswith("modules")
assert um.calculate_metrics.__module__.endswith("metrics")
assert list(model.state_dict().keys()) == keys                      # module tree / names untouched
try:
    model(torch.randn(2, 1, 41, 16), torch.tensor([16, 12], dtype=torch.int32), torch.randint(3, 20, (2, 5)))
    raise SystemExit("expected the CUDA-only error")
except RuntimeError as e:
    assert "CUDA" in str(e)
b200asr.uninstall()
assert tr.Transformer.forward is orig
pred, gold, hyp, _ = model(torch.randn(2, 1, 41, 16), torch.tensor([16, 12], dtype=torch.int32), torch.randint(3, 20, (2, 5)))
assert pred.shape == (2, 8, 20)
print("OK")
''' % (REF, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    out = subprocess.run([sys.executable, "-W", "ignore", "-c", code], capture_output=True, text=True, timeout=300)
    assert out.returncode == 0 and "OK" in out.stdout, out.stderr[-2000:]


def test_bench_flop_accounting_reads_integer_dimensions_of_the_abi():
    """bench.algorithmic_flops picks problem sizes out of the raw C-ABI argument tuples by position: every position it reads
    must be a C int of that entry point's prototype (guards the indices against ABI edits)."""
    import ctypes
    import importlib
    import bench
    L = importlib.import_module(b200asr.__name__ + "._lib")
    for name in ("linear_fwd", "linear_bwd_data", "linear_bwd_weight", "conv3x3_fwd", "conv3x3_fwd_pool", "conv3x3_bwd_data", "conv3x3_bwd_weight",
                 "conv3x3_c1_fwd", "conv3x3_c1_bwd_weight", "sdpa_fwd", "sdpa_bwd", "sdpa_mat_fwd", "sdpa_mat_bwd", "sdpa_fused_fwd",
                 "sdpa_fused_bwd"):
        argtypes = L.SIGNATURES["b200asr_" + name][1]

        class Probe(tuple):
            def __getitem__(self, i):
                idx = range(len(self))[i] if isinstance(i, slice) else [i]
                for j in idx:
                    assert argtypes[j] is ctypes.c_int, (name, j, argtypes[j])
                return [3] * len(idx) if isinstance(i, slice) else 3

        assert bench.algorithmic_flops(name, Probe(range(len(argtypes)))) > 0


def test_weight_operand_cache_converts_once_per_change(monkeypatch):
    """ops.WeightOperandCache bookkeeping with the conversion kernel stubbed out (no GPU): a weight is registered on first use,
    converted by the refresh of the optimizer step, NOT converted again by the first get() after that (the regression: every
    weight's first get() re-converted all of them -- 46 launches in the step after registration), and converted again when
    the tensor changes in place behind the optimizer's back."""
    ops = importlib.import_module(b200asr.__name__ + ".ops")
    L = importlib.import_module(b200asr.__name__ + "._lib")
    calls = []

    class FakeLib:
        def b200asr_split_bf16_batched(self, *a):
            calls.append(a[4])          # number of matrices in the batch
            return 0

    monkeypatch.setattr(ops, "_lib", lambda: FakeLib())
    monkeypatch.setattr(ops, "_stream", lambda: 0)

    class Flat:
        flat = torch.zeros(4096)
    cache = ops.WeightOperandCache(Flat())
    w1, w2 = Flat.flat[:512].view(16, 32), Flat.flat[1024:2048].view(32, 32)
    assert cache.owns(w1) and not cache.owns(torch.zeros(16, 32))
    assert cache.get(w1, L.PREC_BF16X3) is None and cache.get(w2, L.PREC_BF16X3) is None      # registered, not converted yet
    assert calls == []
    cache.after_optimizer_step()
    assert calls == [2]                                                                      # one launch for both
    s1 = cache.get(w1, L.PREC_BF16X3)
    s2 = cache.get(w2, L.PREC_BF16X3)
    assert s1 is not None and s2 is not None and calls == [2]                                # fresh: no second conversion
    assert tuple(s1.fwd.shape) == (2, 16, 32) and tuple(s2.bwd.shape) == (2, 32, 32)
    cache.after_optimizer_step()
    cache.get(w1, L.PREC_BF16X3)
    assert calls == [2, 2]                                                                   # the optimizer's refresh only
    w1.add_(1.0)                                                                             # in-place edit: version counter moves
    cache.get(w1, L.PREC_BF16X3)
    assert calls == [2, 2, 2]
    cache.get(w1, L.PREC_BF16X3)
    cache.get(w2, L.PREC_BF16X3)                 # w2 shares the buffer's version counter: its view changed version too, but
    assert calls == [2, 2, 2]                    # the refresh that followed the edit already covers it
