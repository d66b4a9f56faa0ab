#!/usr/bin/env python
"""Generate golden fixtures by importing the UNMODIFIED reference from /root/reference.

Run in the build container only (the GPU box has no reference checkout):

    python tests/golden/make_golden.py            # regenerates every case

Each case runs in its own interpreter because the reference parses its flags at
import time (utils/constant.py:99).  Shims (none edit the reference):
  * sys.modules['Levenshtein'] stub -- python-Levenshtein is not installed and is only
    called by calculate_cer/wer, which are off the hot path (utils/metrics.py:3,56,76);
  * sys.argv set before the first `import utils.constant`.
A fixture holds: the inputs, the full state_dict (reference names), pred / gold /
hyp_seq of Transformer.forward (models/asr/transformer.py:59-85), the loss and
num_correct of calculate_metrics (utils/metrics.py:78-95) and every parameter gradient
after loss.backward() -- all fp32 from torch CPU kernels.
"""
import os
import subprocess
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
REF = "/root/reference"

CASES = {
    # name: (flags, B, T_src, freq, V, smoothing, ragged)
    "none_l1": (["--num-layers", "1", "--num-heads", "2", "--dim-model", "128", "--dim-emb", "128",
                 "--dim-key", "64", "--dim-value", "64", "--dim-inner", "256", "--feat_extractor", "",
                 "--tgt-max-len", "10"], 2, 50, 161, 32, 0.1, True),
    "none_ce": (["--num-layers", "2", "--num-heads", "4", "--dim-model", "64", "--dim-emb", "64",
                 "--dim-key", "16", "--dim-value", "32", "--dim-inner", "96", "--feat_extractor", "",
                 "--tgt-max-len", "12"], 3, 37, 161, 50, 0.0, True),
    "vgg_l2": (["--num-layers", "2", "--num-heads", "2", "--dim-model", "64", "--dim-emb", "64",
                "--dim-key", "32", "--dim-value", "32", "--dim-inner", "128", "--feat_extractor", "vgg_cnn",
                "--sample-rate", "4000", "--tgt-max-len", "8"], 2, 24, 41, 40, 0.1, True),
    "emb_l1": (["--num-layers", "1", "--num-heads", "2", "--dim-model", "64", "--dim-emb", "64",
                "--dim-key", "32", "--dim-value", "32", "--dim-inner", "128", "--feat_extractor", "emb_cnn",
                "--tgt-max-len", "8"], 3, 40, 161, 40, 0.1, False),
}


def run_case(name):
    import types
    flags, B, T, freq, V, smoothing, ragged = CASES[name]
    sys.path.insert(0, REF)
    sys.modules["Levenshtein"] = types.ModuleType("Levenshtein")
    sys.argv = ["make_golden"] + flags + ["--label-smoothing", str(smoothing), "--dropout", "0.0"]
    import torch
    from utils import constant
    from utils.functions import init_transformer_model
    from utils.metrics import calculate_metrics

    labels = ["_", "<s>", "</s>"] + ["t%d" % i for i in range(V - 3)]
    label2id = {l: i for i, l in enumerate(labels)}
    id2label = {i: l for i, l in enumerate(labels)}
    torch.manual_seed(123456)
    model = init_transformer_model(constant.args, label2id, id2label)
    model.train()
    # nudge norm/bias parameters away from (1, 0) so their gradients and use are exercised
    g = torch.Generator().manual_seed(7)
    with torch.no_grad():
        for n, p in model.named_parameters():
            if p.dim() == 1:
                p.add_(0.1 * torch.randn(p.shape, generator=g))

    g = torch.Generator().manual_seed(0)
    src = torch.randn(B, 1, freq, T, generator=g)
    if ragged:
        lens = (T * (0.5 + 0.5 * torch.rand(B, generator=g))).long().clamp(1, T)
        lens[0] = T
        lens, _ = torch.sort(lens, descending=True)
    else:
        lens = torch.full((B,), T, dtype=torch.long)
    for i in range(B):
        src[i, :, :, int(lens[i]):] = 0
    L = constant.args.tgt_max_len - 1
    tgt = torch.randint(3, V, (B, L), generator=g)
    tl = (L * (0.4 + 0.6 * torch.rand(B, generator=g))).long().clamp(1, L)
    tl[0] = L
    for i in range(B):
        tgt[i, int(tl[i]):] = 0
    lens32 = lens.to(torch.int32)

    pred, gold, hyp, _ = model(src, lens32, tgt, verbose=False)
    loss, ncorrect = calculate_metrics(pred, gold, smoothing=smoothing, loss_type="ce")
    loss.backward()

    out = {"in.src": src.numpy(), "in.lengths": lens32.numpy(), "in.tgt": tgt.numpy(),
           "out.pred": pred.detach().numpy(), "out.gold": gold.numpy(), "out.hyp": hyp.numpy(),
           "out.loss": np.float32(loss.item()), "out.num_correct": np.int64(ncorrect),
           "meta.smoothing": np.float32(smoothing)}
    for n, p in model.state_dict().items():
        if n.endswith("positional_encoding.pe") or "num_batches_tracked" in n or "running_" in n:
            continue
        out["param." + n] = p.detach().numpy()
    for n, p in model.named_parameters():
        out["grad." + n] = p.grad.numpy() if p.grad is not None else np.zeros(p.shape, np.float32)
    a = constant.args
    out["meta.cfg"] = np.array([a.num_layers, a.num_heads, a.dim_model, a.dim_key, a.dim_value, a.dim_inner,
                                V, a.tgt_max_len, freq], dtype=np.int64)
    out["meta.feat"] = np.array(a.feat_extractor)
    path = os.path.join(HERE, name + ".npz")
    np.savez_compressed(path, **out)
    print(name, "pred", tuple(pred.shape), "loss %.6f" % loss.item(), "->", path,
          "%.1f KB" % (os.path.getsize(path) / 1024))


def run_greedy():
    """Fixture `greedy`: token ids of the reference's Decoder.greedy_search (models/asr/transformer.py:316-394) -- 300 fixed
    steps of full-prefix re-decode, strings cut at the first EOS (:385-393).  Shims (SURVEY.md 8c, Q12; none edit the
    reference): get_subsequent_mask(...).bool() (the uint8 mask no longer adds to a bool one on torch >= 1.2) and
    --tgt-max-len 301 (the positional table must cover 300 positions).  Every id >= 3 maps to its own character, so
    the returned strings map back to ids.  The EOS row of output_linear is scaled so that utterances end at different,
    non-trivial steps (a random-init model would otherwise hardly ever emit EOS)."""
    sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
    from oracle import ref_shim
    V, B, Te = 40, 4, 23
    ns = ref_shim.load(["--num-layers", "2", "--num-heads", "2", "--dim-model", "64", "--dim-emb", "64", "--dim-key", "32",
                        "--dim-value", "32", "--dim-inner", "128", "--feat_extractor", "", "--tgt-max-len", "301",
                        "--dropout", "0.0"], q12_shim=True)
    import torch
    l2i, i2l = ref_shim.labels(V)
    torch.manual_seed(123456)
    model = ns.functions.init_transformer_model(ns.constant.args, l2i, i2l)
    model.eval()
    g = torch.Generator().manual_seed(11)
    with torch.no_grad():
        for n, p in model.named_parameters():
            if p.dim() == 1:
                p.add_(0.1 * torch.randn(p.shape, generator=g))
        model.decoder.output_linear.weight.mul_(4.0)            # spread the logits (fewer near-ties)
        model.decoder.output_linear.weight[2].mul_(2.2)         # EOS wins now and then
    enc = torch.randn(B, Te, 64, generator=g)
    with torch.no_grad():
        strs = model.decoder.greedy_search(enc)
    ids = np.full((B, 300), -1, dtype=np.int64)                 # -1 = not produced (after the EOS cut)
    for b, s in enumerate(strs):
        ids[b, :len(s)] = [l2i[c] for c in s]
    out = {"in.enc": enc.numpy(), "out.ids": ids, "out.lengths": np.array([len(s) for s in strs], dtype=np.int64)}
    for n, p in model.state_dict().items():
        if n.startswith("decoder.") and not n.endswith("positional_encoding.pe"):
            out["param." + n] = p.detach().numpy()
    out["meta.cfg"] = np.array([2, 2, 64, 32, 32, 128, V, 301, 161], dtype=np.int64)
    path = os.path.join(HERE, "greedy.npz")
    np.savez_compressed(path, **out)
    print("greedy: utterance lengths (cut at EOS)", [len(s) for s in strs], "->", path, "%.1f KB" % (os.path.getsize(path) / 1024))


SMALL_VGG = ["--num-layers", "2", "--num-heads", "2", "--dim-model", "64", "--dim-emb", "64", "--dim-key", "32", "--dim-value", "32",
             "--dim-inner", "128", "--feat_extractor", "vgg_cnn", "--sample-rate", "4000", "--tgt-max-len", "12"]
SMALL_EMB = ["--num-layers", "1", "--num-heads", "2", "--dim-model", "64", "--dim-emb", "64", "--dim-key", "32", "--dim-value", "32",
             "--dim-inner", "128", "--feat_extractor", "emb_cnn", "--tgt-max-len", "10"]
CFG2_ARCH = ["--num-layers", "4", "--num-heads", "8", "--dim-model", "512", "--dim-emb", "512", "--dim-key", "64", "--dim-value", "64",
             "--dim-inner", "2048", "--feat_extractor", "vgg_cnn", "--tgt-max-len", "40"]
# name: (flags, V, freq, B, T_src)
REFERENCE_CASES = {"small_vgg": (SMALL_VGG, 40, 41, 3, 32), "small_emb": (SMALL_EMB, 40, 161, 3, 48),
                   "cfg2_arch": (CFG2_ARCH, 4364, 161, 2, 200)}
TRAINER_CASES = {"small_vgg": (SMALL_VGG, 40, 41, 4, 32), "small_emb": (SMALL_EMB, 40, 161, 4, 48)}
SEEDED_STATE = 2024
# arrays up to `limit` elements are stored whole, larger ones as a fixed sample of n elements: (limit, n).  Inputs and
# parameters are regenerated from their seeds; the five fixtures stay under 300 KB together.
STORE = {"pred": (4096, 4096), "grad": (512, 128), "dec": (8192, 8192)}
STORE_CFG2 = dict(STORE, grad=(64, 64))             # ~190 gradient tensors


def _ref_model(flags, vocab):
    """The reference's own Transformer (utils/functions.py:116-152) with helpers.seeded_state parameters (regenerated by the
    tests instead of being stored)."""
    import torch
    sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
    from oracle import ref_shim
    from tests.helpers import seeded_state
    ns = ref_shim.load(list(flags) + ["--dropout", "0.0", "--label-smoothing", "0.1"])
    l2i, i2l = ref_shim.labels(vocab)
    model = ns.functions.init_transformer_model(ns.constant.args, l2i, i2l)
    state = seeded_state({n: p.shape for n, p in model.named_parameters()}, SEEDED_STATE)
    with torch.no_grad():
        for n, p in model.named_parameters():
            p.copy_(state[n])
    return ns, model, l2i, i2l


def _pack(out, group, items, seed0, limit, n):
    """Arrays (name, a) of one group in three entries: `<group>.names`, `<group>.values` (each array whole, or -- more than
    `limit` elements -- its values at helpers.sample_index(a.size, n, seed), concatenated) and `<group>.info`, one row per
    array: [seed (-1: whole), max |a|, L2 norm of a, offset, count, ndim, shape padded to 4 dims]."""
    from tests.helpers import sample_index
    names, values, info, off = [], [], [], 0
    for i, (name, a) in enumerate(items):
        a = np.asarray(a)
        whole = a.size <= limit
        v = a.reshape(-1) if whole else a.reshape(-1)[sample_index(a.size, n, seed0 + i)]
        info.append([-1 if whole else seed0 + i, np.abs(a).max(), np.linalg.norm(a.astype(np.float64)), off, v.size, a.ndim]
                    + list(a.shape) + [1] * (4 - a.ndim))
        names.append(name)
        values.append(v)
        off += v.size
    out[group + ".names"], out[group + ".values"] = np.array(names, dtype=str), np.concatenate(values)
    out[group + ".info"] = np.array(info, dtype=np.float64)


def run_reference_case(name):
    """Fixture `ref_<name>`: the reference's own CPU forward / calculate_metrics / backward, with the branch every ReLU /
    Hardtanh unit took (forward hooks on nn.ReLU / nn.Hardtanh and on the FFN's conv_1 output, in execution order)."""
    import torch
    flags, V, freq, B, T = REFERENCE_CASES[name]
    ns, model, _, _ = _ref_model(flags, V)
    from tests.helpers import batch_checksum, reference_batch
    src, lens, tgt, _ = reference_batch(B, freq, T, V, ns.constant.args.tgt_max_len - 1, seed=0)
    dec, handles = [], []

    def hook(kind, transpose=False):
        def f(_m, _i, o):
            o = o.detach().transpose(1, 2) if transpose else o.detach()
            dec.append((o > 0).to(torch.int8) + ((o >= 20).to(torch.int8) if kind == "hardtanh" else 0))
        return f
    for m in model.modules():
        if isinstance(m, torch.nn.Hardtanh):
            handles.append(m.register_forward_hook(hook("hardtanh")))
        elif isinstance(m, torch.nn.ReLU):
            handles.append(m.register_forward_hook(hook("relu")))
        elif type(m).__name__ == "PositionwiseFeedForwardWithConv":      # F.relu of conv_1's [B, d_inner, T] output
            handles.append(m.conv_1.register_forward_hook(hook("relu", transpose=True)))
    model.train()
    pred, gold, hyp, _ = model(src, lens, tgt, verbose=False)
    for h in handles:
        h.remove()
    loss, ncorrect = ns.metrics.calculate_metrics(pred, gold, smoothing=0.1, loss_type="ce")
    loss.backward()
    a = ns.constant.args
    out = {"in.shape": np.array([B, T]), "in.seed": np.int64(0), "in.checksum": batch_checksum(src, lens, tgt), "out.gold": gold.numpy(),
           "out.hyp": hyp.numpy(), "out.loss": np.float32(loss.item()), "out.num_correct": np.int64(ncorrect),
           "meta.cfg": np.array([a.num_layers, a.num_heads, a.dim_model, a.dim_key, a.dim_value, a.dim_inner, V,
                                 a.tgt_max_len, freq], dtype=np.int64),
           "meta.feat": np.array(a.feat_extractor), 
           "meta.seeded_state": np.int64(SEEDED_STATE)}
    store = STORE_CFG2 if name == "cfg2_arch" else STORE
    _pack(out, "pred", [("pred", pred.detach().numpy())], 1, *store["pred"])
    _pack(out, "grad", [(n, p.grad.numpy()) for n, p in sorted(model.named_parameters())], 100, *store["grad"])
    _pack(out, "dec", [(str(i), d.numpy()) for i, d in enumerate(dec)], 10000, *store["dec"])
    path = os.path.join(HERE, "ref_%s.npz" % name)
    np.savez_compressed(path, **out)
    print("ref_%s: loss %.6f, %d decision tensors -> %s %.1f KB" % (name, loss.item(), len(dec), path, os.path.getsize(path) / 1024))


def run_trainer_case(name):
    """Fixture `trainer_<name>`: one epoch of the reference's own Trainer.train (trainer/asr/trainer.py:20-211) on the CPU --
    3 training iterations (NoamOpt + torch Adam, gradient clipping) and one eval-mode validation batch -- on synthetic
    _collate_fn-shaped batches: the loss of every calculate_metrics call, the learning rate of every step, and the state
    before and after."""
    import copy
    import tempfile
    import torch
    flags, V, freq, B, T = TRAINER_CASES[name]
    ns, model, l2i, i2l = _ref_model(flags + ["--warmup", "4", "--k-lr", "0.02", "--min-lr", "1e-6", "--clip", "--max-norm", "400"], V)
    frozen = []
    if name == "small_emb":
        # a conv bias in front of BatchNorm is a gauge freedom: its true gradient is zero, Adam turns the rounding noise into
        # +-lr steps, and running_mean absorbs the resulting random walk.  Frozen so that the buffers are comparable.
        frozen = ["conv.0.bias", "conv.3.bias"]
        model.conv[0].bias.requires_grad_(False)
        model.conv[3].bias.requires_grad_(False)
    init = {k: v.detach().clone() for k, v in model.state_dict().items()}
    Lt = ns.constant.args.tgt_max_len - 1

    from tests.helpers import batch_checksum, reference_batch

    def batch(seed):
        src, lens, tgt, tl = reference_batch(B, freq, T, V, Lt, seed=seed)
        return (src, tgt, lens.float() / float(T), lens, tl)            # _collate_fn order, utils/data_loader.py:213
    train, valid = [batch(s) for s in range(3)], [batch(100)]          # seeds stored below
    opt = ns.functions.init_optimizer(ns.constant.args, model, "noam")
    losses, rates = [], []
    cur, opt_step = ns.trainer.calculate_metrics, opt.step

    def recording(*a, **k):
        r = cur(*a, **k)
        losses.append(float(r[0].item()))
        return r

    def step():
        opt_step()
        rates.append(opt._rate)
    ns.trainer.calculate_metrics, opt.step = recording, step
    with tempfile.TemporaryDirectory() as tmp:
        ns.constant.args.save_folder, ns.constant.args.name = tmp, "golden"
        ns.trainer.Trainer().train(model, copy.deepcopy(train), None, [copy.deepcopy(valid)], opt, "ce", 0, 1, l2i, i2l)
    ns.trainer.calculate_metrics = cur
    a = ns.constant.args
    out = {"out.losses": np.array(losses, dtype=np.float64), "out.rates": np.array(rates, dtype=np.float64),
           "meta.cfg": np.array([a.num_layers, a.num_heads, a.dim_model, a.dim_key, a.dim_value, a.dim_inner, V,
                                 a.tgt_max_len, freq], dtype=np.int64),
           "meta.feat": np.array(a.feat_extractor), "meta.frozen": np.array(frozen, dtype=str),
           "meta.max_norm": np.float32(a.max_norm), "meta.seeded_state": np.int64(SEEDED_STATE)}
    deltas = []
    for k, v in sorted(model.state_dict().items()):
        if k.endswith("positional_encoding.pe"):
            continue
        if "running_" in k or "num_batches_tracked" in k:
            out["final." + k] = v.numpy()
        else:                                   # parameters: the change made by the three optimizer steps
            deltas.append((k, (v - init[k]).numpy()))
    _pack(out, "delta", deltas, 200, *STORE["grad"])
    out["in.shape"], out["in.train.seeds"], out["in.valid.seed"] = np.array([B, T]), np.arange(3), np.int64(100)
    out["in.checksum"] = np.stack([batch_checksum(src, lens, tgt) for src, tgt, _, lens, _ in train + valid])
    path = os.path.join(HERE, "trainer_%s.npz" % name)
    np.savez_compressed(path, **out)
    print("trainer_%s: losses %s -> %s %.1f KB" % (name, losses, path, os.path.getsize(path) / 1024))


if __name__ == "__main__":
    if len(sys.argv) == 3 and sys.argv[1] == "--case":
        c = sys.argv[2]
        if c == "greedy":
            run_greedy()
        elif c.startswith("ref_"):
            run_reference_case(c[len("ref_"):])
        elif c.startswith("trainer_"):
            run_trainer_case(c[len("trainer_"):])
        else:
            run_case(c)
    else:
        for c in list(CASES) + ["greedy"] + ["ref_" + n for n in REFERENCE_CASES] + ["trainer_" + n for n in TRAINER_CASES]:
            subprocess.check_call([sys.executable, "-W", "ignore", os.path.abspath(__file__), "--case", c])
