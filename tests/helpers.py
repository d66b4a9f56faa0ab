"""Shared helpers for the tests (fixtures loading, tolerances)."""
import os

import numpy as np
import torch

from oracle import asr_oracle as O

GOLDEN_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
GOLDEN_CASES = ["none_l1", "none_ce", "vgg_l2", "emb_l1"]


def load_golden(name):
    z = np.load(os.path.join(GOLDEN_DIR, name + ".npz"))
    c = z["meta.cfg"]
    cfg = O.OracleConfig(num_layers=int(c[0]), num_heads=int(c[1]), dim_model=int(c[2]), dim_key=int(c[3]),
                         dim_value=int(c[4]), dim_inner=int(c[5]), vocab=int(c[6]), tgt_max_len=int(c[7]),
                         freq=int(c[8]), feat_extractor=str(z["meta.feat"]))
    P = {k[len("param."):]: torch.from_numpy(z[k]) for k in z.files if k.startswith("param.")}
    G = {k[len("grad."):]: torch.from_numpy(z[k]) for k in z.files if k.startswith("grad.")}
    io = {k: torch.from_numpy(np.asarray(z[k])) for k in z.files if k.startswith("in.") or k.startswith("out.")}
    return cfg, P, G, io, float(z["meta.smoothing"])


def rel_err(a: torch.Tensor, b: torch.Tensor) -> float:
    """max|a-b| / max|b| -- the 'relative fp32' measure used for every parity statement."""
    a = a.detach().double().cpu()
    b = b.detach().double().cpu()
    denom = b.abs().max().item()
    if denom == 0.0:
        return (a - b).abs().max().item()
    return (a - b).abs().max().item() / denom


def grads_rel_err(grads: dict, ref: dict) -> dict:
    """Per-tensor max|g-g_ref| / max(max|g_ref|, 1e-3 * largest gradient magnitude in the model).
    The floor keeps mathematically-zero gradients (e.g. key_linear.bias: softmax is shift invariant)
    from turning rounding noise into a relative error of O(1)."""
    gmax = max(float(v.abs().max()) for v in ref.values())
    out = {}
    for k, r in ref.items():
        denom = max(float(r.abs().max()), 1e-3 * gmax)
        out[k] = float((grads[k].detach().double().cpu() - r.double().cpu()).abs().max()) / denom
    return out


def pool_windows_well_separated(h, rel_gap=3e-6):
    """True if no 2x2 max-pool window of h (B,C,F,T) has its two largest entries within rel_gap of each other
    (unless the max is <= 0, where the ReLU mask zeroes the gradient anyway).  Max-pool routing is discontinuous:
    a near-tie lets fp32 rounding noise move the whole gradient to the neighbouring pixel (observed: values
    0.00735714 vs 0.00735718), so parity inputs must avoid them -- the reference has the same sensitivity.
    rel_gap is a few times the fp32 agreement between two correct implementations (~1e-6 of the tensor's scale)."""
    B, C, Fh, Tw = h.shape
    w = h[:, :, :Fh // 2 * 2, :Tw // 2 * 2].reshape(B, C, Fh // 2, 2, Tw // 2, 2).permute(0, 1, 2, 4, 3, 5).reshape(B, C, Fh // 2, Tw // 2, 4)
    top = w.topk(2, dim=-1).values
    live = top[..., 0] > 0
    gap = (top[..., 0] - top[..., 1])[live]
    return bool((gap > rel_gap * h.abs().max()).all())



def vgg_pools_well_separated(P, x, rel_gap=3e-6):
    """Both max-pool inputs of the VGG front end (models/asr/transformer.py:47,52) for input x are free of near-ties."""
    import torch.nn.functional as F
    with torch.no_grad():
        h2 = F.relu(F.conv2d(F.relu(F.conv2d(x, P["conv.0.weight"], P["conv.0.bias"], padding=1)), P["conv.2.weight"], P["conv.2.bias"], padding=1))
        h4 = F.relu(F.conv2d(F.relu(F.conv2d(F.max_pool2d(h2, 2, 2), P["conv.5.weight"], P["conv.5.bias"], padding=1)), P["conv.7.weight"], P["conv.7.bias"], padding=1))
    return pool_windows_well_separated(h2, rel_gap) and pool_windows_well_separated(h4, rel_gap)


def assert_grads_close(grads: dict, ref: dict, tol: float, exact_kernels: bool):
    """Gradient parity criterion.
    exact_kernels=True (fp32 CUDA-core mode): every tensor within `tol` in the max norm (with the floor of grads_rel_err).
    Tensor-core default mode: arithmetic differs from fp32 by ~1e-5, which is enough to flip individual ReLU / max-pool
    decisions that sit within rounding of their threshold (a discontinuity of the MODEL -- the reference on a GPU with TF32
    convolutions shows the same); a flipped unit moves O(1/n_tokens) of a weight-gradient row.  The bound is therefore:
    median tensor error <= tol, and every tensor <= 10*tol in the relative L2 norm."""
    errs = grads_rel_err(grads, ref)
    worst = max(errs, key=errs.get)
    if exact_kernels:
        assert errs[worst] < tol, (worst, errs[worst])
        return
    med = sorted(errs.values())[len(errs) // 2]
    assert med < tol, ("median", med)
    gmax = max(float(v.abs().max()) for v in ref.values())
    for k, r in ref.items():
        g = grads[k].detach().double().cpu()
        denom = max(float(r.double().norm()), 1e-3 * gmax * r.numel() ** 0.5)
        assert float((g - r.double()).norm()) / denom < 10 * tol, k


def sample_index(numel: int, n: int, seed: int) -> np.ndarray:
    """Fixed flat indices of a large tensor that a fixture stores a sample of (numpy's legacy generator: a stable stream)."""
    if numel <= n:
        return np.arange(numel)
    return np.random.RandomState(seed).randint(0, numel, n)


def reference_batch(B, freq, T, vocab, Lt, seed=0):
    """Ragged, length-sorted synthetic batch (src [B,1,freq,T] zero past each length, int32 lengths, PAD-padded targets
    and their int32 lengths), in the shape utils/data_loader.py's _collate_fn hands it over."""
    g = torch.Generator().manual_seed(seed)
    src = torch.randn(B, 1, freq, T, generator=g)
    lens = (T * (0.5 + 0.5 * torch.rand(B, generator=g))).long().clamp(1, T)
    lens[0] = T
    lens = torch.sort(lens, descending=True).values
    for i in range(B):
        src[i, :, :, int(lens[i]):] = 0
    tgt = torch.randint(3, vocab, (B, Lt), generator=g)
    tl = (Lt * (0.4 + 0.6 * torch.rand(B, generator=g))).long().clamp(1, Lt)
    tl[0] = Lt
    for i in range(B):
        tgt[i, int(tl[i]):] = 0
    return src, lens.to(torch.int32), tgt, tl.to(torch.int32)


def batch_checksum(src, lens, tgt) -> np.ndarray:
    """Stored next to a regenerated batch so that a change of torch's random stream shows up as such."""
    return np.array([float(src.double().sum()), float(src.double().abs().sum()), float(lens.sum()), float(tgt.sum())])


def seeded_state(shapes: dict, seed: int) -> dict:
    """Parameters regenerated from a seed instead of stored in a fixture: N(0, 1/fan_in) for matrices and convolution
    kernels, 1 + N(0, 0.01) for 1-d weights (LayerNorm / BatchNorm scales), N(0, 0.01) for biases."""
    out = {}
    for i, (name, shape) in enumerate(sorted(shapes.items())):
        r = np.random.RandomState(seed + i)
        shape = tuple(shape)
        if len(shape) >= 2:
            v = r.standard_normal(shape) / np.sqrt(float(np.prod(shape[1:])))
        elif name.endswith("weight"):
            v = 1.0 + 0.1 * r.standard_normal(shape)
        else:
            v = 0.1 * r.standard_normal(shape)
        out[name] = torch.from_numpy(v.astype(np.float32))
    return out


def load_greedy_golden():
    """tests/golden/greedy.npz: token ids of the reference's Decoder.greedy_search (cut at EOS), the encoder output fed to it
    and the decoder parameters (generated by tests/golden/make_golden.py::run_greedy from the live reference)."""
    z = np.load(os.path.join(GOLDEN_DIR, "greedy.npz"))
    c = z["meta.cfg"]
    cfg = O.OracleConfig(num_layers=int(c[0]), num_heads=int(c[1]), dim_model=int(c[2]), dim_key=int(c[3]),
                         dim_value=int(c[4]), dim_inner=int(c[5]), vocab=int(c[6]), tgt_max_len=int(c[7]),
                         freq=int(c[8]), feat_extractor="")
    P = {k[len("param."):]: torch.from_numpy(z[k]) for k in z.files if k.startswith("param.")}
    return cfg, P, torch.from_numpy(z["in.enc"]), torch.from_numpy(z["out.ids"]), torch.from_numpy(z["out.lengths"])


def cut_at_eos(ids_row, eos=2):
    """Tokens before the first EOS (the reference's string building, models/asr/transformer.py:385-393)."""
    out = []
    for t in ids_row.tolist():
        if t == eos:
            break
        out.append(t)
    return out
