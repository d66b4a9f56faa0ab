"""The oracle (oracle/asr_oracle.py) replayed against fixtures produced by the live reference
(tests/golden/make_golden.py).  This is what pins the oracle; CPU only."""
import pytest
import torch

from oracle import asr_oracle as O
from tests.helpers import GOLDEN_CASES, load_golden, rel_err, grads_rel_err


@pytest.mark.parametrize("case", GOLDEN_CASES)
def test_forward_loss_and_grads_match_reference(case):
    cfg, P, G, io, smoothing = load_golden(case)
    pred, gold, hyp, loss, n_word, grads = O.forward_backward(P, cfg, io["in.src"], io["in.lengths"],
                                                              io["in.tgt"], smoothing)
    assert torch.equal(gold, io["out.gold"])
    assert rel_err(pred, io["out.pred"]) < 2e-5
    # bit-exact argmax ids on every real decoder position.  Padded positions (seq_in == EOS) have an
    # exactly-zero logit row (x *= non_pad_mask, bias-free output_linear), so the reference's topk there
    # is an arbitrary tie-break (SURVEY.md §8 A12); they are PAD in `gold` and ignored by loss/metrics.
    real = gold.ne(O.PAD)
    assert torch.equal(hyp[real], io["out.hyp"][real])
    assert float(io["out.pred"][~real].abs().max()) == 0.0 if (~real).any() else True
    assert abs(loss.item() - io["out.loss"].item()) < 2e-5 * abs(io["out.loss"].item())
    assert O.num_correct(pred, gold) == int(io["out.num_correct"])
    assert set(G) == set(grads)
    # a convolution bias followed by training-mode BatchNorm (emb_cnn: conv.0 -> BN conv.1, conv.3 -> BN conv.4) cancels in
    # the batch mean: its gradient is exactly zero, and both the fixture's and the oracle's values are rounding noise whose
    # pattern depends on the CPU's thread count.  Those tensors must be zero to rounding; every other one must match.
    gmax = max(float(v.abs().max()) for v in G.values())
    gauge = [k for k in ("conv.0.bias", "conv.3.bias") if cfg.feat_extractor == "emb_cnn"]
    for k in gauge:
        assert float(G[k].abs().max()) < 1e-5 * gmax and float(grads[k].abs().max()) < 1e-5 * gmax, k
    errs = {k: v for k, v in grads_rel_err(grads, G).items() if k not in gauge}
    worst = max(errs, key=errs.get)
    assert errs[worst] < 5e-4, (worst, errs[worst])


def test_preprocess_matches_reference_semantics():
    tgt = torch.tensor([[5, 6, 7, 0, 0], [9, 0, 0, 0, 0]])
    s_in, s_out = O.preprocess_targets(tgt, 6)
    assert s_in.tolist() == [[1, 5, 6, 7, 2, 2], [1, 9, 2, 2, 2, 2]]
    assert s_out.tolist() == [[5, 6, 7, 2, 0, 0], [9, 2, 0, 0, 0, 0]]


def test_init_params_names_match_reference_state_dict():
    for case in GOLDEN_CASES:
        cfg, P, _, _, _ = load_golden(case)
        mine = O.init_params(cfg)
        assert set(mine) == set(P), case
        for k in P:
            assert tuple(mine[k].shape) == tuple(P[k].shape), k


def test_noam_and_adam_reference():
    assert O.noam_rate(1, 5120, 1.0, 4000, 1e-6) == 1e-6            # floored at min_lr (optimizer.py:30)
    assert abs(O.noam_rate(1, 5120, 1.0, 4000, 0.0) - 5120 ** -0.5 * 4000 ** -1.5) < 1e-15
    p = torch.nn.Parameter(torch.randn(7, 5))
    opt = torch.optim.Adam([p], lr=1e-3, betas=(0.9, 0.98), eps=1e-9)
    m = torch.zeros_like(p); v = torch.zeros_like(p); q = p.detach().clone()
    for step in range(1, 4):
        g = torch.randn_like(p)
        p.grad = g.clone()
        opt.step()
        q, m, v = O.adam_reference(q, g, m, v, step, 1e-3)
        assert torch.allclose(q, p.detach(), rtol=1e-5, atol=1e-7)


def test_greedy_decode_matches_reference_greedy_search():
    """Pins oracle.greedy_decode: the reference's own Decoder.greedy_search output (300 steps, strings cut at EOS; fixture
    generated from the live reference with the Q12 shim) is reproduced id for id."""
    from tests.helpers import cut_at_eos, load_greedy_golden
    cfg, P, enc, ref_ids, ref_len = load_greedy_golden()
    ids, margins = O.greedy_decode(P, cfg, enc, steps=300)
    assert int(ref_len.min()) < 300 <= int(ref_len.max())              # the fixture has both cut and uncut utterances
    for b in range(enc.shape[0]):
        mine = cut_at_eos(ids[b])
        n = int(ref_len[b])
        assert mine == ref_ids[b, :n].tolist(), b
        assert (ref_ids[b, n:] == -1).all()
