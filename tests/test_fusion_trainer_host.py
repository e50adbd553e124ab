"""CPU tests of FusionTrainer's host side (no kernels run): the flat parameter layout stays where it was when the head
moved into the embedded pool trainer (`bench.py --workload fusion --dump-outputs` samples `params` and `grads` at fixed
flat indices, so a moved parameter breaks the comparison of two builds' dumps), `named_grads` names every parameter the
branch trains, and more than 8 classes are refused."""
from argparse import Namespace

import pytest
import torch

ARGS = dict(modality=["CT", "pathology"], model_CT="resnetMC3_18", model_pathology="ABMIL", model_CI="none",
            aggregator="ABMIL", num_classes=2, alignment_base="none", clinical_features=list("abcdefghi"))
POOL_NAMES = ("attention_V.0.weight", "attention_U.0.weight", "attention_V.0.bias", "attention_U.0.bias",
              "attention_weights.weight", "attention_weights.bias")


def _trainer(num_classes=2):
    import mil_b200
    torch.manual_seed(0)
    m = mil_b200.get_model(Namespace(**dict(ARGS, num_classes=num_classes))).eval()
    return mil_b200.FusionTrainer(m, n_text_tokens=1, compute_dtype=torch.float32)


def test_flat_layout_and_named_grads_keep_their_places():
    tr = _trainer()
    m, E, D, C = tr.model, 512, 192, 2
    # the layout as it was written out before the head moved into the pool trainer: fusion program | pool | head.weight
    # | head.bias, each range starting on an 8-element boundary
    up8 = lambda n: (n + 7) // 8 * 8
    n_pool = 2 * D * E + 3 * D + 1
    o_pool = up8(sum(p.numel() for p in tr.tape.params))
    o_head_w = up8(o_pool + n_pool)
    o_head_b = up8(o_head_w + C * E)
    numel = up8(o_head_b + C)
    assert (numel, o_pool, n_pool, o_head_w, o_head_b) == (10054992, 9856768, 197185, 10053960, 10054984)
    assert (tr.numel, tr.o_pool, tr.pool.n_pool) == (numel, o_pool, n_pool)
    pool_at = [o_pool, o_pool + D * E, o_pool + 2 * D * E, o_pool + 2 * D * E + D, o_pool + 2 * D * E + 2 * D,
               o_pool + 2 * D * E + 3 * D]
    want = {n: off for n, off in zip(("aggregator." + k for k in POOL_NAMES), pool_at)}
    want["fc.1.weight"], want["fc.1.bias"] = o_head_w, o_head_b
    names = {id(p): n for n, p in m.named_parameters()}
    for off, p in tr._module_tensors():
        want[names[id(p)]] = off
    got = tr.named_grads()
    assert got.keys() == want.keys()
    params = dict(m.named_parameters())
    for n, g in got.items():
        assert (g.data_ptr() - tr.grads.data_ptr()) // 4 == want[n] and g.shape == params[n].shape, n
    # load_from / store_to move the head through the pool trainer, into and out of the same places
    head = torch.cat([m.fc[1].weight.detach().reshape(-1), m.fc[1].bias.detach()])
    assert torch.equal(tr.params[o_head_w:o_head_b + C], head)
    tr.params[o_head_w:o_head_b + C] += 1.0
    tr.store_to()
    assert torch.equal(torch.cat([m.fc[1].weight.detach().reshape(-1), m.fc[1].bias.detach()]), head + 1.0)


def test_more_than_eight_classes_are_refused():
    with pytest.raises(ValueError, match="1..8 classes"):
        _trainer(num_classes=9)
