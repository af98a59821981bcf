"""Cross-check with fresh seeds and shapes: what the reference's own models/rank/*/net.py and readers
computed, executed unmodified on oracle/paddle_shim.py (recorded by tests/golden/make_live_golden.py),
against oracle/nets.py, oracle/readers.py and the native parsers — forward and every parameter
gradient, float64."""
import os

import numpy as np
import pytest
import torch

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


@pytest.fixture(autouse=True)
def _f64():
    prev = torch.get_default_dtype()
    torch.set_default_dtype(torch.float64)
    yield
    torch.set_default_dtype(prev)


def _case(name):
    """(parameters as float64 leaves, inputs, reference output, reference gradients) of one case."""
    z = np.load(os.path.join(GOLD, "reference_live_%s.npz" % name))
    part = {"param": {}, "in": {}, "grad": {}}
    for k in z.files:
        if k != "out":
            group, _, key = k.partition("/")
            part[group][key] = z[k]
    named = {k: torch.tensor(v).requires_grad_(True) for k, v in part["param"].items()}
    inputs = {k: torch.tensor(v) for k, v in part["in"].items()}
    return named, inputs, z["out"], part["grad"]


def _slots(ids):
    return [ids[:, i:i + 1] for i in range(ids.shape[1])]


def _same(ref_out, ref_grads, ora_out, named):
    assert np.abs(ref_out - ora_out.detach().numpy()).max() < 1e-12
    gs = torch.autograd.grad(ora_out.square().sum(), list(named.values()), allow_unused=True)
    got = {k: (torch.zeros_like(p) if g is None else g) for (k, p), g in zip(named.items(), gs)}
    assert set(got) == set(ref_grads)
    for k in ref_grads:
        assert np.abs(ref_grads[k] - got[k].numpy()).max() < 1e-10, k


@pytest.mark.parametrize("seed,D,B", [(1, 5, 3), (2, 12, 9)])
def test_deepfm_live(seed, D, B):
    from oracle import nets
    named, i, out, grads = _case("deepfm_%d" % seed)
    assert i["ids"].shape == (B, 26) and named["fm.embedding.weight"].shape[1] == D
    _same(out, grads, nets.deepfm_forward(named, _slots(i["ids"]), i["dense"], 3), named)


@pytest.mark.parametrize("mix,stacked", [(False, False), (True, True)])
def test_dcn_v2_live(mix, stacked):
    from oracle import nets
    named, i, out, grads = _case("dcn_v2_%d%d" % (mix, stacked))
    ora = nets.dcn_v2_forward(named, _slots(i["ids"]), i["dense"], n_fc=2, cross_num=3,
                              is_stacked=stacked, use_low_rank_mixture=mix, num_experts=2)
    _same(out, grads, ora, named)


def test_din_and_wide_deep_live():
    from oracle import nets
    named, i, out, grads = _case("wide_deep")
    _same(out, grads, nets.wide_deep_forward(named, _slots(i["ids"]), i["dense"], 2), named)

    named, i, out, grads = _case("din")
    assert "att.linear_0.weight" in named
    L = i["hist_item"].shape[1]
    ti, tc = i["target_item"], i["target_cat"]
    args = (i["hist_item"], i["hist_cat"], ti, tc, None, i["mask"], ti.unsqueeze(1).repeat(1, L),
            tc.unsqueeze(1).repeat(1, L))
    _same(out, grads, nets.din_forward(named, *args), named)


@pytest.mark.parametrize("self_interaction,B,d", [(False, 6, 4), (True, 9, 8)])
def test_dlrm_live(self_interaction, B, d):
    """dlrm/net.py unmodified (train mode: BatchNorm on batch statistics), incl. the
    self_interaction=True branch whose diagonal entries evaluate to 0."""
    from oracle import nets
    named, i, out, grads = _case("dlrm_%d" % self_interaction)
    assert i["ids"].shape == (B, 26) and named["embedding.weight"].shape[1] == d
    ora = nets.dlrm_forward(named, _slots(i["ids"]), i["dense"], n_bot=2, n_top=2,
                            self_interaction=self_interaction)
    _same(out, grads, ora, named)


def test_readers_live():
    """The reference's three Python readers on the reference's own bundled sample files, against
    oracle/readers.py and the native parsers."""
    from oracle import readers
    from paddlerec_b200 import dataio

    gold = np.load(os.path.join(GOLD, "reference_live_readers.npz"))
    sample = os.path.join(GOLD, "reference_criteo_sample.txt")
    ids_ref, dense_ref = gold["deepfm/ids"], gold["deepfm/dense"]
    label, ids, dense = dataio.parse_slot_text(open(sample, "rb").read())
    assert np.array_equal(label[:, 0], ids_ref[:, 0]) and np.array_equal(ids, ids_ref[:, 1:])
    assert np.array_equal(dense, dense_ref)
    oi, od = readers.slot_text_packed(open(sample).read().split("\n"), ["click"] + [str(i) for i in range(1, 27)],
                                      "dense_feature", 13)
    assert np.array_equal(oi, ids_ref) and np.array_equal(od, dense_ref)

    label, ids, dense = dataio.parse_slot_text(open(sample, "rb").read(), dataio.CRITEO_DCN_V2)
    assert np.array_equal(ids, gold["dcn_v2/ids"])
    # log(v+1): numpy's and libm's double log may differ in the last place before the float32 cast
    assert np.allclose(dense, gold["dcn_v2/dense"], rtol=2e-7, atol=0)

    din_sample = os.path.join(GOLD, "reference_din_sample.txt")
    batches = list(dataio.DinBatchReader([din_sample], 8, as_torch=False))
    assert len(batches) == int(gold["din/n_samples"]) // 8 > 0
    for b, batch in enumerate(batches):
        for j in range(8):
            assert np.array_equal(batch[j], gold["din/b%d/%d" % (b, j)]), (b, j)
