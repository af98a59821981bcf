"""Records what the reference's own code computes for the cross-checks that once ran it live, so
that those checks run from the repository alone:

  reference_live_<case>.npz        one per case of tests/test_oracle_reference_live.py: the reference's
                                   models/rank/*/net.py (unmodified, on oracle/paddle_shim.py, float64)
                                   -> `param/<name>`, `in/<name>`, `out` and the gradient of
                                   out.square().sum() per parameter, `grad/<name>`
  reference_criteo_sample.txt      the reference's bundled sample of deepfm / dcn_v2 (the same file)
  reference_din_sample.txt         the reference's bundled DIN sample
  reference_live_readers.npz       what the reference's deepfm/criteo_reader.py, dcn_v2/reader.py and
                                   din/dinReader.py (batch size 8) yield for those two files
  criteo_tsv_parser_cpp_live.txt.gz  what tools/dataset/parser.cpp (compiled unmodified by
                                   oracle/Makefile) prints for the seeded TSV of
                                   tests/test_dataio.py::_random_criteo_tsv

usage: python tests/golden/make_live_golden.py <reference checkout>
"""
import gzip
import importlib.util
import os
import shutil
import subprocess
import sys
import tempfile

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)

from oracle import paddle_shim  # noqa: E402


def _record(cases, case, named, inputs, pred):
    out = cases[case] = {}
    gs = torch.autograd.grad(pred.square().sum(), list(named.values()), allow_unused=True)
    for (k, p), g in zip(named.items(), gs):
        out["param/" + k] = p.detach().numpy()
        out["grad/" + k] = (torch.zeros_like(p) if g is None else g).detach().numpy()
    for k, v in inputs.items():
        out["in/" + k] = v.numpy()
    out["out"] = pred.detach().numpy()


def nets(ref_root):
    """Same seeds, shapes and call order as the live test had."""
    torch.set_default_dtype(torch.float64)
    net = lambda m: paddle_shim.import_reference_net(m, ref_root)  # noqa: E731
    out = {}
    for seed, D, B in [(1, 5, 3), (2, 12, 9)]:
        torch.manual_seed(seed)
        V, fc = 61, [7, 5, 3]
        layer = net("deepfm").DeepFMLayer(V, D, 13, 26, fc)
        ids = [torch.randint(0, V, (B, 1)) for _ in range(26)]
        dense = torch.rand(B, 13)
        _record(out, "deepfm_%d" % seed, dict(layer.named_parameters()),
                {"ids": torch.cat(ids, 1), "dense": dense}, layer(ids, dense))

    for mix, stacked in [(False, False), (True, True)]:
        torch.manual_seed(11)
        V, D, B, fc = 43, 3, 5, [9, 6]
        layer = net("dcn_v2").DCN_V2Layer(V, D, 13, 26, fc, 3, stacked, mix, 4, 2)
        layer.eval()
        ids = [torch.randint(0, V, (B, 1)) for _ in range(26)]
        dense = torch.rand(B, 13)
        _record(out, "dcn_v2_%d%d" % (mix, stacked), dict(layer.named_parameters()),
                {"ids": torch.cat(ids, 1), "dense": dense}, layer(ids, dense))

    torch.manual_seed(5)
    V, D, B, fc = 37, 6, 4, [8, 4]
    layer = net("wide_deep").WideDeepLayer(V, D, 13, 26, fc)
    ids = [torch.randint(0, V, (B, 1)) for _ in range(26)]
    dense = torch.rand(B, 13)
    _record(out, "wide_deep", dict(layer.named_parameters()),
            {"ids": torch.cat(ids, 1), "dense": dense}, layer(ids, dense))

    layer = net("din").DINLayer(4, 4, "sigmoid", False, False, 29, 7)
    B, L = 3, 5
    hi, hc = torch.randint(0, 29, (B, L)), torch.randint(0, 7, (B, L))
    ti, tc = torch.randint(0, 29, (B,)), torch.randint(0, 7, (B,))
    mask = torch.zeros(B, L, 1, dtype=torch.int64)
    mask[1, 3:] = int(-1e9)
    named = dict(layer.named_parameters())
    # the attention-unit linears are hidden from named_parameters() by a name collision
    for i, m in enumerate([m for m in layer.attention_layer if hasattr(m, "weight")]):
        named["att.linear_%d.weight" % i], named["att.linear_%d.bias" % i] = m.weight, m.bias
    args = (hi, hc, ti, tc, None, mask, ti.unsqueeze(1).repeat(1, L), tc.unsqueeze(1).repeat(1, L))
    _record(out, "din", named, {"hist_item": hi, "hist_cat": hc, "target_item": ti,
                                "target_cat": tc, "mask": mask}, layer(*args))

    for self_interaction, B, d in [(False, 6, 4), (True, 9, 8)]:
        torch.manual_seed(21 + B)
        V, bot, top = 53, [10, d], [12, 2]
        layer = net("dlrm").DLRMLayer(13, bot, V, d, top, 26, self_interaction=self_interaction)
        layer.train()
        ids = [torch.randint(0, V, (B, 1)) for _ in range(26)]
        dense = torch.rand(B, 13)
        _record(out, "dlrm_%d" % self_interaction, dict(layer.named_parameters()),
                {"ids": torch.cat(ids, 1), "dense": dense}, layer(ids, dense))
    torch.set_default_dtype(torch.float32)
    return out


def _load(path, name):
    spec = importlib.util.spec_from_file_location(name, path)
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def readers(ref_root):
    paddle_shim.install()
    rank = os.path.join(ref_root, "models", "rank")
    criteo = os.path.join(HERE, "reference_criteo_sample.txt")
    din = os.path.join(HERE, "reference_din_sample.txt")
    shutil.copyfile(os.path.join(rank, "deepfm/data/sample_data/train/sample_train.txt"), criteo)
    with open(os.path.join(rank, "dcn_v2/data/sample_data/sample_train.txt"), "rb") as a, \
            open(criteo, "rb") as b:
        assert a.read() == b.read()
    shutil.copyfile(os.path.join(rank, "din/data/train_data/sample_data.txt"), din)

    out = {}
    ds = _load(os.path.join(rank, "deepfm/criteo_reader.py"), "ref_criteo_reader").RecDataset([criteo], None)
    ds.inference = False
    rows = list(ds)
    out["deepfm/ids"] = np.stack([np.concatenate(r[:27]) for r in rows])
    out["deepfm/dense"] = np.stack([r[27] for r in rows])

    rows = list(_load(os.path.join(rank, "dcn_v2/reader.py"), "ref_dcn_reader").RecDataset([criteo], None))
    out["dcn_v2/ids"] = np.stack([np.concatenate(r[1:27]) for r in rows])
    out["dcn_v2/dense"] = np.stack([r[27] for r in rows])

    cwd = os.getcwd()
    os.chdir(tempfile.mkdtemp())                         # dinReader.py writes ./tmp.txt
    try:
        rd = _load(os.path.join(rank, "din/dinReader.py"), "ref_din_reader")
        samples = list(rd.RecDataset([din], {"runner.train_batch_size": 8}))
    finally:
        os.chdir(cwd)
    out["din/n_samples"] = np.asarray(len(samples))
    for b in range(len(samples) // 8):
        for j in range(8):
            out["din/b%d/%d" % (b, j)] = np.stack([np.asarray(s[j]) for s in samples[8 * b:8 * b + 8]])
    return out


def parser_cpp(ref_root):
    from tests.test_dataio import _random_criteo_tsv

    subprocess.run(["make", "-s", "-C", os.path.join(ROOT, "oracle"), "REF=" + ref_root], check=True)
    exe = os.path.join(ROOT, "oracle", "_ref", "criteo_parser")
    return subprocess.run([exe], input=_random_criteo_tsv(), capture_output=True, check=True).stdout


def main():
    ref_root = os.path.abspath(sys.argv[1])
    for case, arrays in nets(ref_root).items():
        np.savez_compressed(os.path.join(HERE, "reference_live_%s.npz" % case), **arrays)
    np.savez_compressed(os.path.join(HERE, "reference_live_readers.npz"), **readers(ref_root))
    with gzip.GzipFile(os.path.join(HERE, "criteo_tsv_parser_cpp_live.txt.gz"), "wb", mtime=0) as fh:
        fh.write(parser_cpp(ref_root))
    for f in sorted(os.listdir(HERE)):
        if f.startswith(("reference_", "criteo_tsv_parser_cpp_live")):
            print("%-36s %8.1f KB" % (f, os.path.getsize(os.path.join(HERE, f)) / 1024))


if __name__ == "__main__":
    main()
