"""libb200rec_io.so (include/b200rec_io.h) against the reference's own readers.

Pinned parity for this row: the goldens under tests/golden/ were produced by the reference's code
itself (tools/dataset/parser.cpp compiled unmodified; models/rank/deepfm/criteo_reader.py imported
unmodified) — see tests/golden/make_reader_golden.py.  Integer output (ids, labels, offsets) must
be bit-exact; float32 dense values bit-exact against the Python reader, and within the 6
significant digits parser.cpp prints against its text output.
"""
import gzip
import os

import numpy as np
import pytest

from oracle import readers
from paddlerec_b200 import dataio

HERE = os.path.dirname(os.path.abspath(__file__))
GOLD = os.path.join(HERE, "golden")
ROOT = os.path.dirname(HERE)
CRITEO_SPARSE = ["click"] + [str(i) for i in range(1, 27)]


def _read(name, mode="rb"):
    with open(os.path.join(GOLD, name), mode) as fh:
        return fh.read()


def test_library_exports_every_declared_symbol():
    lib = dataio.load()
    declared = dataio.declared_symbols()
    assert len(declared) == 11 and set(declared) == set(dataio._SIG)
    for name in declared:
        assert hasattr(lib, name), name
    assert lib.b200rec_io_abi_version() == dataio.IO_ABI_VERSION


def test_plain_and_ex_entry_points_agree_through_raw_ctypes():
    """The Python binding always calls the _ex entry point; the plain one must stay equivalent
    (flags = 0) for C callers that bind the shorter signature."""
    import ctypes
    lib = dataio.load()
    text = _read("slot_text_sample.txt")
    n_lines = dataio.count_lines(text)
    names = (ctypes.c_char_p * 26)(*[str(i).encode() for i in range(1, 27)])
    outs = []
    for ex in (False, True):
        label = np.empty((n_lines, 1), np.int64)
        ids = np.empty((n_lines, 26), np.int64)
        dense = np.empty((n_lines, 13), np.float32)
        n = ctypes.c_int64()
        args = [text, len(text), b"click", names, 26, b"dense_feature", 13]
        if ex:
            args.append(0)
        args += [label.ctypes.data, ids.ctypes.data, dense.ctypes.data, n_lines, ctypes.byref(n), 2]
        fn = lib.b200rec_io_parse_slot_text_ex if ex else lib.b200rec_io_parse_slot_text
        assert fn(*args) == 0, lib.b200rec_io_last_error()
        outs.append((n.value, label.copy(), ids.copy(), dense.copy()))
    assert outs[0][0] == outs[1][0] == 48
    assert all(np.array_equal(a, b) for a, b in zip(outs[0][1:], outs[1][1:]))
    bad = ctypes.c_int64()
    assert lib.b200rec_io_parse_slot_text_ex(text, len(text), b"click", names, 26, b"dense_feature", 13,
                                             64, None, outs[0][2].ctypes.data, None, 48,
                                             ctypes.byref(bad), 1) == -1          # unknown flag
    assert b"unknown flags" in lib.b200rec_io_last_error()


# ---- hashes ---------------------------------------------------------------------------------------
def test_xxh32_published_vectors():
    # test vectors of the xxHash specification / reference implementation (seed 0 and a prime seed)
    kat = [(b"", 0, 0x02CC5D05), (b"", 1, 0x0B2CB792), (b"a", 0, 0x550D7456), (b"abc", 0, 0x32D153FF),
           (b"Nobody inspects the spammish repetition", 0, 0xE2293B2F)]
    for s, seed, want in kat:
        assert readers.xxh32(s, seed) == want, s
        assert dataio.xxh32(s, seed) == want, s
    rng = np.random.default_rng(0)
    for n in list(range(0, 40)) + [63, 64, 65, 255]:
        s = rng.integers(0, 256, n, dtype=np.uint8).tobytes()
        assert dataio.xxh32(s, 7) == readers.xxh32(s, 7)


def test_std_hash_matches_restatement():
    rng = np.random.default_rng(1)
    for n in list(range(0, 26)) + [31, 32, 33, 100]:
        s = rng.integers(1, 256, n, dtype=np.uint8).tobytes()
        assert dataio.hash_std_string(s) == readers.std_hash_string(s)


# ---- raw Criteo TSV vs the reference's parser.cpp ---------------------------------------------------
def _parser_cpp_output(text: bytes):
    rows = readers.multislot_lines(text.decode().split("\n"), [True] + [False] * 27)
    dense = np.asarray([r[0] for r in rows], np.float64)
    ids = np.asarray([[s[0] for s in r[1:27]] for r in rows], np.int64)
    label = np.asarray([r[27][0] for r in rows], np.int64)
    return label, ids, dense


def test_criteo_tsv_matches_golden_from_reference_parser_cpp():
    tsv = _read("criteo_tsv_sample.tsv")
    label, ids, dense, skipped = dataio.parse_criteo_tsv(tsv)
    rl, rid, rd = _parser_cpp_output(_read("criteo_tsv_parser_cpp.txt"))
    assert skipped == 2 and ids.shape == (62, 26)
    assert np.array_equal(ids, rid)
    assert np.array_equal(label[:, 0], rl)
    assert np.allclose(dense, rd, rtol=1e-5, atol=1e-9)      # cout prints 6 significant digits
    ol, oi, od, osk = readers.criteo_tsv_lines(tsv.decode().split("\n"))
    assert osk == 2 and np.array_equal(oi, ids) and np.array_equal(ol, label[:, 0])
    assert np.array_equal(od, dense)                          # bit-exact vs the restatement


def _random_criteo_tsv():
    rng = np.random.default_rng(5)
    lines = []
    for _ in range(700):
        cols = [str(rng.integers(0, 2))]
        cols += ["" if rng.random() < 0.3 else str(rng.integers(-3, 70000)) for _ in range(13)]
        cols += ["" if rng.random() < 0.2 else "%x" % rng.integers(0, 1 << 40) for _ in range(26)]
        lines.append("\t".join(cols))
    return ("\n".join(lines) + "\n").encode()


def test_criteo_tsv_matches_reference_binary_live():
    """700 seeded lines against what parser.cpp printed for them (tests/golden/make_live_golden.py)."""
    tsv = _random_criteo_tsv()
    rl, rid, rd = _parser_cpp_output(gzip.decompress(_read("criteo_tsv_parser_cpp_live.txt.gz")))
    assert rid.shape == (700, 26)
    for threads in (1, 3):
        label, ids, dense, skipped = dataio.parse_criteo_tsv(tsv, threads=threads)
        assert skipped == 0 and np.array_equal(ids, rid) and np.array_equal(label[:, 0], rl)
        assert np.allclose(dense, rd, rtol=1e-5, atol=1e-9)


def test_criteo_tsv_xxh32_kind_matches_benchmark_reader_restatement():
    tsv = _read("criteo_tsv_sample.tsv").decode().split("\n")
    good = "\n".join(l for l in tsv if l.count("\t") == 39) + "\n"
    label, ids, dense, skipped = dataio.parse_criteo_tsv(good, dataio.HASH_XXH32, hash_dim=1000001)
    ol, oi, od, _ = readers.criteo_tsv_lines(good.split("\n"), "xxh32")
    assert np.array_equal(ids, oi) and np.array_equal(label[:, 0], ol) and np.array_equal(dense, od)
    assert ids.min() >= 0 and ids.max() < 1000001
    with pytest.raises(dataio.B200RecIOError, match="fewer than 40 columns"):
        dataio.parse_criteo_tsv("1\t2\t3\n", dataio.HASH_XXH32)   # line_process would IndexError


# ---- slot text vs the reference's criteo_reader.py -------------------------------------------------
def test_slot_text_matches_golden_from_reference_reader():
    text = _read("slot_text_sample.txt")
    gold = np.load(os.path.join(GOLD, "slot_text_criteo_reader.npz"))
    for threads in (1, 4):
        label, ids, dense = dataio.parse_slot_text(text, threads=threads)
        assert np.array_equal(label[:, 0], gold["ids"][:, 0])
        assert np.array_equal(ids, gold["ids"][:, 1:])
        assert np.array_equal(dense, gold["dense"])          # float32 bit-exact
    oi, od = readers.slot_text_packed(text.decode().split("\n"), CRITEO_SPARSE, "dense_feature", 13)
    assert np.array_equal(oi, gold["ids"]) and np.array_equal(od, gold["dense"])


def test_slot_text_matches_python_reader_on_bundled_sample():
    from paddlerec_b200.rank.deepfm import criteo_reader

    path = os.path.join(ROOT, "paddlerec_b200", "rank", "deepfm", "data", "sample_data", "train",
                        "sample_train.txt")
    samples = list(criteo_reader.RecDataset([path]))
    label, ids, dense = dataio.parse_slot_text(open(path, "rb").read())
    assert np.array_equal(label[:, 0], np.stack([s[0] for s in samples])[:, 0])
    assert np.array_equal(ids, np.stack([np.concatenate(s[1:27]) for s in samples]))
    assert np.array_equal(dense, np.stack([s[27] for s in samples]))


def test_slot_text_thread_count_does_not_change_the_result():
    rng = np.random.default_rng(2)
    lines = []
    for _ in range(5000):
        toks = ["click:%d" % rng.integers(0, 2)]
        toks += ["dense_feature:%.9g" % rng.random() for _ in range(13)]
        toks += ["%d:%d" % (s, rng.integers(0, 1 << 40)) for s in range(1, 27) if rng.random() > 0.05]
        lines.append(" ".join(toks))
    text = "\n".join(lines).encode()                        # no trailing newline on purpose
    ref = dataio.parse_slot_text(text, threads=1)
    for threads in (2, 5, 8, 0):
        got = dataio.parse_slot_text(text, threads=threads)
        assert all(np.array_equal(a, b) for a, b in zip(ref, got))
    oi, od = readers.slot_text_packed(lines[:300], CRITEO_SPARSE, "dense_feature", 13)
    assert np.array_equal(ref[1][:300], oi[:, 1:]) and np.array_equal(ref[2][:300], od)


def test_slot_text_edge_cases():
    sch = dataio.SlotSchema(sparse_slots=("a", "b"), label_slot="y", dense_slot="d", dense_dim=2)
    lab, ids, dense = dataio.parse_slot_text("\n\n  \ny:1 a:5 d:0.5 d:1e-3 b:-7\n\nb:+3\n", sch)
    assert lab.tolist() == [[1], [0]] and ids.tolist() == [[5, -7], [0, 3]]
    assert np.array_equal(dense, np.asarray([[0.5, 1e-3], [0, 0]], np.float32))   # missing dense -> zeros
    lab, ids, dense = dataio.parse_slot_text("", sch)
    assert ids.shape == (0, 2) and dense.shape == (0, 2)
    # "a:1:2".split(":")[1] == "1"; a second ':' part is ignored like the reference does
    assert dataio.parse_slot_text("a:1:2 b:9", sch)[1].tolist() == [[1, 9]]
    # values float32 cannot hold exactly round like numpy's astype
    _, _, dense = dataio.parse_slot_text("d:0.1 d:16777217", sch)
    assert np.array_equal(dense, np.asarray([[0.1, 16777217.0]], np.float64).astype(np.float32))
    _, _, dense = dataio.parse_slot_text("d:1e400 d:-1e-400", sch)                # Python: inf, -0.0
    assert np.isposinf(dense[0, 0]) and dense[0, 1] == 0
    no_label = dataio.SlotSchema(sparse_slots=("a",), label_slot=None, dense_slot=None)
    lab, ids, dense = dataio.parse_slot_text("a:4 y:1 d:3", no_label)
    assert lab is None and dense is None and ids.tolist() == [[4]]


def test_slot_text_errors_name_the_line():
    sch = dataio.SlotSchema(sparse_slots=("a", "b"), label_slot="y", dense_slot="d", dense_dim=2)
    with pytest.raises(dataio.B200RecIOError, match="line 2: bad integer") as e:
        dataio.parse_slot_text("a:1\na:x1\n", sch)
    assert e.value.code == -2
    with pytest.raises(dataio.B200RecIOError, match="line 1: bad float"):
        dataio.parse_slot_text("d:zz d:1\n", sch)
    with pytest.raises(dataio.B200RecIOError, match="without ':value'"):
        dataio.parse_slot_text("a b:1\n", sch)
    with pytest.raises(dataio.B200RecIOError, match="second value") as e:
        dataio.parse_slot_text("a:1 a:2\n", sch)            # multi-hot needs the _lod entry point
    assert e.value.code == -4
    with pytest.raises(dataio.B200RecIOError, match="shorter than dense_dim"):
        dataio.parse_slot_text("d:1\n", sch)
    with pytest.raises(dataio.B200RecIOError, match="too many dense"):
        dataio.parse_slot_text("d:1 d:2 d:3\n", sch)
    out = (np.empty((1, 1), np.int64), np.empty((1, 2), np.int64), np.empty((1, 2), np.float32))
    with pytest.raises(dataio.B200RecIOError, match="cap = 1") as e:
        dataio.parse_slot_text("a:1\na:2\n", sch, out=out)
    assert e.value.code == -3
    # the first bad line (in file order) is the one reported, whatever the thread count
    lines = ["a:%d" % i for i in range(4000)]
    lines[1234] = "a:oops"
    lines[3456] = "a:later"
    with pytest.raises(dataio.B200RecIOError, match="line 1235:"):
        dataio.parse_slot_text("\n".join(lines), sch, threads=8)


def test_slot_text_lod_matches_restatement():
    rng = np.random.default_rng(3)
    slots = ["s%d" % i for i in range(5)]
    lines = []
    for _ in range(1500):
        toks = ["y:%d" % rng.integers(0, 2)]
        for s in slots:
            toks += ["%s:%d" % (s, rng.integers(0, 10**12)) for _ in range(rng.integers(0, 4))]
        toks += ["d:%r" % float(rng.random()) for _ in range(3)]
        rng.shuffle(toks[1:-3])
        lines.append(" ".join(toks))
    sch = dataio.SlotSchema(sparse_slots=tuple(slots), label_slot="y", dense_slot="d", dense_dim=3)
    want = readers.slot_text_lines(lines, ["y"] + slots, "d", 3)
    for threads in (1, 4):
        label, keys, offsets, dense = dataio.parse_slot_text_lod("\n".join(lines), sch, threads=threads)
        assert offsets[0] == 0 and offsets[-1] == keys.size and np.all(np.diff(offsets) >= 1)
        flat = [v for r in want for bag in r[1:-1] for v in bag]
        lens = [len(bag) for r in want for bag in r[1:-1]]
        assert keys.tolist() == flat and np.diff(offsets).tolist() == lens
        assert label[:, 0].tolist() == [r[0][0] for r in want]
        assert np.array_equal(dense, np.asarray([r[-1] for r in want], np.float64).astype(np.float32))


def test_multislot_roundtrip_through_reference_parser_output():
    # parser.cpp's stdout IS the multislot wire format: parsing it must give back what the TSV
    # parser produced directly (ids exact; feasigns are uint64)
    text = _read("criteo_tsv_parser_cpp.txt")
    got = dataio.parse_multislot(text, [True] + [False] * 27, threads=2)
    label, ids, dense, _ = dataio.parse_criteo_tsv(_read("criteo_tsv_sample.tsv"))
    n = got["n"]
    assert n == 62 and got["keys"].dtype == np.uint64
    keys = got["keys"].reshape(n, 27)
    assert np.array_equal(keys[:, :26].astype(np.int64), ids) and np.array_equal(keys[:, 26].astype(np.int64), label[:, 0])
    assert np.array_equal(got["key_offsets"], np.arange(n * 27 + 1))
    assert np.array_equal(got["float_offsets"], np.arange(n + 1) * 13)
    assert np.allclose(got["fvals"].reshape(n, 13), dense, rtol=1e-5, atol=1e-9)


def test_multislot_variable_length_and_errors():
    # the example of tools/dataset/README.MD: 4 slots per line, counts 2,2,2,2 ...
    text = "2 1 2 2 5 4 2 2 7 2 1 3\n2 6 2 2 1 4 2 2 4 2 2 3\n"
    got = dataio.parse_multislot(text, [False] * 4)
    assert got["keys"].tolist() == [1, 2, 5, 4, 2, 7, 1, 3, 6, 2, 1, 4, 2, 4, 2, 3]
    assert got["key_offsets"].tolist() == list(range(0, 17, 2))
    got = dataio.parse_multislot("3 1 2 3 1 0.5\n1 18446744073709551615 2 1.5 2.5\n", [False, True])
    assert got["keys"].tolist() == [1, 2, 3, 18446744073709551615]
    assert got["key_offsets"].tolist() == [0, 3, 4] and got["float_offsets"].tolist() == [0, 1, 3]
    want = readers.multislot_lines(["3 1 2 3 1 0.5", "1 18446744073709551615 2 1.5 2.5"], [False, True])
    assert want == [[[1, 2, 3], [0.5]], [[18446744073709551615], [1.5, 2.5]]]
    with pytest.raises(dataio.B200RecIOError, match="positive integer"):
        dataio.parse_multislot("0 1 5\n", [False, False])
    with pytest.raises(dataio.B200RecIOError, match="line ends inside slot"):
        dataio.parse_multislot("2 1\n", [False])
    with pytest.raises(dataio.B200RecIOError, match="tokens left"):
        dataio.parse_multislot("1 1 9\n", [False])


# ---- batch reader ---------------------------------------------------------------------------------
def _write_files(tmp_path, n_files=3, n_lines=(700, 1, 333)):
    rng = np.random.default_rng(4)
    paths, all_lines = [], []
    for k in range(n_files):
        lines = []
        for _ in range(n_lines[k]):
            toks = ["click:%d" % rng.integers(0, 2)] + ["dense_feature:%.6f" % rng.random() for _ in range(13)]
            toks += ["%d:%d" % (s, rng.integers(1, 10**6)) for s in range(1, 27)]
            lines.append(" ".join(toks))
        p = tmp_path / ("part-%d.txt" % k)
        p.write_text("\n".join(lines) + ("\n" if k != 1 else ""))
        paths.append(str(p))
        all_lines += lines
    return paths, all_lines


def test_packed_batch_reader_matches_dataloader_order(tmp_path):
    import torch

    paths, all_lines = _write_files(tmp_path)
    oi, od = readers.slot_text_packed(all_lines, CRITEO_SPARSE, "dense_feature", 13)
    for chunk, prefetch in ((1 << 12, 2), (1 << 24, 0)):       # chunks smaller / larger than a file
        rd = dataio.PackedBatchReader(paths[::-1], batch_size=128, chunk_bytes=chunk, prefetch=prefetch)
        batches = list(rd)
        assert len(batches) == len(all_lines) // 128            # drop_last
        label = torch.cat([b[0] for b in batches]).numpy()
        ids = torch.cat([b[1] for b in batches]).numpy()
        dense = torch.cat([b[2] for b in batches]).numpy()
        n = len(batches) * 128
        assert batches[0][1].shape == (128, 26) and batches[0][1].dtype == torch.int64
        assert np.array_equal(label[:, 0], oi[:n, 0]) and np.array_equal(ids, oi[:n, 1:])
        assert np.array_equal(dense, od[:n])
    rd = dataio.PackedBatchReader(paths, batch_size=1000, drop_last=False, as_torch=False)
    sizes = [b[1].shape[0] for b in rd]
    assert sizes == [1000, 34]
    # rank sharding of FILES like criteo_reader.py:30-43
    r1 = dataio.PackedBatchReader(paths, batch_size=1, rank=1, world_size=2, shard_files=True, as_torch=False)
    assert sum(1 for _ in r1) == 1
    with pytest.raises(ValueError, match="less than the number of workers"):
        dataio.PackedBatchReader(paths, batch_size=1, rank=0, world_size=4, shard_files=True)


def test_packed_batch_reader_surfaces_parse_errors(tmp_path):
    p = tmp_path / "bad.txt"
    p.write_text("click:1 1:5\nclick:x 1:6\n")
    with pytest.raises(dataio.B200RecIOError, match="line 2"):
        list(dataio.PackedBatchReader([str(p)], batch_size=1))


def test_packed_cache_roundtrip(tmp_path):
    paths, all_lines = _write_files(tmp_path)
    label, ids, dense = dataio.parse_slot_text(open(paths[0], "rb").read())
    cache = str(tmp_path / "part-0.b2r")
    dataio.write_packed(cache, label, ids, dense)
    l2, i2, d2 = dataio.read_packed(cache)
    assert np.array_equal(l2, label) and np.array_equal(i2, ids) and np.array_equal(d2, dense)
    rd = dataio.PackedBatchReader([cache], batch_size=100, fmt="packed", as_torch=False, prefetch=0)
    got = np.concatenate([b[1] for b in rd])
    assert np.array_equal(got, ids)
    with pytest.raises(ValueError, match="not a b200rec packed file"):
        dataio.read_packed(paths[0])


def test_dygraph_model_consumes_packed_batches(tmp_path):
    """The packed triple is what DygraphModel.create_feeds takes (dygraph_model.py:41-50 mirror)."""
    import torch

    from paddlerec_b200.rank.deepfm.dygraph_model import DygraphModel

    paths, _ = _write_files(tmp_path, n_lines=(64, 1, 1))
    batch = next(iter(dataio.PackedBatchReader(paths[:1], batch_size=32, prefetch=0)))
    cfg = {"hyper_parameters.sparse_inputs_slots": 27, "hyper_parameters.dense_input_dim": 13}
    dm = DygraphModel()
    dm.device = "cpu"
    label, ids, dense = dm.create_feeds(batch, cfg)
    assert label.shape == (32, 1) and dense.shape == (32, 13) and dense.dtype == torch.float32
    assert ids.shape == (32, 26) and torch.equal(ids, batch[1])


# ---- DIN behaviour logs vs the reference's dinReader.py ---------------------------------------------
DIN_FIELDS = ["hist_item", "hist_cat", "target_item", "target_cat", "label", "mask", "target_item_seq",
              "target_cat_seq"]


def test_din_batches_match_golden_from_reference_reader():
    gold = np.load(os.path.join(GOLD, "din_reader_batches.npz"))
    rd = dataio.DinBatchReader([os.path.join(GOLD, "din_sample.txt")], batch_size=3, as_torch=False)
    batches = list(rd)
    assert len(batches) == 25                      # 60-record group + 17-record tail minus 2
    for b, batch in enumerate(batches):
        for j, name in enumerate(DIN_FIELDS):
            want = gold["b%d/%s" % (b, name)]
            assert batch[j].shape == want.shape and batch[j].dtype == want.dtype, (b, name)
            assert np.array_equal(batch[j], want), (b, name)
    # lengths are sorted inside a group, every batch is padded to its own maximum
    Ls = [b[0].shape[1] for b in batches]
    assert Ls[:20] == sorted(Ls[:20]) and Ls[20:] == sorted(Ls[20:]) and Ls[19] > Ls[20]
    assert batches[0][5].min() in (0, int(-1e9)) and batches[-1][5].dtype == np.int64


def test_din_native_reader_matches_python_reader_through_the_dataloader():
    import torch

    from paddlerec_b200 import runner

    d = os.path.join(ROOT, "paddlerec_b200", "rank", "din")
    cfg = runner.load_yaml(os.path.join(d, "config.yaml"))
    cfg["config_abs_dir"] = d
    for bs in (32, 2):                             # bs=2: 100 records = 2 full groups + a tail of 20
        cfg["runner.train_batch_size"] = bs
        plain = list(runner.create_data_loader(cfg))
        native = list(dataio.DinBatchReader([os.path.join(d, "data", "train_data", "sample_data.txt")], bs))
        assert len(plain) == len(native) == 100 // bs
        for a, b in zip(plain, native):
            for j in range(8):
                assert torch.equal(a[j], b[j]) and a[j].dtype == b[j].dtype, j


def test_din_parse_edge_cases():
    r = dataio.parse_din("1 2;3 4;5;6;1\nbroken;line\n\n 7 ; 8 ;9; 10 ;0.5;extra;fields\n")
    assert r["n_skipped"] == 1 and r["offsets"].tolist() == [0, 2, 3]
    assert r["hist_items"].tolist() == [1, 2, 7] and r["hist_cats"].tolist() == [3, 4, 8]
    assert r["target_item"].tolist() == [5, 9] and r["target_cat"].tolist() == [6, 10]
    assert r["label"].tolist() == [1.0, 0.5]
    with pytest.raises(dataio.B200RecIOError, match="differ in length") as e:
        dataio.parse_din("1 2 3;4 5;6;7;1\n")
    assert e.value.code == -4
    with pytest.raises(dataio.B200RecIOError, match="line 2: bad id"):
        dataio.parse_din("1;2;3;4;1\n1 x;2 3;3;4;0\n")
    with pytest.raises(dataio.B200RecIOError, match="bad label"):
        dataio.parse_din("1;2;3;4;yes\n")
    # thread count does not change the result
    rng = np.random.default_rng(8)
    lines = []
    for _ in range(4000):
        k = int(rng.integers(1, 30))
        lines.append("%s;%s;%d;%d;%d" % (" ".join(map(str, rng.integers(1, 10**6, k))),
                                        " ".join(map(str, rng.integers(1, 800, k))),
                                        rng.integers(1, 10**6), rng.integers(1, 800), rng.integers(0, 2)))
    text = "\n".join(lines)
    a, b = dataio.parse_din(text, threads=1), dataio.parse_din(text, threads=8)
    assert all(np.array_equal(a[k], b[k]) for k in a if k != "n_skipped")
    assert a["offsets"][-1] == a["hist_items"].size == a["hist_cats"].size


def test_pack_dataset_tool_and_packed_training_input(tmp_path):
    """tools/pack_dataset.py: text -> .b2r once; the packed reader then yields the same batches as
    the text reader, and runner.create_data_loader accepts `packed_format: packed`."""
    import importlib.util

    import torch

    from paddlerec_b200 import runner

    spec = importlib.util.spec_from_file_location("pack_dataset", os.path.join(ROOT, "tools", "pack_dataset.py"))
    tool = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(tool)
    paths, _ = _write_files(tmp_path)
    cache = tmp_path / "cache"
    assert tool.main(["--out", str(cache)] + paths) == 700 + 1 + 333
    packed = sorted(str(p) for p in cache.iterdir())
    assert [os.path.basename(p) for p in packed] == ["part-0.txt.b2r", "part-1.txt.b2r", "part-2.txt.b2r"]
    a = list(dataio.PackedBatchReader(paths, batch_size=64, prefetch=0))
    b = list(dataio.PackedBatchReader(packed, batch_size=64, fmt="packed", prefetch=0))
    assert len(a) == len(b) == (700 + 1 + 333) // 64
    assert all(torch.equal(x, y) for p, q in zip(a, b) for x, y in zip(p, q))
    # raw TSV (parser.cpp semantics: the two malformed lines of the sample are skipped)
    tsv = tmp_path / "day_0"
    tsv.write_bytes(_read("criteo_tsv_sample.tsv"))
    assert tool.main(["--out", str(cache), "--format", "criteo_tsv", str(tsv)]) == 62
    lab, ids, dense = dataio.read_packed(str(cache / "day_0.b2r"))
    rl, rid, _ = _parser_cpp_output(_read("criteo_tsv_parser_cpp.txt"))
    assert np.array_equal(ids, rid) and np.array_equal(lab[:, 0], rl)
    with pytest.raises(dataio.B200RecIOError, match="fewer than 40 columns"):   # benchmark_reader raises
        tool.main(["--out", str(cache), "--format", "criteo_tsv", "--hash", "xxh32", str(tsv)])
    # through the runner: a data dir of .b2r files
    cfg = {"runner.train_data_dir": str(cache), "runner.train_batch_size": 100, "config_abs_dir": "/",
           "runner.reader_type": "PackedReader", "runner.packed_format": "packed"}
    (cache / "day_0.b2r").unlink()
    batches = list(runner.create_data_loader(cfg))
    assert len(batches) == 10 and batches[0][1].shape == (100, 26)


def test_lod_and_multislot_outputs_are_trimmed_to_the_parsed_samples():
    """ADVICE r1: whitespace-only lines are counted for the capacity but dropped by the parser; the
    returned label / offsets / dense must be cut to the n samples actually produced (the tail was
    uninitialised memory and the offsets fed out-of-bounds reads of the pooled gather)."""
    sch = dataio.SlotSchema(sparse_slots=("a", "b"), label_slot="y", dense_slot="d", dense_dim=1)
    text = "y:1 a:5 a:6 b:7 d:0.5\n   \n\ny:0 a:8 b:9 b:10 d:0.25\n \t \n"
    label, keys, offsets, dense = dataio.parse_slot_text_lod(text, sch)
    assert label.shape == (2, 1) and dense.shape == (2, 1)
    assert offsets.tolist() == [0, 2, 3, 4, 6] and keys.tolist() == [5, 6, 7, 8, 9, 10]
    got = dataio.parse_multislot("1 3 1 4\n   \n2 5 6 1 7\n\n", [False, False])
    assert got["n"] == 2 and got["key_offsets"].tolist() == [0, 1, 2, 4, 5]
