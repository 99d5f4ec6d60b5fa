"""TrialList, the O(trials) trial container: text formats, conversion from Key / Ndx, and the id join (CPU only)."""
import logging
import os

import numpy
import pytest

import sidekit_b200 as sk

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "text_io")


def _pairs(key):
    """{(model, segment): is_target} of every trial of a Key."""
    out = {}
    for m in range(key.modelset.shape[0]):
        for s in range(key.segset.shape[0]):
            if key.tar[m, s] or key.non[m, s]:
                out[(str(key.modelset[m]), str(key.segset[s]))] = bool(key.tar[m, s])
    return out


def test_read_txt_matches_key_read_txt():
    path = os.path.join(GOLD, "key.txt")
    tl = sk.TrialList.read_txt(path)
    key = sk.Key.read_txt(path)
    assert len(tl) == int(key.tar.sum() + key.non.sum())
    assert dict(zip(zip(tl.enrolset.tolist(), tl.testset.tolist()), tl.labels.tolist())) == _pairs(key)
    with open(path) as f:            # file order is kept
        first = f.readline().split()
    assert [tl.enrolset[0], tl.testset[0], "target" if tl.labels[0] else "nontarget"] == first


def test_round_trip_with_key_write_txt(tmp_path):
    key = sk.Key.read_txt(os.path.join(GOLD, "key.txt"))
    key.write_txt(str(tmp_path / "k.txt"))
    tl = sk.TrialList.read_txt(str(tmp_path / "k.txt"))
    assert dict(zip(zip(tl.enrolset.tolist(), tl.testset.tolist()), tl.labels.tolist())) == _pairs(key)
    tl.write_txt(str(tmp_path / "t.txt"))
    back = sk.TrialList.read_txt(str(tmp_path / "t.txt"))
    assert numpy.array_equal(back.enrolset, tl.enrolset) and numpy.array_equal(back.testset, tl.testset)
    assert numpy.array_equal(back.labels, tl.labels)
    assert _pairs(sk.Key.read_txt(str(tmp_path / "t.txt"))) == _pairs(key)


def test_read_txt_rejects_unknown_label(tmp_path):
    (tmp_path / "bad.txt").write_text("m1 s1 target\nm1 s2 maybe\n")
    with pytest.raises(ValueError, match="maybe"):
        sk.TrialList.read_txt(str(tmp_path / "bad.txt"))


def test_read_voxceleb(tmp_path):
    (tmp_path / "veri.txt").write_text("1 id10270/x6uYqmx31kE/00001.wav id10270/8jEAjG6SegY/00008.wav\n"
                                       "0 id10270/x6uYqmx31kE/00001.wav id10300/ize_eiCFEg0/00003.wav\n"
                                       "\n"
                                       "1 id10309/0cYFdtyWVds/00005.wav id10309/Zx-zA-D_DvI/00001.wav\n")
    tl = sk.TrialList.read_voxceleb(str(tmp_path / "veri.txt"))
    assert len(tl) == 3
    assert tl.enrolset.tolist() == ["id10270/x6uYqmx31kE/00001.wav", "id10270/x6uYqmx31kE/00001.wav", "id10309/0cYFdtyWVds/00005.wav"]
    assert tl.testset.tolist() == ["id10270/8jEAjG6SegY/00008.wav", "id10300/ize_eiCFEg0/00003.wav", "id10309/Zx-zA-D_DvI/00001.wav"]
    assert tl.labels.tolist() == [True, False, True]
    (tmp_path / "bad.txt").write_text("2 a b\n")
    with pytest.raises(ValueError):
        sk.TrialList.read_voxceleb(str(tmp_path / "bad.txt"))


def test_from_ndx_and_from_key_follow_row_major_mask_order():
    rng = numpy.random.default_rng(3)
    ndx = sk.Ndx()
    ndx.modelset = numpy.array(["m%02d" % i for i in rng.permutation(7)])
    ndx.segset = numpy.array(["s%02d" % i for i in rng.permutation(11)])
    ndx.trialmask = rng.random((7, 11)) < 0.4
    tl = sk.TrialList.from_ndx(ndx)
    r, c = numpy.nonzero(ndx.trialmask)
    assert numpy.array_equal(tl.enrolset, ndx.modelset[r]) and numpy.array_equal(tl.testset, ndx.segset[c])
    assert tl.labels is None

    tar = ndx.trialmask & (rng.random((7, 11)) < 0.3)
    key = sk.Key.create(ndx.modelset, ndx.segset, tar, ndx.trialmask & ~tar)
    tk = sk.TrialList.from_key(key)
    assert numpy.array_equal(tk.enrolset, ndx.modelset[r]) and numpy.array_equal(tk.testset, ndx.segset[c])
    assert numpy.array_equal(tk.labels, tar[r, c])


def test_index_permuted_duplicate_and_missing_ids(caplog):
    tl = sk.TrialList(["a", "b", "zz", "c", "a", "b"], ["x", "y", "x", "nope", "z", "x"], [1, 0, 1, 0, 0, 1])
    enrol_ids = numpy.array(["c", "b", "a", "b"])             # permuted; "b" twice: the first occurrence (row 1) wins
    test_ids = numpy.array(["z", "x", "y", "x"])
    with caplog.at_level(logging.INFO):
        rows, cols, keep = tl.index(enrol_ids, test_ids)
    assert keep.tolist() == [True, True, False, False, True, True]
    assert rows.dtype == numpy.int32 and cols.dtype == numpy.int32
    assert rows.tolist() == [2, 1, 2, 1] and cols.tolist() == [1, 2, 0, 1]
    assert "trials reduced from 6 to 4" in caplog.text
    kept = tl.subset(keep)
    assert kept.enrolset.tolist() == ["a", "b", "a", "b"] and kept.labels.tolist() == [True, False, False, True]


def test_index_keeps_everything_silently(caplog):
    tl = sk.TrialList(["a", "b"], ["x", "x"])
    with caplog.at_level(logging.INFO):
        rows, cols, keep = tl.index(numpy.array(["b", "a"]), numpy.array(["x"]))
    assert keep.all() and rows.tolist() == [1, 0] and cols.tolist() == [0, 0]
    assert "reduced" not in caplog.text


def test_misaligned_arrays_and_unlabelled_tar_non_are_errors():
    with pytest.raises(ValueError):
        sk.TrialList(["a", "b"], ["x"])
    with pytest.raises(ValueError):
        sk.TrialList(["a"], ["x"], [True, False])
    ts = sk.TrialScores(sk.TrialList(["a"], ["x"]), None)
    with pytest.raises(ValueError, match="labels"):
        ts.get_tar_non()
