"""Jay ingest (datatable_b200/jay.py): files written by the reference itself (tests/golden/make_golden_jay.py,
Frame.to_jay = src/core/jay/save_jay.cc) must come back as the reference's NA-sentinel buffers.
CPU tests parse the meta section and read into numpy; the GPU test reads straight into HBM and runs a query."""
import os

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
J1 = os.path.join(HERE, "golden", "jay_v1.jay")
JK = os.path.join(HERE, "golden", "jay_keyed.jay")
EXP = np.load(os.path.join(HERE, "golden", "jay_expected.npz"))
FIXED = ["b", "i8", "i16", "i32", "i64", "f32", "f64", "d32"]


def same(a, b):
    if a.dtype.kind == "f":
        return a.dtype == b.dtype and np.array_equal(a.view(np.uint32 if a.dtype == np.float32 else np.uint64)[~np.isnan(a)],
                                                     b.view(np.uint32 if b.dtype == np.float32 else np.uint64)[~np.isnan(b)]) \
            and np.array_equal(np.isnan(a), np.isnan(b))
    return a.dtype == b.dtype and np.array_equal(a, b)


def test_meta_of_reference_written_file():
    from datatable_b200 import jay
    m = jay.read_meta(open(J1, "rb").read())
    assert (m["nrows"], m["ncols"], m["nkeys"]) == (1000, 9, 0)
    assert [c["name"] for c in m["columns"]] == FIXED + ["s"]
    assert [c["jay_stype"] for c in m["columns"]] == [0, 1, 2, 3, 4, 5, 6, 9, 7]
    for c in m["columns"][:-1]:
        assert c["offset"] % 8 == 0 and c["nrows"] == 1000
        assert c["nullcount"] == int(np.sum(np.isnan(EXP[c["name"]]) if EXP[c["name"]].dtype.kind == "f" else
                                            EXP[c["name"]] == np.iinfo(EXP[c["name"]].dtype).min))
    assert jay.read_meta(open(JK, "rb").read())["nkeys"] == 1


def test_buffers_are_the_reference_na_sentinel_arrays():
    from datatable_b200 import jay, _lib
    DT = jay.open_jay(J1, columns=FIXED, device=False)
    assert DT.names == tuple(FIXED) and DT.nrows == 1000
    for nm in FIXED:
        assert same(DT.to_numpy(nm), EXP[nm]), nm
    assert [DT.stypes[i] for i in range(8)] == [_lib.BOOL, _lib.INT8, _lib.INT16, _lib.INT32, _lib.INT64, _lib.FLOAT32,
                                                _lib.FLOAT64, _lib.DATE32]
    K = jay.open_jay(JK, device=False)
    assert same(K.to_numpy("k"), EXP["keyed.k"]) and same(K.to_numpy("v"), EXP["keyed.v"]) and K.key == ("k",)


def test_string_columns_and_broken_files_are_refused(tmp_path):
    from datatable_b200 import jay, _lib
    with pytest.raises(_lib.DtbNotImplError):
        jay.open_jay(J1, device=False)                                   # column `s` is str32
    raw = open(J1, "rb").read()
    for bad in (raw[:-8] + b"\0\0\0\0XJAY", b"JAX1" + raw[4:], raw[:len(raw) // 2 // 8 * 8], raw[:16],
                raw[:-16] + (2**40).to_bytes(8, "little") + raw[-8:], raw[:-16] + (12).to_bytes(8, "little") + raw[-8:]):
        p = tmp_path / "bad.jay"
        p.write_bytes(bad)
        with pytest.raises(_lib.DtbValueError):
            jay.open_jay(str(p), device=False)


@pytest.mark.gpu
def test_jay_straight_to_hbm_and_grouped():
    import torch
    import datatable_b200 as dt
    from datatable_b200 import jay
    from oracle import oracle as orc
    from helpers import OPS, INT16, FLOAT64
    f, by = dt.f, dt.by
    DT = jay.open_jay(J1, columns=["i16", "f64", "b"])
    assert all(torch.is_tensor(DT._cols[n]) and DT._cols[n].is_cuda for n in DT.names)
    R = DT[:, {"s": dt.sum(f.f64), "n": dt.count(f.f64)}, by(f.b)]
    order, offsets, _ = orc.group([EXP["b"]], [0], 1, stypes=[1])
    want_s = orc.reduce(OPS["sum"], EXP["f64"], order, offsets, stype=FLOAT64)
    want_n = orc.reduce(OPS["count"], EXP["f64"], order, offsets, stype=FLOAT64)
    assert np.array_equal(R.to_numpy("b"), EXP["b"][order[offsets[:-1]]])
    assert np.allclose(R.to_numpy("s"), want_s, rtol=1e-12) and np.array_equal(R.to_numpy("n"), want_n)
    S = DT[:, f.i16, dt.sort(f.i16)]
    so, _, _ = orc.group([EXP["i16"]], [4], 1, stypes=[INT16])
    assert np.array_equal(S.to_numpy("i16"), EXP["i16"][so])


def test_writer_round_trip_and_key(tmp_path):
    from datatable_b200 import jay
    F = jay.open_jay(J1, columns=FIXED, device=False)
    p = str(tmp_path / "out.jay")
    F.to_jay(p)
    G = jay.open_jay(p, device=False)
    assert G.names == F.names and list(G.stypes) == list(F.stypes)
    for nm in FIXED:
        assert same(G.to_numpy(nm), EXP[nm]), nm
    K = jay.open_jay(JK, device=False)
    pk = str(tmp_path / "keyed.jay")
    K.to_jay(pk)
    assert jay.read_meta(open(pk, "rb").read())["nkeys"] == 1 and jay.open_jay(pk, device=False).key == ("k",)


def test_reference_opens_what_the_writer_wrote(tmp_path):
    """The reference's own reader (flatbuffers::Verifier + open_jay.cc) accepts the file and sees the same frame:
    checked by tests/golden/make_golden_v4.py on jay_written.jay, which the writer must reproduce byte for byte."""
    from datatable_b200 import jay
    F = jay.open_jay(J1, columns=FIXED, device=False)
    p = str(tmp_path / "out.jay")
    F.to_jay(p)
    assert open(p, "rb").read() == open(os.path.join(HERE, "golden", "jay_written.jay"), "rb").read()


def test_time64_and_empty_frames():
    """Files written by the reference: a 0-row frame, and a time64 column (int64 nanoseconds, NA = INT64_MIN)."""
    from datatable_b200 import jay, _lib
    E = jay.open_jay(os.path.join(HERE, "golden", "jay_empty.jay"), device=False)
    assert E.names == ("a", "b") and E.nrows == 0 and list(E.stypes) == [_lib.INT32, _lib.FLOAT64]
    T = jay.open_jay(os.path.join(HERE, "golden", "jay_time.jay"), device=False)
    assert list(T.stypes) == [_lib.TIME64, _lib.INT32]
    assert np.array_equal(T.to_numpy("t"), np.array([1577880000000000000, -2**63, -1000000000], dtype=np.int64))
    assert np.array_equal(T.to_numpy("x"), np.array([1, 2, 3], dtype=np.int32))
