"""SURVEY 8f N3: the importers of the reference's own on-disk artefacts and the exports in the reference's schema, against
files written by the UNMODIFIED reference (tests/golden/make_golden_files.py): <ref>-FM.json (ExactMatch.py:22-41),
rmi_file.pkl (RMI_LUT.py:186-198).  Host-side only; the LUT file and the single-file index need a GPU (test_gpu_files.py)."""
import gzip
import json
import os
import pickle
import shutil
import sys
import time

import numpy as np
import pytest

from tests import golden_util as gu


@pytest.fixture()
def workdir(tmp_path, monkeypatch):
    """cwd with data/medium_data.fa, as the reference's cwd-relative paths expect."""
    g = gu.load_index("medium_data")
    os.makedirs(tmp_path / "data")
    with open(tmp_path / "data" / "medium_data.fa", "w") as f:
        f.write(">medium_data\n")
        f.write("\n".join(g["text"][i:i + 50] for i in range(0, len(g["text"]), 50)))
        f.write("\n")
    monkeypatch.chdir(tmp_path)
    return tmp_path, g


def _ref_fm_json():
    with gzip.open(os.path.join(gu.GOLDEN, "ref_medium_data-FM.json.gz"), "rt") as f:
        return f.read()


def test_load_fm_index_reads_the_reference_json_and_export_writes_the_same_schema(workdir):
    import genie_smem_b200 as gs
    tmp, g = workdir
    with open(tmp / "data" / "medium_data-FM.json", "w") as f:
        f.write(_ref_fm_json())
    m = gs.ExactMatch("medium_data.fa")
    m.load_fm_index()
    sa, bwt = m._host.export()
    assert np.array_equal(sa, g["suffix_array"]) and bwt.decode() == g["bwt"]
    ref = json.loads(_ref_fm_json())
    assert m.ref_size == ref["ref_size"] and m.fm_index["count_dic"] == ref["count_dic"]
    # export in the reference's schema == what the reference's own create_fm_index wrote, key for key
    out = m.export_reference_json(str(tmp / "export.json"))
    mine = json.load(open(out))
    assert set(mine) == set(ref) == {"bwt_array", "suffix_array", "occurance_matrix", "count_dic", "ref_size"}
    for k in ref:
        assert mine[k] == ref[k], k


def test_load_fm_index_prefers_the_newer_file_and_validates_the_size(workdir):
    import genie_smem_b200 as gs
    tmp, g = workdir
    m = gs.ExactMatch("medium_data.fa")
    with pytest.raises(FileNotFoundError):
        m.load_fm_index()
    m.create_fm_index()                                     # writes data/medium_data-FM.npz (host SA-IS at this size)
    assert os.path.exists(tmp / "data" / "medium_data-FM.npz")
    # a NEWER reference JSON of another text: it is the one read, and it is refused
    bad = json.loads(_ref_fm_json())
    bad["suffix_array"] = bad["suffix_array"][:-5]
    bad["ref_size"] -= 5
    time.sleep(0.05)
    with open(tmp / "data" / "medium_data-FM.json", "w") as f:
        json.dump(bad, f)
    os.utime(tmp / "data" / "medium_data-FM.json", (time.time() + 5, time.time() + 5))
    with pytest.raises(ValueError):
        gs.ExactMatch("medium_data.fa").load_fm_index()
    # the correct JSON, newer than the npz: read without complaint
    with open(tmp / "data" / "medium_data-FM.json", "w") as f:
        f.write(_ref_fm_json())
    os.utime(tmp / "data" / "medium_data-FM.json", (time.time() + 9, time.time() + 9))
    m2 = gs.ExactMatch("medium_data.fa")
    m2.load_fm_index()
    assert np.array_equal(m2._host.export()[0], g["suffix_array"])
    m3 = gs.ExactMatch("medium_data.fa")
    m3.create_fm_index(reference_json=True)                 # both files written by this package: the JSON is the reference's schema
    assert json.load(open(tmp / "data" / "medium_data-FM.json")) == json.loads(_ref_fm_json())


def test_rmi_lut_load_reads_the_reference_pickle_and_fit_reproduces_it(workdir):
    """RMI_LUT.load on a pickle written by the reference (sklearn LinearRegression models inside): parameters equal the ones
    make_golden.py extracted from the same training run; and RMI.fit (the per-bucket loop) retrains them from the same keys
    to rounding (sklearn solves the same least squares with LAPACK gelsd: the fit itself is not bit-pinned, SURVEY 8c)."""
    import genie_smem_b200 as gs
    tmp, g = workdir
    m = gs.ExactMatch.from_text(g["text"], suffix_array=g["suffix_array"], name="medium_data.fa")
    shutil.copy(os.path.join(gu.GOLDEN, "ref_rmi_medium_k6.pkl"), tmp / "rmi_file.pkl")
    r = gs.RMI_LUT.load("rmi_file.pkl", matcher=m)
    p = gu.load_rmi("medium_data_k6")
    assert r.prediction_size == p["K"] == 6 and list(r.structure) == p["experts"]
    assert list(r.rmi.level_sizes) == p["level_sizes"]
    assert np.array_equal(r.rmi.coef, p["coef"]) and np.array_equal(r.rmi.intercept, p["intercept"])
    # retrain with this package's trainer on the same keys
    r2 = gs.RMI_LUT(p["experts"], 6, "medium_data.fa", matcher=m)
    r2.train_RMI()
    keys = np.arange(4 ** 6, dtype=np.int64)
    a, b = r.rmi.predict(keys), r2.rmi.predict(keys)
    assert np.abs(a - b).max() < 1e-6
    assert np.array_equal(np.trunc(a), np.trunc(b))         # same start rows for the last-mile search on every 6-mer
    assert np.allclose(r2.rmi.coef, p["coef"], rtol=1e-9, atol=1e-12) and np.allclose(r2.rmi.intercept, p["intercept"], rtol=1e-9, atol=1e-9)


def test_rmi_big_k15_fit_matches_reference_trained_parameters():
    """surface.RMI.fit (loop) on big_data K=15 against the parameters the reference trained (tests/golden/rmi_big_data_k15.npz)."""
    import genie_smem_b200 as gs
    g = gu.load_index("big_data")
    p = gu.load_rmi("big_data_k15")
    m = gs.ExactMatch.from_text(g["text"], suffix_array=g["suffix_array"], name="big_data.fa")
    r = gs.RMI_LUT(p["experts"], 15, "big_data.fa", matcher=m)
    r.train_RMI()
    ref = gs.RMI.from_params(p["level_sizes"], p["coef"], p["intercept"])
    rng = np.random.default_rng(1)
    keys = rng.integers(0, 4 ** 15, 20000)
    d = np.abs(r.rmi.predict(keys) - ref.predict(keys))
    assert d.max() < 1e-4, d.max()                          # rows; models route identically up to rounding at bucket borders
    assert np.allclose(r.rmi.coef, p["coef"], rtol=1e-7, atol=1e-18)


def test_rmi_lut_save_in_reference_format_is_loadable_as_the_reference_class(workdir):
    """reference_format=True pickles an RMI.RMI whose .models hold sklearn LinearRegression objects (what RMI_LUT.load of the
    reference unpickles, RMI_LUT.py:192-198).  Routing k-mers through those models as the reference's RMI.predict does
    (RMI.py:52-69) gives, bit for bit, the predictions the reference made with the same model
    (tests/golden/rmi_lookups_medium_data_k6.json.gz)."""
    import genie_smem_b200 as gs
    tmp, g = workdir
    m = gs.ExactMatch.from_text(g["text"], suffix_array=g["suffix_array"], name="medium_data.fa")
    p = gu.load_rmi("medium_data_k6")
    r = gs.RMI_LUT(p["experts"], 6, "medium_data.fa", matcher=m)
    r.rmi = gs.RMI.from_params(p["level_sizes"], p["coef"], p["intercept"])
    had = sys.modules.pop("RMI", None)
    try:
        r.save("ref_style.pkl", reference_format=True)
        with open("ref_style.pkl", "rb") as f:
            structure, K, data_file, obj = pickle.load(f)   # plain pickle.load, as the reference does
        assert (list(structure), K, data_file) == (p["experts"], 6, "medium_data.fa")
        assert type(obj).__module__ == "RMI" and type(obj).__name__ == "RMI"
        assert [len(l) for l in obj.models] == p["level_sizes"]
        assert float(obj.models[1][3].coef_[0]) == float(p["coef"][4]) and float(obj.models[1][3].intercept_) == float(p["intercept"][4])
        rows = [row for row in gu.load_json("rmi_lookups_medium_data_k6.json.gz") if row[1] is not None]
        assert len(rows) > 2000
        scales = [len(l) for l in obj.models[1:]] + [1]
        for q, ref_pred, _, _ in rows:
            x = np.asarray([[gs.LUT.convert_seq_to_num(q)]], np.float64)
            k = 0
            for level, scale in zip(obj.models, scales):
                y = float(level[k].predict(x)[0])
                k = min(scale - 1, max(0, int(y)))
            assert y == ref_pred, q
        keys = np.asarray([gs.LUT.convert_seq_to_num(row[0]) for row in rows], np.int64)
        assert np.array_equal(r.rmi.predict(keys), np.asarray([row[1] for row in rows]))
        back = gs.RMI_LUT.load("ref_style.pkl", matcher=m)   # and this package reads it back
        assert np.array_equal(back.rmi.coef, p["coef"]) and np.array_equal(back.rmi.intercept, p["intercept"])
    finally:
        sys.modules.pop("RMI", None)
        if had is not None:
            sys.modules["RMI"] = had
