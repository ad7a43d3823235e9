"""Training-data reader/writer (SURVEY row N4): format round trip, mixed delimiters, truncated tail, and the notebooks'
recipe on a verbatim sample of the reference's bundled files against the golden rows."""
import json
import os

import numpy as np
import pytest

from traffic_classifier_sdn_b200 import dataio, flows

HERE = os.path.dirname(os.path.abspath(__file__))
SAMPLE = os.path.join(HERE, "golden", "datasets")


def _table():
    t = flows.FlowTable()
    lines = [b"data\t1\t1\t1\taa\tbb\t2\t0\t0\n", b"data\t2\t1\t1\taa\tbb\t2\t3\t300\n",
             b"data\t3\t1\t2\tbb\taa\t1\t1\t60\n", b"data\t7\t1\t1\taa\tbb\t2\t10\t1000\n"]
    for ln in lines:
        rec = flows.parse_monitor_line(ln)
        assert rec is not None
        t.ingest(rec)
    return t


def test_feature_names_are_the_predict_order():
    assert len(dataio.COLUMNS) == 17 and dataio.COLUMNS[-1] == "Traffic Type"
    assert len(dataio.FEATURE_NAMES) == 12
    assert dataio.FEATURE_NAMES[0] == "Delta Forward Packets" and dataio.FEATURE_NAMES[6] == "Delta Reverse Packets"


def test_write_then_read_round_trip(tmp_path):
    t = _table()
    p = tmp_path / "voice_training_data.csv"
    n = dataio.write_training_file(str(p), [t, t], "voice")
    assert n == 2 * len(t)
    X, y = dataio.read_training_file(str(p))
    assert X.shape == (n, 12) and set(y) == {"voice"}
    # the reader parses like the notebooks' pandas (not correctly rounded): within one ulp of what was written
    assert np.allclose(X[: len(t)], t.features(), rtol=4e-16, atol=0) and np.array_equal(X[len(t):], X[: len(t)])


def test_mixed_delimiters_and_truncated_tail(tmp_path):
    hdr = list(dataio.COLUMNS)
    a = tmp_path / "a.csv"
    b = tmp_path / "b.csv"
    row1 = [str(i) for i in range(16)] + ["ping"]
    row2 = [str(i + 0.5) for i in range(16)] + ["ping"]
    a.write_text("\t".join(hdr) + "\n" + "\t".join(row1) + "\n" + "\t".join(row2) + "\n" + "\t".join(row1[:10]))   # no newline, 10 fields
    b.write_text(",".join(hdr) + "\n" + ",".join(row2[:16] + ["game"]) + "\n" + ",".join(row1[:5] + [""] + row1[6:]) + "\n")
    X, y = dataio.load_training_set([str(a), str(b)])
    assert X.shape == (3, 12) and list(y) == ["ping", "ping", "game"]
    keep = [i for i, c in enumerate(hdr[:16]) if c not in dataio.DROPPED]
    assert np.array_equal(X[0], np.array([float(row1[i]) for i in keep]))
    assert np.array_equal(X[2], np.array([float(row2[i]) for i in keep]))


def test_parse_float_is_the_pandas_tokenizer_not_strtod():
    assert dataio.parse_float("98") == 98.0 and dataio.parse_float("-1.5e2") == -150.0 and dataio.parse_float("0.0") == 0.0
    assert dataio.parse_float("205.33333333333334") == 205.33333333333334 or \
        abs(dataio.parse_float("205.33333333333334") - 205.33333333333334) <= 2.9e-14
    for bad in ("", "abc", "1.2.3", "nan", "inf", "1e", "--1"):
        with pytest.raises(ValueError):
            dataio.parse_float(bad)


def test_errors(tmp_path):
    p = tmp_path / "x.csv"
    p.write_text("")
    with pytest.raises(ValueError):
        dataio.read_training_file(str(p))
    p.write_text("a,b,c\n1,2,3\n")
    with pytest.raises(ValueError):
        dataio.read_training_file(str(p))
    with pytest.raises(ValueError):
        dataio.load_training_set([])


def test_notebook_recipe_reproduces_the_golden_rows():
    """The reference's five bundled files, sampled verbatim (tests/golden/make_datasets_sample.py): read in the notebooks'
    order, every kept line must parse to the golden row pandas made of it, and ping's truncated last line must go."""
    z = np.load(os.path.join(HERE, "golden", "bundled.npz"))
    with open(os.path.join(SAMPLE, "sample.json")) as fh:
        meta = json.load(fh)
    X, y = dataio.load_training_set([os.path.join(SAMPLE, m["file"]) for m in meta])
    rows, offset = [], 0
    for m in meta:
        rows += [offset + i for i in m["lines"] if i < m["rows"]]
        offset += m["rows"]
    assert offset == len(z["X"]) == 7653 and len(rows) < sum(len(m["lines"]) for m in meta)
    assert X.shape == (len(rows), 12)
    assert np.array_equal(X, z["X"][rows]) and np.array_equal(y, z["y"][rows].astype(str))
