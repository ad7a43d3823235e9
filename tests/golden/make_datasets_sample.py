#!/usr/bin/env python
"""Write tests/golden/datasets/: a sample of the reference's five bundled training files, for the reader test.

    python tests/golden/make_datasets_sample.py REFERENCE_CHECKOUT

Each ``<kind>_training_data.csv`` keeps its header, delimiter and last line (ping's last line is truncated, so the
reader must drop it), its first data line, up to 20 lines holding a value that pandas parses one ulp away from
``float(text)``, and 20 more lines drawn with a fixed seed, all verbatim and in file order.  ``sample.json`` records,
per file, how many rows the whole file contributes to tests/golden/bundled.npz's ``X`` (the files are concatenated
in the notebooks' order) and which data lines the sample kept, so the test can find each kept row there.
"""
import json
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))

from traffic_classifier_sdn_b200 import dataio  # noqa: E402

KINDS = ("ping", "voice", "dns", "telnet", "game")


def main():
    ref = sys.argv[1]
    X = np.load(os.path.join(HERE, "bundled.npz"))["X"]
    out = os.path.join(HERE, "datasets")
    os.makedirs(out, exist_ok=True)
    keep = [i for i, c in enumerate(dataio.COLUMNS[:16]) if c not in dataio.DROPPED]
    rng = np.random.default_rng(7653)
    meta, offset = [], 0
    for kind in KINDS:
        name = f"{kind}_training_data.csv"
        with open(os.path.join(ref, "datasets", name), "rb") as fh:
            lines = fh.read().split(b"\n")
        header, body = lines[0], lines[1:]
        if body and body[-1] == b"":          # the file ends with a newline
            body = body[:-1]
            end = b"\n"
        else:
            end = b""
        delim = "," if b"," in header else "\t"
        rows = len(dataio.read_training_file(os.path.join(ref, "datasets", name))[0])
        off_by_ulp = []
        for i, ln in enumerate(body[:rows]):
            fields = ln.decode().split(delim)
            if any(float(fields[c]) != X[offset + i, j] for j, c in enumerate(keep)):
                off_by_ulp.append(i)
        pick = {0, len(body) - 1}
        if off_by_ulp:
            pick.update(rng.choice(off_by_ulp, min(20, len(off_by_ulp)), replace=False).tolist())
        rest = sorted(set(range(len(body))) - pick)
        pick.update(rng.choice(rest, 20, replace=False).tolist())
        pick = sorted(int(i) for i in pick)
        with open(os.path.join(out, name), "wb") as fh:
            fh.write(b"\n".join([header] + [body[i] for i in pick]) + end)
        meta.append({"file": name, "rows": rows, "lines": pick})
        offset += rows
    assert offset == len(X), (offset, len(X))
    with open(os.path.join(out, "sample.json"), "w") as fh:
        fh.write("[\n" + ",\n".join(json.dumps(m) for m in meta) + "\n]\n")
    print("wrote", out)


if __name__ == "__main__":
    main()
