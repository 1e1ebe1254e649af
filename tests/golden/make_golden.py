"""Rewrites tests/golden/uk_cities.json from the lat/lng columns it already stores (the reference's only data fixture).

    python tests/golden/make_golden.py
The lat/lng columns are the 37 rows of the reference's test/data/uk_cities_with_headers.csv, kept in
uk_cities.json itself, so the script needs nothing outside this repository; the
`reference_asserts` block restates the numbers the reference's own tests assert on this fixture
(src/dataframe.rs:803-808,835; src/lazyframe.rs:393-407).  `derived` values are produced by the CPU oracle
(sequential folds, glibc sin) and are NOT asserted by the reference -- they pin the oracle against
accidental change and give the GPU path a committed target.
"""
import json
import os
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))

import numpy as np  # noqa: E402

from oracle import pyoracle as orc  # noqa: E402

OUT = os.path.join(HERE, "uk_cities.json")


class _Chunk:
    def __init__(self, v):
        self.values, self.validity, self.offset, self.length, self.null_count, self.dtype = v, None, 0, len(v), 0, orc.F64


def main():
    with open(OUT) as f:
        stored = json.load(f)
    lat, lng = stored["lat"], stored["lng"]
    la, ln = np.array(lat), np.array(lng)
    _, added = orc.col_binary(orc.ADD, orc.F64, [_Chunk(la)], [_Chunk(ln)])
    _, sin_lat = orc.col_unary(orc.SIN, orc.F64, [_Chunk(la)])
    _, abs_lng = orc.col_unary(orc.ABS, orc.F64, [_Chunk(ln)])
    out = {
        "source": "reference test/data/uk_cities_with_headers.csv (37 rows, columns lat,lng)",
        "lat": lat,
        "lng": lng,
        "reference_asserts": {
            "n_rows": 37,
            "lat_plus_lng_row0": 54.31776,       # src/dataframe.rs:803-808 (tolerance 1e-4, one-sided)
            "abs_lng_row0": 3.335724,            # src/dataframe.rs:835
            "lat_row0": 57.653484, "lng_row0": -3.335724,  # src/lazyframe.rs:393-407
        },
        "derived": {
            "lat_plus_lng_hex": [float(x).hex() for x in added[0].values],
            "sin_lat_hex": [float(x).hex() for x in sin_lat[0].values],
            "abs_lng_hex": [float(x).hex() for x in abs_lng[0].values],
            "sum_lat_hex": float(orc.aggregate(orc.SUM, orc.F64, [_Chunk(la)])[1]).hex(),
            "sum_lat_plus_lng_hex": float(orc.aggregate(orc.SUM, orc.F64, [_Chunk(added[0].values)])[1]).hex(),
            "min_lat": float(la.min()), "max_lat": float(la.max()),
        },
    }
    with open(OUT, "w") as f:
        json.dump(out, f, indent=1)
    print("wrote uk_cities.json; sum(lat) =", float.fromhex(out["derived"]["sum_lat_hex"]))


if __name__ == "__main__":
    main()
