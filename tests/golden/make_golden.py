"""tests/golden/make_golden.py -- regenerates the committed fixtures in tests/golden/.

Needs a checkout of the reference R package (no R itself):

    python tests/golden/make_golden.py <reference checkout>

Outputs
  yeast_missing.npz      data/yeast_missing.rda of the reference converted to NumPy
                         (6887 features x 96 samples, column names), read with the small
                         XDR reader below.  Stored as per-column dense ranks (uint16; 0 where
                         the value is 0, i.e. missing): every pair statistic depends only on
                         the order and ties within each column and on which entries are
                         missing, so results are those of the original values, in under 1 MB.
  yeast_oracle.npz       oracle (oracle/icikt_oracle.cpp) results for all 4560 column
                         pairs of yeast_missing, global and local perspective:
                         tau/pvalue/tau_max/completeness/status + int64 counts.
  reference_snapshots.json
                         values transcribed from the reference's own test snapshot
                         /root/reference/tests/testthat/_snaps/kendall-tau.md (file:line
                         recorded per entry), used to pin the oracle.
"""
from __future__ import annotations

import bz2
import gzip
import json
import lzma
import os
import struct
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)


class _XDR:
    """Minimal reader of R's XDR serialization (enough for a numeric matrix with dimnames)."""

    def __init__(self, buf):
        self.b, self.o, self.refs = buf, 0, []

    def i32(self):
        v = struct.unpack_from(">i", self.b, self.o)[0]
        self.o += 4
        return v

    def f64(self, n):
        a = np.frombuffer(self.b, dtype=">f8", count=n, offset=self.o).astype(np.float64)
        self.o += 8 * n
        return a

    def length(self):
        n = self.i32()
        if n == -1:
            hi, lo = self.i32(), self.i32()
            n = (hi << 32) + lo
        return n

    def item(self):
        flags = self.i32()
        t = flags & 0xFF
        has_attr, has_tag = bool(flags & 0x200), bool(flags & 0x400)
        if t == 254:  # NILVALUE_SXP
            return None
        if t == 255:  # REFSXP
            return self.refs[(flags >> 8) - 1] if (flags >> 8) else self.refs[self.i32() - 1]
        if t == 1:  # SYMSXP
            s = self.item()
            self.refs.append(s)
            return s
        if t == 9:  # CHARSXP
            n = self.i32()
            if n == -1:
                return None
            s = self.b[self.o:self.o + n].decode("utf-8", "replace")
            self.o += n
            return s
        if t == 2:  # LISTSXP (pairlist)
            out = []
            while True:
                attr = self.item() if has_attr else None
                tag = self.item() if has_tag else None
                out.append((tag, self.item()))
                flags = self.i32()
                t2 = flags & 0xFF
                if t2 == 254:
                    break
                assert t2 == 2, t2
                has_attr, has_tag = bool(flags & 0x200), bool(flags & 0x400)
                del attr
            return out
        if t == 14:  # REALSXP
            v = self.f64(self.length())
            attr = dict(self.item()) if has_attr else {}
            return ("real", v, attr)
        if t == 13 or t == 10:  # INTSXP / LGLSXP
            n = self.length()
            v = np.frombuffer(self.b, dtype=">i4", count=n, offset=self.o).astype(np.int32)
            self.o += 4 * n
            attr = dict(self.item()) if has_attr else {}
            return ("int", v, attr)
        if t == 16:  # STRSXP
            v = [self.item() for _ in range(self.length())]
            attr = dict(self.item()) if has_attr else {}
            return ("str", v, attr)
        if t == 19:  # VECSXP
            v = [self.item() for _ in range(self.length())]
            attr = dict(self.item()) if has_attr else {}
            return ("list", v, attr)
        if t == 238:  # ALTREP: (info pairlist, state, attr) -- expand compact seqs only
            info, state, attr = self.item(), self.item(), self.item()
            return ("altrep", info, state, attr)
        raise NotImplementedError(f"SEXP type {t} at {self.o}")


def read_rda(path):
    raw = open(path, "rb").read()
    for opener in (bz2.decompress, gzip.decompress, lzma.decompress):
        try:
            raw = opener(raw)
            break
        except Exception:
            continue
    assert raw[:5] in (b"RDX2\n", b"RDX3\n"), raw[:8]
    x = _XDR(raw[5:])
    assert x.b[:2] == b"X\n"
    x.o = 2
    version = x.i32()
    x.i32()
    x.i32()
    if version == 3:
        n = x.i32()
        x.o += n
    return x.item()


def load_yeast(ref):
    top = read_rda(os.path.join(ref, "data", "yeast_missing.rda"))
    (tag, (kind, vals, attr)), = top
    assert tag == "yeast_missing" and kind == "real", (tag, kind)
    dim = attr["dim"][1]
    dimnames = attr["dimnames"][1]
    data = vals.reshape(int(dim[0]), int(dim[1]), order="F")
    colnames = np.array(dimnames[1][1])
    return data, colnames


def column_ranks(data):
    """Dense ranks of the positive values of every column, from 1; zeros stay 0."""
    assert (data >= 0).all()
    out = np.zeros(data.shape, dtype=np.uint16)
    for j in range(data.shape[1]):
        pos = data[:, j] > 0
        _, inv = np.unique(data[pos, j], return_inverse=True)
        assert inv.size == 0 or inv.max() + 1 < 2 ** 16
        out[pos, j] = inv + 1
    return out


def main(ref):
    from oracle import oracle as O

    data, colnames = load_yeast(ref)
    print("yeast_missing", data.shape, "zeros:", int((data == 0).sum()))
    np.savez_compressed(os.path.join(HERE, "yeast_missing.npz"), data=column_ranks(data), colnames=colnames)

    excl = O.setup_missing_matrix(data)
    ex = data.copy()
    ex[excl] = np.nan
    pi, pj = O.setup_comparisons(data.shape[1], None, True)
    out = {}
    for persp in ("global", "local"):
        r = O.pair_loop(ex, pi, pj, perspective=persp, ncore=8, want_counts=True)
        for k, v in r.items():
            out[f"{persp}_{k}"] = v
    np.savez_compressed(os.path.join(HERE, "yeast_oracle.npz"), pi=pi, pj=pj, **out)

    snaps = {
        "_source": "/root/reference/tests/testthat/_snaps/kendall-tau.md",
        "large_kendall": {  # :1-7 ; test-kendall-tau.R:72-78 (set.seed(1234); rnorm(50000) x2; global)
            "lines": "1-7", "tau": -0.00123518, "pvalue": 0.67867094, "tau_max": 1.0, "completeness": 1.0},
        "completeness_rows_4_6": {  # :9-17 ; test-kendall-tau.R:138-151
            "lines": "9-17", "s1": [1, 1, 1], "s2": [5, 6, 7], "missingness": [1, 2, 2],
            "completeness": [0.98, 0.96, 0.96]},
        "kt_fast_na_pairs_complete": {  # :35-47
            "lines": "35-47", "tau01": 0.003092146, "p_diag": 1.076521e-48, "p01": 9.638307e-01},
        "kt_fast_na_matrix_complete": {  # :49-68
            "lines": "49-68",
            "tau": [[1.0, 0.0030921459, 0.0072150072, 0.10904968],
                    [0.003092146, 1.0, 0.0006184292, 0.04555762],
                    [0.007215007, 0.0006184292, 1.0, 0.01669759],
                    [0.109049680, 0.0455576170, 0.0166975881, 1.0]],
            "pvalue": [[1.076521e-48, 9.638307e-01, 9.157333e-01, 1.097676e-01],
                       [9.638307e-01, 1.076521e-48, 9.927638e-01, 5.040615e-01],
                       [9.157333e-01, 9.927638e-01, 1.076521e-48, 8.065540e-01],
                       [1.097676e-01, 5.040615e-01, 8.065540e-01, 1.076521e-48]]},
        "kt_fast_na_matrix_pairwise": {  # :70-90
            "lines": "70-90",
            "tau": [[1.0, 0.003092146, 0.007215007, 0.10904968],
                    [0.003092146, 1.0, 0.002424242, 0.04444444],
                    [0.007215007, 0.002424242, 1.0, 0.01010101],
                    [0.109049680, 0.044444444, 0.010101010, 1.0]],
            "pvalue": [[1.076521e-48, 9.638307e-01, 9.157333e-01, 1.097676e-01],
                       [9.638307e-01, 3.480281e-49, 9.714917e-01, 5.123482e-01],
                       [9.157333e-01, 9.714917e-01, 3.480281e-49, 8.816279e-01],
                       [1.097676e-01, 5.123482e-01, 8.816279e-01, 3.480281e-49]]},
    }
    with open(os.path.join(HERE, "reference_snapshots.json"), "w") as f:
        json.dump(snaps, f, indent=1)
    print("wrote fixtures to", HERE)


if __name__ == "__main__":
    main(sys.argv[1])
