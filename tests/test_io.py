"""CPU suite: native count-table ingestion (pydeseq2_b200.io) against pandas, the reference's loader
(examples/plot_pandas_io_example.py:57-66)."""
import os

import numpy as np
import pandas as pd
import pytest

from conftest import GOLDEN
from pydeseq2_b200.io import read_counts_csv

# the reference's shipped synthetic dataset (datasets/synthetic/test_counts.csv), stored as is
REF = os.path.join(GOLDEN, "synthetic_test_counts.csv")


def _write(path, df, **kw):
    df.to_csv(path, **kw)


@pytest.mark.parametrize("quoting", [0, 1])  # csv.QUOTE_MINIMAL / QUOTE_ALL (labels quoted like the reference's files)
def test_genes_in_rows_matches_pandas_transpose(tmp_path, quoting):
    rng = np.random.default_rng(0)
    df = pd.DataFrame(rng.negative_binomial(2, 0.01, (257, 33)), index=[f"gene{i}" for i in range(257)],
                      columns=[f"sample{j}" for j in range(33)])
    p = tmp_path / "counts.csv"
    df.to_csv(p, quoting=quoting)
    want = pd.read_csv(p, index_col=0).T
    got = read_counts_csv(p)
    assert got.counts.dtype == np.int64 and got.counts.flags.c_contiguous and got.counts.shape == (33, 257)
    np.testing.assert_array_equal(got.counts, want.values)
    assert got.samples == list(want.index) and got.genes == list(want.columns)
    np.testing.assert_array_equal(got.to_frame().values, want.values)
    one = read_counts_csv(p, threads=1)
    np.testing.assert_array_equal(one.counts, got.counts)


def test_samples_in_rows_crlf_and_float_notation(tmp_path):
    p = tmp_path / "c.csv"
    p.write_bytes(b"id,g1,g2,g3\r\ns1,1,20.0,3e2\r\ns2,0,5,7\r\n\r\n")
    got = read_counts_csv(p, genes_in_rows=False)
    np.testing.assert_array_equal(got.counts, [[1, 20, 300], [0, 5, 7]])
    assert got.samples == ["s1", "s2"] and got.genes == ["g1", "g2", "g3"]


@pytest.mark.parametrize("cell", ["-3", "1.5", "abc", ""])
def test_invalid_counts_are_rejected(tmp_path, cell):
    p = tmp_path / "bad.csv"
    p.write_text(f"id,a,b\ng1,1,2\ng2,{cell},4\n")
    with pytest.raises(ValueError, match="row 1, column 0"):
        read_counts_csv(p)


def test_ragged_line_is_rejected(tmp_path):
    p = tmp_path / "ragged.csv"
    p.write_text("id,a,b\ng1,1,2\ng2,3\n")
    with pytest.raises(ValueError):
        read_counts_csv(p)


def test_reference_shipped_dataset():
    want = pd.read_csv(REF, index_col=0).T
    got = read_counts_csv(REF)
    np.testing.assert_array_equal(got.counts, want.values)
    assert got.samples == list(want.index) and got.genes == list(want.columns)
