"""ClickBench `hits`-shaped batches for the 43-query sweep (BASELINE.json configs[4], SURVEY.md §8d row 5).

Rows are drawn with replacement from the 24 586-row sample of the real table that ships with the reference
(tests/golden/hits_sample.parquet, made by synth/make_sample.py), in runs: a batch keeps the sample's locality by taking
consecutive sample rows from a random start, so per-batch dictionary sizes and bit widths look like the real column's
(URL ~0.23 distinct values per row, EventTime a narrow window, flag columns one or two values). Two things the sample
lacks are added: the token `google` is spliced into URL with probability 4e-5, as configs[1] does (paper Table 1: Q20
selects < 0.01 %; the sample's titles already carry `Google`), and a batch's EventDate is moved to one of the 31 days of
July 2013 so the date-range conjuncts of q36-q42 select something other than everything.
Input data only: no liquid-cache logic here.
"""
from __future__ import annotations

import os

import numpy as np
import pyarrow as pa
import pyarrow.parquet as pq

_HERE = os.path.dirname(os.path.abspath(__file__))
ROWS_PER_BATCH = 8192
SEED = 50
JULY_1_2013 = 15887  # days since 1970-01-01; the sample's only EventDate is 15901 (2013-07-15)


class HitsSample:
    def __init__(self):
        self.table = pq.read_table(os.path.join(os.path.dirname(_HERE), "tests", "golden", "hits_sample.parquet"))
        self.n = self.table.num_rows
        self.cols = {c: self.table[c].combine_chunks() for c in self.table.column_names}

    def most_frequent(self, column: str):
        import pyarrow.compute as pc

        vc = pc.value_counts(self.cols[column])
        best = max(vc.to_pylist(), key=lambda d: d["counts"])
        return best["values"]

    def batches(self, columns, first_batch: int, n_batches: int):
        """{column: [Array of 8192 rows] * n_batches} for batches first_batch .. first_batch + n_batches - 1."""
        out = {c: [] for c in columns}
        run = 512  # consecutive sample rows per run
        idx_all = np.empty(n_batches * ROWS_PER_BATCH, dtype=np.int64)
        days = np.empty(n_batches, dtype=np.uint16)
        for b in range(n_batches):
            rng = np.random.default_rng([SEED, first_batch + b])
            starts = rng.integers(0, self.n, size=ROWS_PER_BATCH // run)
            idx_all[b * ROWS_PER_BATCH:(b + 1) * ROWS_PER_BATCH] = ((starts[:, None] + np.arange(run)[None, :]) % self.n).ravel()
            days[b] = JULY_1_2013 + rng.integers(0, 31)
        for c in columns:
            big = self.cols[c].take(pa.array(idx_all))
            if c == "URL":
                big = self._splice(big, first_batch)
            if c == "EventDate":
                big = pa.array(np.repeat(days, ROWS_PER_BATCH), pa.uint16())
            out[c] = [big.slice(b * ROWS_PER_BATCH, ROWS_PER_BATCH) for b in range(n_batches)]
        return out

    @staticmethod
    def _splice(big: pa.Array, first_batch: int) -> pa.Array:
        import pyarrow.compute as pc

        n_batches = len(big) // ROWS_PER_BATCH
        hits = []
        for b in range(n_batches):  # per batch, so a batch does not depend on how the caller groups its requests
            rng = np.random.default_rng([SEED + 1, first_batch + b])
            hits.extend((b * ROWS_PER_BATCH + np.flatnonzero(rng.random(ROWS_PER_BATCH) < 4e-5)).tolist())
        if not hits:
            return big
        mask = np.zeros(len(big), dtype=bool)
        mask[hits] = True
        repl = []
        for i in hits:
            s = big[int(i)].as_py()
            repl.append(s[: len(s) // 2] + "google" + s[len(s) // 2:])
        return pc.replace_with_mask(big, pa.array(mask), pa.array(repl, big.type))
