#!/usr/bin/env python
"""Builds tests/golden/hits_sample.parquet FROM THE REFERENCE CHECKOUT: the 25 columns of examples/nano_hits.parquet (24 586
real ClickBench rows shipped with the reference) that the 43 ClickBench queries touch (benchmark/clickbench/queries/q0-q42.sql).
bench.py's clickbench_sweep workload and its CPU test draw their rows from this sample (synth/hits.py). Needs the reference
checkout:
    python synth/make_sample.py <reference checkout>/examples/nano_hits.parquet
the output is committed with the other stored test data. Brotli, large pages, dictionaries only where values repeat and delta
coding of the random WatchID keep the file under 1 MB; the rows and their order are those of the input."""
import os
import sys

import pyarrow.parquet as pq

COLUMNS = ["AdvEngineID", "ResolutionWidth", "UserID", "SearchPhrase", "EventDate", "RegionID", "MobilePhoneModel", "MobilePhone",
           "SearchEngineID", "EventTime", "URL", "Title", "CounterID", "Referer", "IsRefresh", "ClientIP", "WatchID",
           "DontCountHits", "IsLink", "IsDownload", "TraficSourceID", "URLHash", "RefererHash", "WindowClientWidth",
           "WindowClientHeight"]
DICTIONARY = ["SearchPhrase", "MobilePhoneModel", "URL", "Title", "Referer", "IsRefresh", "DontCountHits"]
OUT = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden", "hits_sample.parquet")

if __name__ == "__main__":
    t = pq.read_table(sys.argv[1], columns=COLUMNS)
    pq.write_table(t, OUT, compression="brotli", compression_level=11, write_statistics=False, use_dictionary=DICTIONARY,
                   column_encoding={"WatchID": "DELTA_BINARY_PACKED"}, data_page_size=1 << 24, dictionary_pagesize_limit=1 << 24)
    print(t.num_rows, "rows,", os.path.getsize(OUT), "bytes")
