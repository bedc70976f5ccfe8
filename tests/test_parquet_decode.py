"""Device Parquet decoder, checked in the CPU container: the page / run-header walker is host code inside libqk.so
(`qk_parquet_walk_chunk`) and runs here for real; the per-value decode function the CUDA kernel calls
(quokka_b200/csrc/parquet_core.h: decode_value) is compiled with g++ (tests/native/pq_core_check.cpp) and driven
over the walker's run tables.  The expected values are pyarrow's own reading of the same files.  The same scenarios
run against the CUDA kernel in tests/test_gpu_zz_parquet.py."""
import ctypes as C

import numpy as np
import pyarrow as pa
import pyarrow.parquet as pq
import pytest
import torch

import cpu_shim
import parquet_cases as P
from quokka_b200 import _lib as L
from quokka_b200 import parquet as PQ

CPU = torch.device("cpu")


@pytest.fixture(autouse=True)
def shim(monkeypatch):
    cpu_shim.install(monkeypatch)


@pytest.mark.parametrize("version,dict_on,page", P.LINEITEM_SHAPES)
def test_lineitem_shapes(tmp_path, version, dict_on, page): P.case_lineitem_shapes(tmp_path, CPU, version, dict_on, page)
def test_required_columns_and_dictionary_fallback(tmp_path): P.case_required_and_fallback(tmp_path, CPU)
def test_strings_share_codes_across_row_groups(tmp_path): P.case_strings_share_codes(tmp_path, CPU)
def test_bit_widths(tmp_path): P.case_bit_widths(tmp_path, CPU)
@pytest.mark.parametrize("seed", [1, 2, 3])
def test_random_files(tmp_path, seed): P.case_random_files(tmp_path, CPU, seed)
def test_spark_layout(tmp_path): P.case_spark_layout(tmp_path, CPU)
def test_decimals(tmp_path):
    P.case_decimals(tmp_path, CPU)
    P.case_decimals(tmp_path, CPU, "snappy")


# ---- SNAPPY pages: inflated, walked and decoded by the device pipeline (here: its per-page functions under g++)
@pytest.mark.parametrize("version,dict_on,page", P.LINEITEM_SHAPES)
def test_snappy_lineitem_shapes(tmp_path, version, dict_on, page): P.case_lineitem_shapes(tmp_path, CPU, version, dict_on, page, compression="snappy")
def test_snappy_fallback_strings_widths(tmp_path):
    P.case_required_and_fallback(tmp_path, CPU, "snappy")
    P.case_strings_share_codes(tmp_path, CPU, "snappy")
    P.case_bit_widths(tmp_path, CPU, "snappy")
def test_snappy_streams(tmp_path): P.case_snappy_streams(tmp_path, CPU)


# ---- ZSTD pages (Polars' default codec): one sequential frame decoder per page, a few workspace slots shared round-robin
@pytest.mark.parametrize("version,dict_on,page", P.LINEITEM_SHAPES)
def test_zstd_lineitem_shapes(tmp_path, version, dict_on, page): P.case_lineitem_shapes(tmp_path, CPU, version, dict_on, page, compression="zstd")
def test_zstd_fallback_strings_widths(tmp_path):
    P.case_required_and_fallback(tmp_path, CPU, "zstd")
    P.case_strings_share_codes(tmp_path, CPU, "zstd")
    P.case_bit_widths(tmp_path, CPU, "zstd")
def test_zstd_streams(tmp_path): P.case_snappy_streams(tmp_path, CPU, "zstd")


# ---- GZIP pages (Athena / Glue / older Hive writers): a DEFLATE decoder per page, same workspace slots
@pytest.mark.parametrize("version,dict_on,page", P.LINEITEM_SHAPES)
def test_gzip_lineitem_shapes(tmp_path, version, dict_on, page): P.case_lineitem_shapes(tmp_path, CPU, version, dict_on, page, compression="gzip")
def test_gzip_fallback_strings_widths_streams(tmp_path):
    P.case_required_and_fallback(tmp_path, CPU, "gzip")
    P.case_strings_share_codes(tmp_path, CPU, "gzip")
    P.case_bit_widths(tmp_path, CPU, "gzip")
    P.case_snappy_streams(tmp_path, CPU, "gzip")


def test_deflate_decoder_against_zlib():
    """csrc/deflate_core.h on gzip members from Arrow's codec and on zlib's own output: dynamic, fixed and stored blocks,
    zlib and gzip framing, concatenated members; truncated / mis-sized / bit-flipped streams are errors, not crashes."""
    import zlib
    rng = np.random.default_rng(3)
    n = 150_000
    vocab = [bytes(rng.integers(97, 123, rng.integers(2, 12), dtype=np.uint8)) for _ in range(3000)]
    samples = [b"", b"a", b"hello hello hello hello hello", bytes(1000), bytes(1_000_000), rng.bytes(70_000), b"ab" * 70_000,
               (rng.bytes(300) + b"xyz" * 50) * 500, bytes(rng.integers(0, 4, 200_000, dtype=np.uint8)),
               (rng.integers(90000, 10500000, n) / 100.0).tobytes(), np.cumsum(rng.integers(1, 8, n)).astype(np.int64).tobytes(),
               b" ".join(vocab[i] for i in rng.zipf(1.3, 120_000) % 3000),
               bytes(np.minimum(rng.geometric(0.3, 300_000), 255).astype(np.uint8))]
    lib = cpu_shim._pq_check_lib()

    def run(z, size):
        src = np.frombuffer(z, dtype=np.uint8).copy()
        out = np.zeros(size + 8, dtype=np.uint8)
        return lib.pq_check_gzip(src.ctypes.data, len(src), out.ctypes.data, size), out[:size].tobytes()
    for i, s in enumerate(samples):
        streams = [pa.Codec("gzip", compression_level=lv).compress(s, asbytes=True) for lv in (1, 6, 9)]
        streams += [zlib.compress(s, 6), zlib.compress(s, 0)]
        co = zlib.compressobj(6, zlib.DEFLATED, 31, 9, zlib.Z_FIXED)
        streams.append(co.compress(s) + co.flush())
        for z in streams:
            rc, out = run(z, len(s))
            assert rc == 0 and out == s, i
            if len(s) > 10:
                assert run(z, len(s) - 1)[0] != 0 and run(z[:-9], len(s))[0] != 0
                for _ in range(3):
                    bad = bytearray(z)
                    bad[int(rng.integers(10, len(z)))] ^= 1 << int(rng.integers(8))
                    run(bytes(bad), len(s))
    a, b = samples[2], samples[9]
    rc, out = run(pa.Codec("gzip").compress(a, asbytes=True) + pa.Codec("gzip").compress(b, asbytes=True), len(a) + len(b))
    assert rc == 0 and out == a + b


def test_zstd_decoder_against_arrow_codec():
    """csrc/zstd_core.h on raw frames from Arrow's zstd encoder: every block type (raw / RLE / compressed), literal
    modes (raw, RLE, Huffman with direct and FSE-coded weights, 1 and 4 streams, treeless), sequence table modes
    (predefined, RLE, FSE, repeat), repeat offsets, multi-block frames; and corrupt frames are errors."""
    rng = np.random.default_rng(11)
    n = 150_000
    vocab = [bytes(rng.integers(97, 123, rng.integers(2, 12), dtype=np.uint8)) for _ in range(3000)]
    samples = [b"", b"a", b"hello hello hello hello hello", bytes(1000), bytes(1_000_000), rng.bytes(70_000), rng.bytes(300_000),
               b"ab" * 70_000, (rng.bytes(300) + b"xyz" * 50) * 500, bytes(rng.integers(0, 4, 200_000, dtype=np.uint8)),
               (rng.integers(90000, 10500000, n) / 100.0).tobytes(), np.cumsum(rng.integers(1, 8, n)).astype(np.int64).tobytes(),
               rng.integers(8000, 10500, n).astype(np.int32).tobytes(), rng.normal(size=n).astype(np.float32).tobytes(),
               b" ".join(vocab[i] for i in rng.zipf(1.3, 120_000) % 3000),
               bytes(np.minimum(rng.geometric(0.3, 300_000), 255).astype(np.uint8)),
               bytes((np.cumsum(rng.integers(-5, 6, 400_000)) % 251).astype(np.uint8))]
    lib = cpu_shim._pq_check_lib()
    for i, s in enumerate(samples):
        for level in (-3, 1, 3, 9, 19):
            z = np.frombuffer(pa.Codec("zstd", compression_level=level).compress(s, asbytes=True), dtype=np.uint8).copy()
            out = np.zeros(len(s) + 8, dtype=np.uint8)
            assert lib.pq_check_zstd(z.ctypes.data, len(z), out.ctypes.data, len(s)) == 0, (i, level)
            assert out[:len(s)].tobytes() == s, (i, level)
            if len(s) > 10:
                assert lib.pq_check_zstd(z.ctypes.data, len(z), out.ctypes.data, len(s) - 1) != 0           # wrong size
                assert lib.pq_check_zstd(z.ctypes.data, len(z) - 3, out.ctypes.data, len(s)) != 0           # truncated
                if len(z) > 40:
                    for _ in range(4):                                                                    # byte flips: no crash
                        bad = z.copy()
                        bad[int(rng.integers(6, len(z)))] ^= 1 << int(rng.integers(8))
                        lib.pq_check_zstd(bad.ctypes.data, len(bad), out.ctypes.data, len(s))


def test_snappy_decoder_against_arrow_codec():
    """The element parser + lane-wise apply on raw streams from Arrow's Snappy encoder, and corrupt streams flagged."""
    rng = np.random.default_rng(9)
    codec = pa.Codec("snappy")
    samples = [b"", b"a", b"ab" * 5000, bytes(100_000), rng.bytes(70_000), (rng.bytes(300) + b"xyz" * 50) * 200,
               bytes(rng.integers(0, 4, 200_000, dtype=np.uint8)), b"0123456789" * 7 + rng.bytes(61) + b"0123456789" * 7]
    streams = [codec.compress(s, asbytes=True) for s in samples]
    raw = np.frombuffer(b"".join(streams) + bytes(16), dtype=np.uint8).copy()
    pages = np.zeros(len(samples) + 2, PQ.PAGE_DTYPE)
    src = dst = 0
    for i, (s, z) in enumerate(zip(samples, streams)):
        pages[i] = (src, dst, 0, len(z), len(s), 0, 0, 0, L.PQ_PAGE_DATA_V1, 0, 1, 0, 0, 0)
        src += len(z)
        dst += (len(s) + 7) // 8 * 8
    # two corrupt pages: a truncated stream, and a wrong uncompressed length
    pages[len(samples)] = (0, dst, 0, len(streams[2]) - 3, len(samples[2]), 0, 0, 0, L.PQ_PAGE_DATA_V1, 0, 1, 0, 0, 0)
    pages[len(samples) + 1] = (0, dst + 16384, 0, len(streams[0]), 5, 0, 0, 0, L.PQ_PAGE_DATA_V1, 0, 1, 0, 0, 0)
    scratch = torch.zeros(dst + 32768, dtype=torch.uint8)
    pt = torch.from_numpy(pages.view(np.uint8).reshape(-1))
    cpu_shim.parquet_inflate(torch.from_numpy(raw), pt, len(pages), scratch)
    out = scratch.numpy()
    for i, s in enumerate(samples):
        assert pages[i]["status"] == 0
        assert out[pages[i]["dst_offset"]:pages[i]["dst_offset"] + len(s)].tobytes() == s, i
    assert pages[len(samples)]["status"] == 8 and pages[len(samples) + 1]["status"] == 8


def test_run_table_shape(tmp_path):
    """One run per PLAIN page; dictionary pages produce RLE / PACKED runs with contiguous dense positions."""
    n = 10_000
    t = pa.table({"x": pa.array(np.arange(n, dtype=np.float64)), "y": pa.array((np.arange(n) // 1000).astype(np.int64))})
    path = str(tmp_path / "r.parquet")
    pq.write_table(t, path, compression=None, use_dictionary=["y"], data_page_size=8000, row_group_size=n)
    paths, plans, rows = PQ.plan_batch([(path, 0)])
    assert rows == n
    raw = open(path, "rb").read()
    for name, kinds in (("x", {L.PQ_RUN_PLAIN}), ("y", {L.PQ_RUN_RLE, L.PQ_RUN_PACKED})):
        p = plans[name]
        _, start, size, nvals, comp, off = p.chunks[0]
        buf = np.frombuffer(raw[start:start + size] + bytes(16), dtype=np.uint8).copy()
        runs, n_runs, dense, info = PQ.walk_chunk(buf.ctypes.data, 0, size, nvals, p.physical, p.max_def, 0, 0,
                                                  np.zeros(4, PQ.RUN_DTYPE), 0, 0)                     # grows from 4
        assert dense == n and info.n_values == n and set(runs["kind"][:n_runs]) <= kinds
        assert np.all(np.diff(runs["dense_start"][:n_runs]) > 0) and runs["dense_start"][0] == 0
        if name == "x":
            assert n_runs == info.n_data_pages > 5 and info.dict_offset == -1
        else:
            assert info.dict_num_values == 10 and n_runs <= 40          # 1000-long runs: a handful of RLE runs


def test_outside_scope_is_loud(tmp_path):
    t = pa.table({"a": pa.array([1, None, 3], pa.int64()), "s": pa.array(["x", "y", "z"]), "b": pa.array([1.0, 2.0, 3.0])})
    nulls = str(tmp_path / "n.parquet")
    pq.write_table(t, nulls, compression=None)
    with pytest.raises(L.QkError, match="nulls"):
        P.read(nulls, CPU, ["a"])
    with pytest.raises(L.QkError, match="nulls"):
        pq.write_table(t, nulls, compression=None, data_page_version="2.0")
        P.read(nulls, CPU, ["a"])
    P.same(P.read(nulls, CPU, ["b", "s"]), pq.read_table(nulls, columns=["b", "s"]))
    br = str(tmp_path / "s.parquet")
    pq.write_table(t.select(["b"]), br, compression="brotli")
    with pytest.raises(L.QkError, match="BROTLI"):
        P.read(br, CPU)
    pq.write_table(t, nulls, compression="snappy")                        # nulls behind a codec are found on the device
    with pytest.raises(L.QkError, match="nulls"):
        P.read(nulls, CPU, ["a"])
    pq.write_table(pa.table({"k": pa.array(np.arange(100))}), nulls, compression="snappy", use_dictionary=False,
                   column_encoding={"k": "DELTA_BINARY_PACKED"})
    with pytest.raises(L.QkError, match="outside PLAIN"):               # an encoding met only after the page is inflated
        P.read(nulls, CPU)
    plain_str = str(tmp_path / "p.parquet")
    pq.write_table(t.select(["s", "b"]), plain_str, compression=None, use_dictionary=False)
    P.same(P.read(plain_str, CPU), pq.read_table(plain_str))           # strings without a dictionary: coded on the host
    for codec in ("snappy", "zstd", "gzip"):                           # ... also when that only shows after inflation
        pq.write_table(t.select(["s", "b"]), plain_str, compression=codec, use_dictionary=False)
        P.same(P.read(plain_str, CPU), pq.read_table(plain_str))
    pq.write_table(t.select(["s", "b"]), plain_str, compression=None, use_dictionary=False)
    with pytest.raises(L.QkError, match="PLAIN BYTE_ARRAY"):           # ... the walker itself still says what it met
        md = pq.ParquetFile(plain_str).metadata.row_group(0).column(0)
        raw_ = np.frombuffer(open(plain_str, "rb").read() + bytes(16), dtype=np.uint8).copy()
        PQ.walk_chunk(raw_.ctypes.data, md.data_page_offset, md.total_compressed_size, md.num_values, L.PQ_BYTE_ARRAY, 1, 0, 0,
                      np.zeros(8, PQ.RUN_DTYPE), 0, 0)
    delta = str(tmp_path / "d.parquet")
    pq.write_table(pa.table({"k": pa.array(np.arange(100))}), delta, compression=None, use_dictionary=False,
                   column_encoding={"k": "DELTA_BINARY_PACKED"})
    with pytest.raises(L.QkError, match="DELTA_BINARY_PACKED"):
        P.read(delta, CPU)
    nested = str(tmp_path / "l.parquet")
    pq.write_table(pa.table({"l": pa.array([[1, 2], [3]])}), nested, compression=None)
    with pytest.raises(L.QkError, match="nested"):
        P.read(nested, CPU)
    # a truncated chunk is an error, not a crash
    raw = np.frombuffer(open(plain_str, "rb").read(), dtype=np.uint8).copy()
    info = L.qk_pq_chunk_info()
    nr, d = C.c_int64(0), C.c_int64(0)
    runs = np.zeros(8, PQ.RUN_DTYPE)
    rc = L.lib().qk_parquet_walk_chunk(raw.ctypes.data, 4, 10, 3, L.PQ_DOUBLE, 0, 0, 0, runs.ctypes.data, 8, C.byref(nr), C.byref(d), C.byref(info))
    assert rc == L.ERR_INVALID and nr.value == 0 and d.value == 0


def test_row_group_pruning(tmp_path):
    n = 10_000
    t = pa.table({"k": pa.array(np.arange(n)), "d": pa.array(np.arange(n) // 100, pa.int32()).cast(pa.date32())})
    path = str(tmp_path / "s.parquet")
    pq.write_table(t, path, compression=None, row_group_size=1000)
    md = pq.ParquetFile(path).metadata
    keep = [g for g in range(10) if PQ.row_group_may_match(md, g, [("k", ">=", 2500), ("k", "<", 4000)])]
    assert keep == [2, 3]
    assert [g for g in range(10) if PQ.row_group_may_match(md, g, [("k", "=", 9999)])] == [9]
    assert [g for g in range(10) if PQ.row_group_may_match(md, g, [("k", "in", [5, 5005])])] == [0, 5]
    assert all(PQ.row_group_may_match(md, g, [("missing", "=", 1)]) for g in range(10))
    import datetime
    day = datetime.date(1970, 1, 1) + datetime.timedelta(days=55)
    assert [g for g in range(10) if PQ.row_group_may_match(md, g, [("d", "=", day)])] == [5]


def test_corrupt_chunks_fail_cleanly(tmp_path):
    """Byte flips and truncations in real column chunks: the walker and the decode / inflate functions must either raise
    QkError or produce SOME values -- never read outside their buffers (the g++ harness would crash the test run)."""
    t = P.lineitem(6000).select(["l_orderkey", "l_returnflag", "l_extendedprice", "l_flag", "l_small"])
    rng = np.random.default_rng(123)
    outcomes = {"ok": 0, "error": 0}
    for codec in (None, "snappy", "zstd", "gzip"):
        path = str(tmp_path / f"fz_{codec}.parquet")
        pq.write_table(t, path, compression=codec, data_page_size=2048, row_group_size=3000, data_page_version="2.0" if codec else "1.0")
        good = open(path, "rb").read()
        md = pq.ParquetFile(path).metadata
        spans = []
        for g in range(md.num_row_groups):
            for c in range(md.num_columns):
                cc = md.row_group(g).column(c)
                start = min(cc.data_page_offset, cc.dictionary_page_offset or cc.data_page_offset)
                spans.append((start, cc.total_compressed_size))
        for trial in range(120):
            bad = bytearray(good)
            start, size = spans[rng.integers(len(spans))]
            for _ in range(int(rng.integers(1, 4))):
                pos = start + int(rng.integers(size))
                bad[pos] = int(rng.integers(256)) if trial % 3 else (bad[pos] ^ (1 << int(rng.integers(8))))
            fz = str(tmp_path / "fz.parquet")
            open(fz, "wb").write(bytes(bad))                       # footer intact: the plan is the good file's
            try:
                P.read(fz, CPU)
                outcomes["ok"] += 1
            except L.QkError:
                outcomes["error"] += 1
            except (MemoryError, RuntimeError, OverflowError, ValueError):
                outcomes["error"] += 1                             # absurd sizes in a corrupted header
    assert outcomes["error"] > 40 and outcomes["ok"] + outcomes["error"] == 480, outcomes


def test_files_from_an_old_writer(golden_dir):
    """Files another writer produced (parquet-cpp 1.3, 2017: Snappy, PLAIN_DICTIONARY ids), from pyarrow's test data."""
    import glob
    import os
    files = sorted(glob.glob(os.path.join(golden_dir, "parquet_v0.7.1", "v0.7.1*.parquet")))
    assert len(files) == 4
    for f in files:
        names = pq.ParquetFile(f).schema_arrow.names
        P.same(P.read(f, CPU, names), pq.read_table(f, columns=names).replace_schema_metadata(None))
