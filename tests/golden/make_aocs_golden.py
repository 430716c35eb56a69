#!/usr/bin/env python3
"""Write tests/golden/aocs_columns.npz (and aocs_zlib_columns.npz / aocs_zstd_columns.npz, bulk-compressed columns;
aocs_text_columns.npz, character(n) / varchar columns kept as strings): AOCS column files produced by the REFERENCE's own block writer
(oracle/_ref/libaocs_ref.so = the reference's datumstreamblock.c + cdbappendonlystorageformat.c + pg_crc32c_sb8.c,
driven by oracle/ref_aocs.c; run `make -C oracle` first) together with the values that went in.

Runs only where /root/reference exists; the .npz is what travels and what the parity tests read."""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from oracle import aocs_format as A  # noqa: E402


def main():
    if A.ref_lib() is None:
        sys.exit("oracle/_ref/libaocs_ref.so missing: run `make -C oracle` where /root/reference exists")
    rng = np.random.default_rng(20260922)
    out = {}
    cases = []

    def add(name, typname, values, nulls, checksum, blocksize, dscale=0, rle=False, zlevel=0, zstd=0):
        raw, nblocks = A.ref_write_column(typname, values, nulls, checksum, blocksize, dscale, rle=rle, zlevel=zlevel,
                                          compressor=A.zstd_compressor(zstd) if zstd else None)
        zlevel = zlevel or zstd
        out[name + "__raw"] = np.frombuffer(raw, dtype=np.uint8)
        if typname in A.STRING_TYPES:
            w = max([len(v) for v in values] + [1])
            out[name + "__values"] = np.array([v if isinstance(v, bytes) else v.encode() for v in values], dtype="S%d" % w)
            out[name + "__lens"] = np.array([len(v) for v in values], dtype=np.int32)      # 'S' arrays drop trailing NULs only
        elif typname == "bpchar":
            out[name + "__values"] = np.array([ord(v[0]) if v else 32 for v in values], dtype=np.int64)
        elif typname == "float8":
            out[name + "__values"] = np.asarray(values, dtype=np.float64)
        else:
            out[name + "__values"] = np.asarray(values, dtype=np.int64)
        out[name + "__nulls"] = np.zeros(len(values), dtype=np.uint8) if nulls is None else np.asarray(nulls, dtype=np.uint8)
        if zlevel:
            cases.append("%s|%s|%d|%d|%d|%d|%d" % (name, typname, 1 if checksum else 0, blocksize, dscale, nblocks, zlevel))
        else:
            cases.append("%s|%s|%d|%d|%d|%d" % (name, typname, 1 if checksum else 0, blocksize, dscale, nblocks))

    n = 20011
    nul = (rng.random(n) < 0.07).astype(np.uint8)
    add("int4_plain", "int4", rng.integers(-2**31, 2**31 - 1, n), None, True, 32768)
    add("int4_nulls_8k", "int4", rng.integers(-10**6, 10**6, n), nul, False, 8192)
    add("int8_nulls", "int8", rng.integers(-2**62, 2**62, n), nul, True, 32768)
    add("date_plain", "date", rng.integers(-3000, 9000, n), None, True, 32768)
    add("float8_nulls", "float8", rng.normal(0, 1e6, n), nul, True, 32768)
    add("bool_plain", "bool", rng.integers(0, 2, n), None, True, 8192)
    # numeric(15,2): TPC-H-like prices, quantities, discounts; zero, negatives, 15-digit extremes
    price = rng.integers(90000, 10500000, n)
    price[:8] = [0, 1, -1, 99, 100, 10**15 - 1, -(10**15 - 1), 10000]
    add("numeric_price", "numeric", price, None, True, 32768, dscale=2)
    add("numeric_disc_nulls_8k", "numeric", rng.integers(0, 11, n), nul, False, 8192, dscale=2)
    add("numeric_scale6", "numeric", rng.integers(-10**12, 10**12, 5003), None, True, 32768, dscale=6)
    add("bpchar1_flags", "bpchar", [("A", "N", "R", "F", "O")[i] for i in rng.integers(0, 5, n)], nul, True, 32768)
    # compresstype = rle_type (Dense blocks with repeat counts); runs, NULLs inside and between runs, one run longer
    # than a SmallContent header can count (-> NonBulkDenseContent header), values that do not repeat at all
    runs = np.repeat(rng.integers(0, 5, 300), rng.integers(1, 120, 300))
    nr = len(runs)
    nulr = (rng.random(nr) < 0.04).astype(np.uint8)
    add("rle_bpchar1_runs_nulls", "bpchar", [("A", "N", "R", "F", "O")[i] for i in runs], nulr, True, 32768, rle=True)
    add("rle_numeric_long_run", "numeric", np.concatenate([np.full(40000, 12345), rng.integers(100, 10**7, 3000), np.full(20000, -5),
                                                              np.repeat(rng.integers(0, 11, 500), rng.integers(1, 9, 500))]),
        None, True, 32768, dscale=2, rle=True)
    add("rle_float8_runs_8k", "float8", np.repeat(rng.normal(0, 1e3, 700), rng.integers(1, 40, 700)), None, False, 8192, rle=True)
    add("rle_bool_norepeat", "bool", rng.integers(0, 2, 3000) * 0 + np.arange(3000) % 2, None, True, 8192, rle=True)
    mixed = np.where(rng.random(9000) < 0.5, np.repeat(rng.normal(0, 10, 900), 10), rng.normal(0, 1e6, 9000))
    add("rle_float8_many_blocks_nulls", "float8", mixed, (rng.random(9000) < 0.05).astype(np.uint8), True, 8192, rle=True)
    # rle_type on integer / date columns also turns delta range encoding on (init_datumstream_info): sorted dates with
    # repeats and NULLs, growing keys with large jumps in both directions, random int4 (deltas too big to encode)
    nd = 30000
    dates = np.cumsum(rng.integers(0, 3, nd)) - 500
    add("delta_date_sorted_nulls", "date", dates, (rng.random(nd) < 0.03).astype(np.uint8), True, 32768, rle=2)
    keys = np.cumsum(rng.integers(-40, 1000, nd)).astype(np.int64) * 7 + 2**40
    keys[100], keys[101], keys[5000] = -2**62, 2**62, 0
    add("delta_int8_keys_8k", "int8", keys, None, False, 8192, rle=2)
    add("delta_int4_random", "int4", rng.integers(-2**31, 2**31 - 1, 5000), None, True, 8192, rle=2)
    add("delta_int4_wrap", "int4", np.array([2**31 - 1, -2**31, -2**31 + 5, 2**31 - 3, 0, 1, 1, 1, 2, 2**29, 2**29 + 2**29 - 1]), None, True, 8192, rle=2)
    add("int4_tiny", "int4", [7], None, True, 32768)
    add("int4_allnull", "int4", [0] * 100, [1] * 100, True, 32768)
    # two files, the first four columns and the rest, to keep each under 1 MB (tests/test_aocs_format.py reads both)
    for fname, part in (("aocs_columns.npz", cases[:4]), ("aocs_columns_2.npz", cases[4:])):
        names = {c.split("|")[0] for c in part}
        path = os.path.join(ROOT, "tests", "golden", fname)
        np.savez_compressed(path, cases=np.array(part), **{k: v for k, v in out.items() if k.rsplit("__", 1)[0] in names})
        print("wrote", path, os.path.getsize(path), "bytes,", len(part), "columns")
    for c in cases:
        print("  ", c)

    # ---- bulk compression: compresstype=zlib compresslevel=L, and rle_type compresslevel 2 / 3 / 4 (= RLE + zlib 1 / 5 / 9)
    out = {}
    cases = []
    rng = np.random.default_rng(20260923)
    n = 20011
    nul = (rng.random(n) < 0.07).astype(np.uint8)
    add("zlib1_int4_sorted", "int4", np.cumsum(rng.integers(0, 4, n)) - 10**6, None, True, 32768, zlevel=1)
    add("zlib5_numeric_price", "numeric", rng.integers(90000, 10500000, n), None, True, 32768, dscale=2, zlevel=5)
    add("zlib9_bpchar1_flags_nulls", "bpchar", [("A", "N", "R", "F", "O")[i] for i in rng.integers(0, 5, n)], nul, True, 32768, zlevel=9)
    # incompressible: compress2 makes it longer, the writer stores those blocks as they are (compressed length 0)
    add("zlib1_int8_random_stored", "int8", rng.integers(-2**62, 2**62, 6000), None, True, 32768, zlevel=1)
    add("zlib6_float8_nulls_8k_nocrc", "float8", np.round(rng.normal(0, 50, n)), nul, False, 8192, zlevel=6)
    # large blocks: 16383 rows of int8 per block, matches reaching far back, several deflate blocks per stream
    big = np.tile(rng.integers(-2**40, 2**40, 2500), 14)[:33000] + np.repeat(np.arange(33), 1000)
    add("zlib6_int8_bigblocks", "int8", big, None, True, 2097152, zlevel=6)
    add("zlib3_date_mixed", "date", np.where(rng.random(n) < 0.3, rng.integers(-3000, 9000, n), 7305), nul, True, 32768, zlevel=3)
    add("zlib1_int4_tiny_stored", "int4", [7], None, True, 32768, zlevel=1)
    add("zlib9_bool_allnull", "bool", [0] * 5000, [1] * 5000, True, 8192, zlevel=9)
    # rle_type compresslevel 2: one 40000-row run -> a Dense block of more than 16383 rows -> BulkDenseContent header
    add("rle2_numeric_long_run", "numeric", np.concatenate([np.full(40000, 12345), rng.integers(100, 10**7, 3000), np.full(20000, -5),
                                                               np.repeat(rng.integers(0, 11, 500), rng.integers(1, 9, 500))]),
        None, True, 32768, dscale=2, rle=True, zlevel=1)
    add("rle3_date_delta_nulls", "date", np.cumsum(rng.integers(0, 3, 30000)) - 500, (rng.random(30000) < 0.03).astype(np.uint8), True, 32768,
        rle=2, zlevel=5)
    add("rle4_float8_runs_8k_nocrc", "float8", np.repeat(rng.normal(0, 1e3, 900), rng.integers(1, 60, 900)), None, False, 8192, rle=True, zlevel=9)
    out["cases"] = np.array(cases)
    path = os.path.join(ROOT, "tests", "golden", "aocs_zlib_columns.npz")
    np.savez_compressed(path, **out)
    print("wrote", path, os.path.getsize(path), "bytes,", len(cases), "columns")
    for c in cases:
        print("  ", c)
        name = c.split("|")[0]
        blocks = A.walk_blocks_ex(bytes(out[name + "__raw"]), int(c.split("|")[2]))
        print("      kinds", sorted(set(b["kind"] for b in blocks)), "compressed", sum(1 for b in blocks if b["clen"]), "of", len(blocks),
              "file", len(out[name + "__raw"]), "bytes for", sum(b["dlen"] for b in blocks), "of content")

    # ---- compresstype=zstd compresslevel=L: the blocks go through a real libzstd (pyarrow's) the way zstd_compress does
    out = {}
    cases = []
    rng = np.random.default_rng(20260924)
    n = 20011
    nul = (rng.random(n) < 0.07).astype(np.uint8)
    add("zstd1_int4_sorted", "int4", np.cumsum(rng.integers(0, 4, n)) - 10**6, None, True, 32768, zstd=1)
    add("zstd3_numeric_price", "numeric", rng.integers(90000, 10500000, n), None, True, 32768, dscale=2, zstd=3)
    add("zstd9_bpchar1_flags_nulls", "bpchar", [("A", "N", "R", "F", "O")[i] for i in rng.integers(0, 5, n)], nul, True, 32768, zstd=9)
    add("zstd1_int8_random_stored", "int8", rng.integers(-2**62, 2**62, 6000), None, True, 32768, zstd=1)
    add("zstd5_float8_nulls_8k_nocrc", "float8", np.round(rng.normal(0, 50, n)), nul, False, 8192, zstd=5)
    big = np.tile(rng.integers(-2**40, 2**40, 2500), 14)[:33000] + np.repeat(np.arange(33), 1000)
    add("zstd3_int8_bigblocks", "int8", big, None, True, 2097152, zstd=3)                      # 131 KB content: two zstd blocks per frame
    add("zstd19_date_mixed", "date", np.where(rng.random(n) < 0.3, rng.integers(-3000, 9000, n), 7305), nul, True, 32768, zstd=19)
    add("zstd1_int4_tiny_stored", "int4", [7], None, True, 32768, zstd=1)
    add("zstd3_bool_allnull", "bool", [0] * 5000, [1] * 5000, True, 8192, zstd=3)               # RLE-ish content
    add("zstd3_int4_constant", "int4", [42] * 16000, None, True, 2097152, zstd=3)
    add("zstd7_numeric_few_values", "numeric", rng.choice([0, 1, 5, 10, 100, 12345678], n), nul, True, 32768, dscale=2, zstd=7)
    out["cases"] = np.array(cases)
    path = os.path.join(ROOT, "tests", "golden", "aocs_zstd_columns.npz")
    np.savez_compressed(path, **out)
    print("wrote", path, os.path.getsize(path), "bytes,", len(cases), "columns")
    for c in cases:
        print("  ", c)
        name = c.split("|")[0]
        blocks = A.walk_blocks_ex(bytes(out[name + "__raw"]), int(c.split("|")[2]))
        print("      kinds", sorted(set(b["kind"] for b in blocks)), "compressed", sum(1 for b in blocks if b["clen"]), "of", len(blocks),
              "file", len(out[name + "__raw"]), "bytes for", sum(b["dlen"] for b in blocks), "of content")

    # ---- character(n) / varchar columns whose values are kept (dictionary columns on the device)
    out = {}
    cases = []
    rng = np.random.default_rng(20260926)
    n = 20011
    nul = (rng.random(n) < 0.05).astype(np.uint8)
    modes = ["REG AIR", "AIR", "RAIL", "SHIP", "TRUCK", "MAIL", "FOB"]
    shipmode = [modes[i].ljust(10) for i in rng.integers(0, 7, n)]                           # character(10): blank padded
    add("shipmode_bpchar10_nulls", "bpchars", shipmode, nul, True, 32768)
    add("shipmode_rle", "bpchars", [modes[i].ljust(10) for i in np.repeat(rng.integers(0, 7, 700), rng.integers(1, 60, 700))], None, True,
        32768, rle=True)
    segs = ["AUTOMOBILE", "BUILDING", "FURNITURE", "MACHINERY", "HOUSEHOLD"]
    add("mktsegment_zlib5", "bpchars", [segs[i].ljust(10) for i in rng.integers(0, 5, n)], None, True, 32768, zlevel=5)
    nations = ["ALGERIA", "ARGENTINA", "BRAZIL", "CANADA", "EGYPT", "ETHIOPIA", "FRANCE", "GERMANY", "INDIA", "INDONESIA", "IRAN", "IRAQ",
               "JAPAN", "JORDAN", "KENYA", "MOROCCO", "MOZAMBIQUE", "PERU", "CHINA", "ROMANIA", "SAUDI ARABIA", "VIETNAM", "RUSSIA",
               "UNITED KINGDOM", "UNITED STATES"]
    add("n_name_bpchar25", "bpchars", [s.ljust(25) for s in nations], None, True, 32768)
    # varchar: lengths 0 .. 300 (1-byte and 4-byte varlena headers), trailing blanks that DO count, the empty string
    words = ["", " ", "a", "a ", "ab", "carefully final deposits", "x" * 126, "y" * 127, "z" * 200, "w" * 300, "quick  ", "quick"]
    add("varchar_mixed_nulls_8k", "varchar", [words[i] for i in rng.integers(0, len(words), 6000)], (rng.random(6000) < 0.1).astype(np.uint8),
        False, 8192)
    add("varchar_many_distinct_zstd", "varchar", ["Customer#%09d" % i for i in rng.integers(0, 3000, n)], None, True, 32768, zstd=3)
    out["cases"] = np.array(cases)
    path = os.path.join(ROOT, "tests", "golden", "aocs_text_columns.npz")
    np.savez_compressed(path, **out)
    print("wrote", path, os.path.getsize(path), "bytes,", len(cases), "columns")
    for c in cases:
        print("  ", c)


if __name__ == "__main__":
    main()
