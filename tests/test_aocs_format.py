"""AOCS column-file format (SURVEY.md 8 rows a3 / a4), CPU side (not gpu).

tests/golden/aocs_columns.npz holds column files written by the REFERENCE's own block writer (datumstreamblock.c +
cdbappendonlystorageformat.c, compiled where they lie and driven by oracle/ref_aocs.c; made by
tests/golden/make_aocs_golden.py).  The restated reader (oracle/aocs_format.py) must give back exactly the values that
went in.  Where the reference library is present (this container) the restated block walker is also checked against the
reference's header accessors and checksum verifiers, and the numeric encoder against utils/numeric.h's macros."""
import ctypes as C
import os

import numpy as np
import pytest

from oracle import aocs_format as A

HERE = os.path.dirname(os.path.abspath(__file__))


def golden():
    """the uncompressed columns, split over two files to keep each under 1 MB"""
    for f in ("aocs_columns.npz", "aocs_columns_2.npz"):
        d = np.load(os.path.join(HERE, "golden", f))
        for c in d["cases"]:
            name, typname, checksum, blocksize, dscale, nblocks = str(c).split("|")
            yield (name, typname, int(checksum), int(blocksize), int(dscale), int(nblocks), bytes(d[name + "__raw"]),
                   d[name + "__values"], d[name + "__nulls"])


CASES = list(golden())


def golden_zlib():
    """bulk-compressed columns (compresstype=zlib, rle_type compresslevel 2-4): the same tuple + the zlib level"""
    d = np.load(os.path.join(HERE, "golden", "aocs_zlib_columns.npz"))
    for c in d["cases"]:
        name, typname, checksum, blocksize, dscale, nblocks, zlevel = str(c).split("|")
        yield (name, typname, int(checksum), int(blocksize), int(dscale), int(nblocks), bytes(d[name + "__raw"]),
               d[name + "__values"], d[name + "__nulls"], int(zlevel))


ZCASES = list(golden_zlib())


def golden_zstd():
    """compresstype=zstd columns: the same tuple, the last field is the zstd level"""
    d = np.load(os.path.join(HERE, "golden", "aocs_zstd_columns.npz"))
    for c in d["cases"]:
        name, typname, checksum, blocksize, dscale, nblocks, zlevel = str(c).split("|")
        yield (name, typname, int(checksum), int(blocksize), int(dscale), int(nblocks), bytes(d[name + "__raw"]),
               d[name + "__values"], d[name + "__nulls"], int(zlevel))


ZSTDCASES = list(golden_zstd())


def golden_text():
    """character(n) / varchar columns kept as strings: (name, typname, checksum, blocksize, nblocks, raw, values, nulls,
    compression: "" / "zlib" / "zstd")"""
    d = np.load(os.path.join(HERE, "golden", "aocs_text_columns.npz"))
    for c in d["cases"]:
        f = str(c).split("|")
        name, typname, checksum, blocksize, nblocks = f[0], f[1], int(f[2]), int(f[3]), int(f[5])
        vals = [bytes(v).ljust(int(n), b"\0") for v, n in zip(d[name + "__values"], d[name + "__lens"])]
        yield (name, typname, checksum, blocksize, nblocks, bytes(d[name + "__raw"]), vals, d[name + "__nulls"],
               "zstd" if "zstd" in name else "zlib" if "zlib" in name else "")


TCASES = list(golden_text())


@pytest.mark.parametrize("case", CASES, ids=[c[0] for c in CASES])
def test_restated_reader_reads_reference_written_columns(case):
    name, typname, checksum, blocksize, dscale, nblocks, raw, values, nulls = case
    blocks = A.walk_blocks(raw, checksum)
    assert len(blocks) == nblocks
    assert sum(b[2] for b in blocks) == len(values)
    assert blocks[0][3] == 1 and all(blocks[i + 1][3] == blocks[i][3] + blocks[i][2] for i in range(len(blocks) - 1))
    got, gotnull = A.decode_column(raw, typname, checksum, dscale)
    assert np.array_equal(gotnull, nulls)
    keep = nulls == 0
    if typname == "float8":
        assert np.array_equal(got[keep].view(np.int64), values[keep].view(np.int64))
    else:
        assert np.array_equal(got[keep], values[keep])


@pytest.mark.skipif(A.ref_lib() is None, reason="reference library only where /root/reference exists")
@pytest.mark.parametrize("case", CASES[:8], ids=[c[0] for c in CASES[:8]])
def test_walker_against_reference_header_accessors(case):
    name, typname, checksum, blocksize, dscale, nblocks, raw, values, nulls = case
    L = A.ref_lib()
    buf = (C.c_ubyte * len(raw)).from_buffer_copy(raw)
    base = C.addressof(buf)
    for off, dlen, rows, first in A.walk_blocks(raw, checksum):
        hlen_guess = 8 + (8 if checksum else 0) + 8
        hdr = base + off - hlen_guess
        hl, rc, dl, kind = C.c_int(), C.c_int(), C.c_int(), C.c_int()
        fr = C.c_int64()
        assert L.ref_aocs_block_info(hdr, checksum, C.byref(hl), C.byref(rc), C.byref(dl), C.byref(fr), C.byref(kind)) == 0
        assert (hl.value, rc.value, dl.value, fr.value, kind.value) == (hlen_guess, rows, dlen, first, 1)
        if checksum:
            assert L.ref_aocs_verify_block(hdr, hlen_guess + (dlen + 7) // 8 * 8) == 0


@pytest.mark.parametrize("case", ZCASES, ids=[c[0] for c in ZCASES])
def test_restated_reader_reads_bulk_compressed_columns(case):
    name, typname, checksum, blocksize, dscale, nblocks, raw, values, nulls, zlevel = case
    blocks = A.walk_blocks_ex(raw, checksum, verify=True)
    assert len(blocks) == nblocks and sum(b["rows"] for b in blocks) == len(values)
    assert blocks[0]["first"] == 1 and all(blocks[i + 1]["first"] == blocks[i]["first"] + blocks[i]["rows"] for i in range(nblocks - 1))
    # the writer keeps a block compressed only when that is shorter (AppendOnlyStorageWrite_CompressAppend :1079-1096)
    assert all(b["clen"] < b["dlen"] for b in blocks)
    assert ("stored" in name) == all(b["clen"] == 0 for b in blocks)
    # more than 16383 rows in a bulk-compressed Dense block -> BulkDenseContent header
    assert all((b["kind"] == 4) == (b["rows"] > 16383) for b in blocks)
    got, gotnull = A.decode_column(raw, typname, checksum, dscale)
    assert np.array_equal(gotnull, nulls)
    keep = nulls == 0
    if typname == "float8":
        assert np.array_equal(got[keep].view(np.int64), values[keep].view(np.int64))
    else:
        assert np.array_equal(got[keep], values[keep])


@pytest.mark.parametrize("case", ZSTDCASES, ids=[c[0] for c in ZSTDCASES])
def test_restated_reader_reads_zstd_columns(case):
    pytest.importorskip("pyarrow")
    name, typname, checksum, blocksize, dscale, nblocks, raw, values, nulls, zlevel = case
    blocks = A.walk_blocks_ex(raw, checksum, verify=True)
    assert len(blocks) == nblocks and sum(b["rows"] for b in blocks) == len(values)
    assert all(b["clen"] < b["dlen"] for b in blocks)
    assert ("stored" in name) == all(b["clen"] == 0 for b in blocks)
    # compressed contents are Zstandard frames
    assert all(raw[b["off"]:b["off"] + 4] == b"\x28\xb5\x2f\xfd" for b in blocks if b["clen"])
    got, gotnull = A.decode_column(raw, typname, checksum, dscale, compresstype="zstd")
    assert np.array_equal(gotnull, nulls)
    keep = nulls == 0
    if typname == "float8":
        assert np.array_equal(got[keep].view(np.int64), values[keep].view(np.int64))
    else:
        assert np.array_equal(got[keep], values[keep])


@pytest.mark.parametrize("case", TCASES, ids=[c[0] for c in TCASES])
def test_restated_reader_reads_string_columns(case):
    name, typname, checksum, blocksize, nblocks, raw, values, nulls, comp = case
    if comp == "zstd":
        pytest.importorskip("pyarrow")
    assert len(A.walk_blocks_ex(raw, checksum, verify=True)) == nblocks
    got, gotnull = A.decode_column(raw, typname, checksum, compresstype=comp or "zlib")
    assert np.array_equal(gotnull, nulls)
    assert [g for g, z in zip(got, nulls) if not z] == [v for v, z in zip(values, nulls) if not z]


@pytest.mark.skipif(A.ref_lib() is None, reason="reference library only where /root/reference exists")
def test_bulk_header_fields_against_reference_accessors():
    L = A.ref_lib()
    for name, typname, checksum, blocksize, dscale, nblocks, raw, values, nulls, zlevel in ZCASES + ZSTDCASES:
        buf = (C.c_ubyte * len(raw)).from_buffer_copy(raw)
        for b in A.walk_blocks_ex(raw, checksum):
            hl, rc, dl, kind = C.c_int(), C.c_int(), C.c_int(), C.c_int()
            fr = C.c_int64()
            assert L.ref_aocs_block_info(C.addressof(buf) + b["hoff"], checksum, C.byref(hl), C.byref(rc), C.byref(dl), C.byref(fr),
                                         C.byref(kind)) == 0, name
            assert (hl.value, rc.value, dl.value, fr.value, kind.value) == (b["hlen"], b["rows"], b["dlen"], b["first"], b["kind"]), name
            assert L.ref_aocs_last_compressed_len() == b["clen"]
            if checksum:
                stored = b["clen"] or b["dlen"]
                assert L.ref_aocs_verify_block(C.addressof(buf) + b["hoff"], b["hlen"] + (stored + 7) // 8 * 8) == 0


def test_checksum_restatement_on_reference_written_files():
    """every checksummed fixture (written by the reference's own block writer) verifies under the restated CRC-32C;
    one flipped content bit / one flipped header bit does not; the known CRC-32C check value pins the polynomial"""
    assert A.crc32c_raw(b"123456789") ^ 0xFFFFFFFF == 0xE3069283
    seen = 0
    for name, typname, checksum, blocksize, dscale, nblocks, raw, values, nulls in CASES:
        if not checksum:
            continue
        assert len(A.walk_blocks(raw, checksum, verify=True)) == nblocks
        seen += 1
        bad = bytearray(raw)
        bad[len(raw) // 2 if len(raw) > 64 else 30] ^= 0x10
        with pytest.raises(ValueError, match="checksum"):
            A.walk_blocks(bytes(bad), checksum, verify=True)
        bad = bytearray(raw)
        bad[5] ^= 0x01                                  # inside header bytes [0,12)
        with pytest.raises(ValueError):
            A.walk_blocks(bytes(bad), checksum, verify=True)
    assert seen >= 10


@pytest.mark.skipif(A.ref_lib() is None, reason="reference library only where /root/reference exists")
def test_numeric_encoding_against_reference_macros():
    L = A.ref_lib()
    rng = np.random.default_rng(3)
    vals = [0, 1, -1, 99, 100, 10000, 123456789012345, -999999999999999, 10**14, 5, 50, 500] + rng.integers(-10**15, 10**15, 300).tolist()
    for dscale in (0, 2, 4, 6):
        for v in vals:
            b = A.numeric_varlena(v, dscale)
            buf = (C.c_ubyte * (len(b) + 8)).from_buffer_copy(b + b"\0" * 8)
            sign, ds, weight, nd = C.c_int(), C.c_int(), C.c_int(), C.c_int()
            digits = (C.c_int16 * 16)()
            short = L.ref_numeric_inspect(C.addressof(buf), C.byref(sign), C.byref(ds), C.byref(weight), C.byref(nd), digits, 16)
            assert short == 1 and ds.value == dscale
            acc = 0
            for i in range(nd.value):
                acc = acc * 10000 + digits[i]
            e10 = 4 * (weight.value - nd.value + 1) + dscale
            got = acc * 10 ** e10 if e10 >= 0 else acc // 10 ** (-e10)
            assert (-got if sign.value else got) == v
            assert A.numeric_from_bytes(b[4:], dscale) == v
