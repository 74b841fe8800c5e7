"""Table-driven tests of the reference that need no GPU, re-run against libswec's host-side entry points (and
the oracle): the expected-shard-size table and the .ecx / .ecj / .idx decode-side cases.

  TestCalculateExpectedShardSize              weed/storage/disk_location_ec_shard_size_test.go:7-143
  TestEcVolumeFileAndDeleteCountInitial / AfterDelete
                                              weed/storage/erasure_coding/ec_volume_counts_test.go:61-130
  TestHasLiveNeedles_*, TestWriteIdxFileFromEcIndex_*, TestDecodeWithNonEmptyEcj_*, TestDecodeWithEmptyEcj,
  TestDecodeWithNoEcjFile                     weed/storage/erasure_coding/ec_decoder_test.go:13-390
"""
import os

import pytest

from oracle import rs_numpy as rn

GB, MB = 1 << 30, 1 << 20
LARGE_BATCH, SMALL_BATCH = 10 * GB, 10 * MB

SHARD_SIZE_TABLE = [                       # (name, datFileSize, expectedShardSize) — the reference's table, verbatim
    ("0 bytes (empty file)", 0, 0),
    ("Exact 10GB (1 large batch)", LARGE_BATCH, GB),
    ("Exact 20GB (2 large batches)", 2 * LARGE_BATCH, 2 * GB),
    ("Just under large batch (10GB - 1 byte)", LARGE_BATCH - 1, 1024 * MB),
    ("Just over large batch (10GB + 1 byte)", LARGE_BATCH + 1, GB + MB),
    ("Exact 10MB (1 small batch)", SMALL_BATCH, MB),
    ("Exact 20MB (2 small batches)", 2 * SMALL_BATCH, 2 * MB),
    ("Just under small batch (10MB - 1 byte)", SMALL_BATCH - 1, MB),
    ("Just over small batch (10MB + 1 byte)", SMALL_BATCH + 1, 2 * MB),
    ("10GB + 1MB", LARGE_BATCH + 1 * MB, GB + MB),
    ("10GB + 5MB", LARGE_BATCH + 5 * MB, GB + MB),
    ("10GB + 15MB", LARGE_BATCH + 15 * MB, GB + 2 * MB),
    ("11GB (1 large batch + 103 small blocks)", 11 * GB, GB + 103 * MB),
    ("5MB (requires 1 small block per shard)", 5 * MB, MB),
    ("1KB (minimum size)", 1024, MB),
    ("10.5GB (mixed)", 10 * GB + 512 * MB, GB + 52 * MB),
]


@pytest.mark.parametrize("name,dat_size,want", SHARD_SIZE_TABLE, ids=[t[0] for t in SHARD_SIZE_TABLE])
def test_calculate_expected_shard_size(swec, oracle, name, dat_size, want):
    assert swec.erasure_coding.expected_shard_size(dat_size) == want
    assert oracle.expected_shard_size(dat_size) == want


def entry(key, actual_offset, size):
    """makeNeedleMapEntry(key, types.ToOffset(actual_offset), size)"""
    return rn._entry(key, actual_offset // 8, size)


def sizes(raw):
    return [(k, s) for k, _, s in rn._entries(raw)]


def test_has_live_needles(swec, tmp_path):
    ec = swec.erasure_coding
    base = str(tmp_path / "foo_1")
    open(base + ".ecx", "wb").write(entry(1, 0, rn.TOMBSTONE))
    assert ec.HasLiveNeedles(base) is False                              # _AllDeletedIsFalse
    open(base + ".ecx", "wb").write(entry(1, 0, 1))
    assert ec.HasLiveNeedles(base) is True                               # _WithLiveEntryIsTrue
    open(base + ".ecx", "wb").write(b"")
    assert ec.HasLiveNeedles(base) is False                              # _EmptyFileIsFalse


def test_write_idx_file_from_ec_index_preserves_deleted_needles(swec, tmp_path):
    ec = swec.erasure_coding
    base = str(tmp_path / "foo_1")
    ecx = entry(1, 64, 100) + entry(2, 128, rn.TOMBSTONE)
    open(base + ".ecx", "wb").write(ecx)
    ec.WriteIdxFileFromEcIndex(base)
    idx = open(base + ".idx", "rb").read()
    assert idx == ecx and sizes(idx)[1][1] < 0


def test_write_idx_file_from_ec_index_processes_ecj_journal(swec, tmp_path):
    ec = swec.erasure_coding
    base = str(tmp_path / "foo_1")
    open(base + ".ecx", "wb").write(entry(1, 64, 100) + entry(2, 128, 200))
    open(base + ".ecj", "wb").write((2).to_bytes(8, "big"))
    ec.WriteIdxFileFromEcIndex(base)
    got = sizes(open(base + ".idx", "rb").read())
    assert len(got) == 3 and got[2][0] == 2 and got[2][1] < 0            # 2 from .ecx + 1 deletion record


def test_decode_with_non_empty_ecj_all_deleted(swec, tmp_path):
    ec = swec.erasure_coding
    base = str(tmp_path / "test_1")
    open(base + ".ecx", "wb").write(entry(1, 64, 100) + entry(2, 128, 200))
    open(base + ".ecj", "wb").write((1).to_bytes(8, "big") + (2).to_bytes(8, "big"))
    assert ec.HasLiveNeedles(base) is True                               # before the merge
    ec.RebuildEcxFile(base)
    assert not os.path.exists(base + ".ecj")
    assert ec.HasLiveNeedles(base) is False
    ec.WriteIdxFileFromEcIndex(base)
    got = sizes(open(base + ".idx", "rb").read())
    assert len(got) == 2 and all(s < 0 for _, s in got)


def test_decode_with_non_empty_ecj_partially_deleted(swec, tmp_path):
    ec = swec.erasure_coding
    base = str(tmp_path / "test_1")
    open(base + ".ecx", "wb").write(entry(1, 64, 100) + entry(2, 128, 200) + entry(3, 256, 300))
    open(base + ".ecj", "wb").write((2).to_bytes(8, "big"))
    ec.RebuildEcxFile(base)
    assert ec.HasLiveNeedles(base) is True
    ec.WriteIdxFileFromEcIndex(base)
    got = dict(sizes(open(base + ".idx", "rb").read()))
    assert len(got) == 3 and got[1] == 100 and got[3] == 300 and got[2] < 0


@pytest.mark.parametrize("ecj", [b"", None], ids=["empty_ecj", "no_ecj_file"])
def test_decode_with_empty_or_missing_ecj(swec, tmp_path, ecj):
    """TestDecodeWithEmptyEcj / TestDecodeWithNoEcjFile: nothing to merge, everything stays live."""
    ec = swec.erasure_coding
    base = str(tmp_path / "test_1")
    ecx = entry(1, 64, 100) + entry(2, 128, 200)
    open(base + ".ecx", "wb").write(ecx)
    if ecj is not None:
        open(base + ".ecj", "wb").write(ecj)
    ec.RebuildEcxFile(base)
    assert open(base + ".ecx", "rb").read() == ecx and ec.HasLiveNeedles(base) is True
    ec.WriteIdxFileFromEcIndex(base)
    assert open(base + ".idx", "rb").read() == ecx


def _mount_fixture(ec, tmp_path, ecx, ecj_ids):
    """writeFixture (ec_volume_counts_test.go:34-57): .ecx, .ecj, an 8-byte .ec00 and an EMPTY .vif"""
    base = str(tmp_path / "test_1")
    open(base + ".ecx", "wb").write(ecx)
    open(base + ".ecj", "wb").write(b"".join(i.to_bytes(8, "big") for i in ecj_ids))
    open(base + ".ec00", "wb").write(bytes(8))
    open(base + ".vif", "wb").write(b"")
    return ec.EcVolume(base, device=-1)


def test_ec_volume_file_and_delete_count_initial(swec, tmp_path):
    ec = swec.erasure_coding
    ev = _mount_fixture(ec, tmp_path, entry(1, 64, 100) + entry(2, 128, 200) + entry(3, 256, 300), [2, 3])
    assert ev.FileAndDeleteCount() == (3, 2)
    ev.close()


def test_ec_volume_file_and_delete_count_after_delete(swec, tmp_path):
    ec = swec.erasure_coding
    ev = _mount_fixture(ec, tmp_path, entry(1, 64, 100) + entry(2, 128, 200), [])
    assert ev.FileAndDeleteCount() == (2, 0)
    ev.DeleteNeedleFromEcx(2)
    assert ev.FileAndDeleteCount() == (2, 1)
    ev.DeleteNeedleFromEcx(2)                                            # idempotent
    assert ev.FileAndDeleteCount() == (2, 1)
    ev.DeleteNeedleFromEcx(99)                                           # not in the volume
    assert ev.FileAndDeleteCount() == (2, 1)
    ev.close()


# ---- TestCheckIndexFile (weed/storage/idx/check_test.go:11-108): the reference's six index fixtures with the counts
# ---- and the exact findings its test expects — K11 of oracle/README.md.  EcVolume.ScrubIndex runs this on .ecx.
IDX_FIXTURES = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "fixtures", "idx")
CHECK_INDEX_CASES = [
    ("simple_index.idx", 161, []),
    ("deleted_files.idx", 230, []),
    ("simple_index_bitrot.idx", 161, [
        "needle 3544668469065756977 (#2) at [6602459528-7427766999] overlaps needle 49 at [6602459528-7427766999]",
        "expected an index file of size 2577, got 2576"]),
    ("simple_index_truncated.idx", 158, ["expected an index file of size 2540, got 2528"]),
    ("deleted_files.ecx", 116, []),
    ("deleted_files_bitrot.ecx", 116, [
        "needle 3223857 (#110) at [6602459528-7427767055] overlaps needle 12593 at [6601933184-7407907279]",
        "needle 3544668469065757234 (#43) at [6737203600-7579354079] overlaps needle 3223857 at [6602459528-7427767055]",
        "needle 3421236 (#112) at [7006693800-7899362591] overlaps needle 3544668469065757234 at [6737203600-7579354079]",
        "needle 310 (#113) at [7276179888-8185702583] overlaps needle 3421236 at [7006693800-7899362591]",
        "needle 7089336938131513954 (#52) at [13204919056-13205053935] overlaps needle 27410143614427489 at [13070174984-14703946887]",
        "needle 25186 (#50) at [13204919056-14855533967] overlaps needle 7089336938131513954 at [13204919056-13205053935]",
        "needle 7089336938131513954 (#51) at [13204919056-14855533967] overlaps needle 25186 at [13204919056-14855533967]",
        "expected an index file of size 1857, got 1856"]),
]


@pytest.mark.parametrize("name,want_count,want_errs", CHECK_INDEX_CASES, ids=[c[0] for c in CHECK_INDEX_CASES])
def test_check_index_file_on_reference_fixtures(swec, name, want_count, want_errs):
    path = os.path.join(IDX_FIXTURES, name)
    count, errs = swec.erasure_coding.CheckIndexFile(path, 3)
    assert count == want_count
    assert errs == want_errs
    assert rn.check_index_file(open(path, "rb").read(), 3) == (want_count, want_errs)      # the oracle's restatement too


def test_check_index_file_fuzz_against_oracle(swec, tmp_path):
    """Random indexes with overlaps, tombstones, zero and huge sizes and ragged tails: product == oracle."""
    import numpy as np
    rng = np.random.default_rng(0)
    for case in range(60):
        n = int(rng.integers(0, 60))
        raw = b""
        for _ in range(n):
            size = int(rng.choice([rng.integers(0, 5000), -1, -int(rng.integers(2, 5000)), 0x7FFFFFF0 + int(rng.integers(0, 15)),
                                   int(rng.integers(0, 1 << 31))]))
            raw += rn._entry(int(rng.integers(1, 1 << 40)), int(rng.integers(0, 3000)), size)
        raw += bytes(int(rng.integers(0, 16)) if case % 3 == 0 else 0)
        path = tmp_path / f"f{case}.ecx"
        path.write_bytes(raw)
        for version in (2, 3):
            assert swec.erasure_coding.CheckIndexFile(str(path), version) == rn.check_index_file(raw, version), (case, version)


@pytest.mark.parametrize("dat_size,actual_shard,valid", [(10 * GB, GB, True), (10 * GB, GB - 1, False), (10 * GB, GB + 1, False),
                                                         (5 * MB, MB, True), (5 * MB, 500 * 1024, False)])
def test_shard_size_validation_scenarios(swec, dat_size, actual_shard, valid):
    """TestShardSizeValidationScenarios (disk_location_ec_shard_size_test.go:145-200)"""
    assert (swec.erasure_coding.expected_shard_size(dat_size) == actual_shard) is valid


# ---- the Rust twin's locate tests (seaweed-volume/src/storage/erasure_coding/ec_locate.rs:139-233) -------------

def test_rust_twin_interval_to_shard_id(swec):
    ec = swec.erasure_coding
    L, S = 1 << 30, 1 << 20
    # (BlockIndex, InnerBlockOffset, Size, IsLargeBlock, LargeBlockRowsCount) → (shard, offset)
    assert ec.interval_to_shard((0, 100, 50, True, 1), L, S) == (0, 100)
    assert ec.interval_to_shard((5, 0, 1024, True, 1), L, S)[0] == 5
    assert ec.interval_to_shard((12, 200, 50, True, 5), L, S) == (2, L + 200)      # row 1 of shard 2
    assert ec.interval_to_shard((10, 0, 100, True, 2), L, S) == (0, L)
    assert ec.interval_to_shard((0, 0, 100, False, 2), L, S) == (0, 2 * L)         # test_small_block_after_large


def test_rust_twin_locate_data_small_and_empty(swec):
    ec = swec.erasure_coding
    ivs = ec.LocateData(1 << 30, 1 << 20, 1 << 20, 50, 100)                        # test_locate_data_small_file
    assert len(ivs) == 1 and ivs[0][3] is False
    assert ec.LocateData(1 << 30, 1 << 20, 1 << 20, 0, 0) == []                    # test_locate_data_empty


# ---- the Rust twin's EcVolume tests (seaweed-volume/src/storage/erasure_coding/ec_volume.rs:1097-1230) ----------

def test_rust_twin_ec_volume_find_needle_and_journal(swec, tmp_path):
    ec = swec.erasure_coding
    ev = _mount_fixture(ec, tmp_path, entry(1, 8, 100) + entry(5, 200, 200) + entry(10, 504, 300), [])
    out = ev.ReadEcShardNeedles([5, 7], capacity=16)
    assert (out[0]["offset"], out[0]["size"]) == (200, 200)                    # found (the 16-byte buffer is too small to read into)
    assert out[1]["status"] == "SWEC_ERR_NOT_FOUND"
    assert ev.FileAndDeleteCount() == (3, 0)
    ev.DeleteNeedleFromEcx(1)
    ev.DeleteNeedleFromEcx(10)
    assert open(str(tmp_path / "test_1.ecj"), "rb").read() == (1).to_bytes(8, "big") + (10).to_bytes(8, "big")
    assert ev.FileAndDeleteCount() == (3, 2)
    ev.DeleteNeedleFromEcx(1)                                                  # idempotent
    ev.DeleteNeedleFromEcx(999)                                                # missing
    assert ev.FileAndDeleteCount() == (3, 2)
    ev.close()


@pytest.mark.parametrize("vif,want", [({"dataShards": 6, "parityShards": 3}, (6, 3)),        # config from .vif
                                      ({"dataShards": 30, "parityShards": 9}, (10, 4)),      # invalid: > MaxShardCount ⇒ defaults
                                      ({"dataShards": 0, "parityShards": 4}, (10, 4)),
                                      (None, (10, 4))])
def test_ec_volume_ratio_from_vif(swec, tmp_path, vif, want):
    """NewEcVolume (ec_volume.go:114-154): EC ratio from .vif when valid (ds > 0, ps > 0, ds + ps <= 32), else 10+4."""
    import json
    ec = swec.erasure_coding
    base = str(tmp_path / "pics_1")
    open(base + ".ecx", "wb").write(b"")
    open(base + ".ec00", "wb").write(bytes(8))
    if vif is not None:
        json.dump({"version": 2, "datFileSize": "123456", "ecShardConfig": vif}, open(base + ".vif", "w"))
    ev = ec.EcVolume(base, device=-1)
    info = ev.info()
    assert (info["data_shards"], info["parity_shards"]) == want
    assert info["version"] == (2 if vif is not None else 3) and info["local_shards"] == [0]
    assert info["shard_dat_size"] == (123456 // want[0] if vif is not None else 8 - 1)
    ev.close()


@pytest.mark.parametrize("text,want", [
    # member order reversed, a decoy key inside a string value, escapes, nested arrays before the real object
    ('{"bytesOffset": 7, "note": "\\"ecShardConfig\\": {\\"dataShards\\": 3}", "files": [{"dataShards": 5}], '
     '"ecShardConfig": {"parityShards": "2", "dataShards": 7}, "datFileSize": "99", "version": 3}', (7, 2, 99, 3)),
    # proto field names (protojson accepts both spellings), numbers unquoted, odd whitespace
    ('{\n"version"\t:\t2 ,"dat_file_size":1234,"ec_shard_config":{ "data_shards" : 4 ,\n "parity_shards":1}}', (4, 1, 1234, 2)),
    # dataShards appears only OUTSIDE ecShardConfig: the ratio must fall back to 10+4
    ('{"dataShards": 6, "parityShards": 3, "version": 3, "datFileSize": "50"}', (10, 4, 50, 3)),
    # malformed JSON: nothing is taken from it
    ('{"version": 2, "ecShardConfig": {"dataShards": 6, "parityShards": 3', (10, 4, None, 3)),
])
def test_vif_is_parsed_as_json_not_by_substring(swec, tmp_path, text, want):
    """.vif is protobuf-JSON (weed/storage/volume_info/volume_info.go:73-95): member order, escapes and look-alike keys
    inside strings or other objects must not matter (csrc/mini_json.h)."""
    ec = swec.erasure_coding
    base = str(tmp_path / "v_1")
    open(base + ".ecx", "wb").write(b"")
    open(base + ".ec00", "wb").write(bytes(8))
    open(base + ".vif", "w").write(text)
    ev = ec.EcVolume(base, device=-1)
    info = ev.info()
    ds, ps, dat, ver = want
    assert (info["data_shards"], info["parity_shards"], info["version"]) == (ds, ps, ver)
    assert info["shard_dat_size"] == (dat // ds if dat is not None else 8 - 1)
    ev.close()
