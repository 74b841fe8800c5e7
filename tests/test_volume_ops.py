"""Whole-volume operations — the file work of VolumeEcShardsGenerate / VolumeEcShardsRebuild /
VolumeEcShardsToVolume (weed/server/volume_grpc_erasure_coding.go:43-225,578-668) as single C-ABI calls.
The CPU tests cover everything that needs no GPU (ec.decode side, ordering, cleanup-on-error, error
mapping) with shard files written by the oracle; the GPU tests run the full encode → damage → rebuild →
decode cycle on the reference's fixture volume and compare every produced file with the oracle's."""
import json
import os

import numpy as np
import pytest

from oracle import rs_numpy as rn

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FIXTURES = os.path.join(ROOT, "tests", "golden", "fixtures")
FIXTURE_IDX = os.path.join(FIXTURES, "1.idx")
FIXTURE_DAT = os.path.join(FIXTURES, "1.dat")
MIB = 1 << 20


def synthetic_volume(seed=11, needles=120, version=3):
    """A well-formed miniature volume: 8-byte superblock (byte 0 = needle version) followed by 8-byte
    aligned needle records, plus the .idx that indexes them (with overwrites and deletions)."""
    rng = np.random.default_rng(seed)
    dat = bytearray([version, 0, 0, 0, 0, 0, 0, 0])
    idx = b""
    for i in range(needles):
        key = int(rng.integers(1, needles // 2))
        size = int(rng.integers(1, 40000))
        fixed = 16 + size + 4 + (8 if version == 3 else 0)
        actual = fixed + (8 - fixed % 8)
        offset = len(dat) // 8
        dat += rng.integers(0, 256, actual, dtype=np.uint8).tobytes()
        kind = int(rng.integers(0, 12))
        if kind == 0:
            idx += rn._entry(key, offset, rn.TOMBSTONE)
        else:
            idx += rn._entry(key, offset, size)
    return np.frombuffer(bytes(dat), dtype=np.uint8).copy(), idx


def lay_down_ec_volume(oracle, tmp_path, dat, idx, k=10, m=4, name="7"):
    """What a finished ec.encode leaves on disk, written by the ORACLE (production block sizes)."""
    base = str(tmp_path / name)
    shards = oracle.encode_dat_image(dat, k=k, m=m)
    for i, s in enumerate(shards):
        s.tofile(base + ".ec%02d" % i)
    open(base + ".ecx", "wb").write(rn.sorted_ecx_from_idx(idx))
    return base, shards


def read_vif(path):
    v = json.load(open(path))
    return {"version": int(v["version"]), "datFileSize": int(v["datFileSize"]), "expireAtSec": int(v["expireAtSec"]),
            "ds": int(v["ecShardConfig"]["dataShards"]), "ps": int(v["ecShardConfig"]["parityShards"]),
            "files": v["files"], "readOnly": v["readOnly"], "replication": v["replication"],
            "bytesOffset": v["bytesOffset"]}


# ------------------------------------------------------------------------------------------ CPU

def test_ec_shards_to_volume_roundtrip(swec, oracle, tmp_path):
    """ec.decode: shards + .ecx + .ecj → .dat + .idx.  The decoded .dat is the original up to the end of the
    last live needle (FindDatFileSize), the .idx is .ecx plus one tombstone per journalled id."""
    ec = swec.erasure_coding
    dat, idx = synthetic_volume()
    base, _ = lay_down_ec_volume(oracle, tmp_path, dat, idx)
    ecx = rn.sorted_ecx_from_idx(idx)
    keys = [k for k, _, _ in rn._entries(ecx)]
    ecj = b"".join(k.to_bytes(8, "big") for k in keys[:3])
    open(base + ".ecj", "wb").write(ecj)

    size = ec.VolumeEcShardsToVolume(base)
    folded = rn.fold_ecj_into_ecx(ecx, ecj)
    assert open(base + ".ecx", "rb").read() == folded and not os.path.exists(base + ".ecj")
    assert size == rn.find_dat_file_size(folded, 3)
    out = np.fromfile(base + ".dat", dtype=np.uint8)
    assert len(out) == size <= len(dat) and (out == dat[:size]).all()
    assert open(base + ".idx", "rb").read() == rn.idx_from_ec_index(folded, b"")


def test_ec_shards_to_volume_shards_on_other_disks_and_custom_ratio(swec, oracle, tmp_path):
    """Multi-disk servers keep shards of one volume in several directories; the ratio comes from .vif."""
    ec = swec.erasure_coding
    dat, idx = synthetic_volume(seed=5, needles=60)
    k, m = 6, 3
    base, shards = lay_down_ec_volume(oracle, tmp_path, dat, idx, k=k, m=m)
    json.dump({"version": 3, "datFileSize": str(len(dat)), "ecShardConfig": {"dataShards": k, "parityShards": m}},
              open(base + ".vif", "w"))
    other = tmp_path / "disk2"
    other.mkdir()
    for i in (1, 4):
        os.rename(base + ".ec%02d" % i, str(other / ("7.ec%02d" % i)))
    size = ec.VolumeEcShardsToVolume(base, additional_dirs=[str(other)])
    out = np.fromfile(base + ".dat", dtype=np.uint8)
    assert (out == dat[:size]).all() and size > len(dat) - 64 * 1024

    os.remove(str(other / "7.ec04"))                     # a data shard is gone: the handler refuses
    with pytest.raises(swec.SwecError) as e:
        ec.VolumeEcShardsToVolume(base, additional_dirs=[str(other)])
    assert e.value.name == "SWEC_ERR_TOO_FEW_SHARDS" and "missing shard 4" in str(e.value)


def test_ec_shards_to_volume_without_live_needles(swec, oracle, tmp_path):
    """All needles deleted ⇒ FailedPrecondition 'no live entries' (issue-7748 path): nothing is written."""
    ec = swec.erasure_coding
    dat, idx = synthetic_volume(seed=2, needles=30)
    base, _ = lay_down_ec_volume(oracle, tmp_path, dat, idx)
    keys = [k for k, _, _ in rn._entries(rn.sorted_ecx_from_idx(idx))]
    open(base + ".ecj", "wb").write(b"".join(k.to_bytes(8, "big") for k in keys))
    with pytest.raises(swec.SwecError) as e:
        ec.VolumeEcShardsToVolume(base)
    assert e.value.name == "SWEC_ERR_NO_LIVE_NEEDLES" and "no live entries" in str(e.value)
    assert not os.path.exists(base + ".dat") and not os.path.exists(base + ".idx")


def test_ec_shards_generate_cleans_up_on_error(swec, tmp_path):
    """Any failure after the .ecx was written removes the .ecx and every shard file (the handler's deferred
    cleanup, volume_grpc_erasure_coding.go:78-87).  Here the failure is the missing GPU: device -1 has no
    CPU fallback, so the shard step fails after .ecx and the 14 truncated shard files exist."""
    ec = swec.erasure_coding
    dat, idx = synthetic_volume(seed=3, needles=20)
    base = str(tmp_path / "9")
    dat.tofile(base + ".dat")
    open(base + ".idx", "wb").write(idx)
    with pytest.raises(swec.SwecError) as e:
        ec.VolumeEcShardsGenerate(base, device=-1)
    assert e.value.name == "SWEC_ERR_NO_DEVICE"
    left = sorted(os.listdir(tmp_path))
    assert left == ["9.dat", "9.idx"], left
    # no .idx at all: fails before anything is created
    os.remove(base + ".idx")
    with pytest.raises(swec.SwecError) as e:
        ec.VolumeEcShardsGenerate(base, device=-1)
    assert e.value.name == "SWEC_ERR_IO" and sorted(os.listdir(tmp_path)) == ["9.dat"]


def test_ec_shards_rebuild_prechecks_need_no_gpu(swec, oracle, tmp_path):
    """Too few shards is detected before any output exists; with nothing missing only the .ecj fold runs."""
    ec = swec.erasure_coding
    dat, idx = synthetic_volume(seed=8, needles=25)
    base, _ = lay_down_ec_volume(oracle, tmp_path, dat, idx)
    keys = [k for k, _, _ in rn._entries(rn.sorted_ecx_from_idx(idx))]
    open(base + ".ecj", "wb").write(keys[0].to_bytes(8, "big"))
    assert ec.VolumeEcShardsRebuild(base, device=-1) == []          # nothing missing: no GPU needed
    assert not os.path.exists(base + ".ecj")
    assert sum(1 for _, _, s in rn._entries(open(base + ".ecx", "rb").read()) if s < 0) == 1
    for i in range(5):
        os.remove(base + ".ec%02d" % i)
    with pytest.raises(swec.SwecError) as e:
        ec.VolumeEcShardsRebuild(base, device=-1)
    assert e.value.name == "SWEC_ERR_TOO_FEW_SHARDS"
    assert not any(os.path.exists(base + ".ec%02d" % i) for i in range(5))


def expected_record(dat, offset, size, version=3):
    """What ReadEcShardNeedle's `bytes` holds — the oracle's restatement (GetActualSize applied twice)."""
    return rn.read_needle_record(dat, offset, size, version)


def needle_volume(oracle, tmp_path, seed=17, with_vif=True):
    dat, idx = synthetic_volume(seed=seed, needles=600)          # ≈12 MiB, two small rows: records straddle 1 MiB block borders
    base, shards = lay_down_ec_volume(oracle, tmp_path, dat, idx)
    if with_vif:
        json.dump({"version": 3, "datFileSize": str(len(dat)), "ecShardConfig": {"dataShards": 10, "parityShards": 4}},
                  open(base + ".vif", "w"))
    live = [(k, o, s) for k, o, s in rn._entries(rn.sorted_ecx_from_idx(idx))]
    return base, dat, live


def test_read_ec_needles_all_shards_local_needs_no_gpu(swec, oracle, tmp_path):
    ec = swec.erasure_coding
    base, dat, live = needle_volume(oracle, tmp_path)
    assert len(live) > 50
    open(base + ".ecj", "wb").write(live[3][0].to_bytes(8, "big"))       # deleted after sealing
    ids = [k for k, _, _ in live] + [0xFFFFFFFFFF]
    out = ec.ReadEcShardNeedles(base, ids, device=-1)                     # no recovery ⇒ no device needed
    multi = 0
    for (key, off, size), r in zip(live, out):
        if key == live[3][0]:
            assert r["status"] == "SWEC_ERR_DELETED" and r["size"] == -1
            continue
        assert r["status"] == "SWEC_OK" and r["offset"] == off * 8 and r["size"] == size and r["recovered_intervals"] == 0
        want = expected_record(dat, off * 8, size)
        assert r["n_bytes"] == len(want) and (r["bytes"] == want).all(), key
        multi += (off * 8) // MIB != (off * 8 + len(want) - 1) // MIB
    assert multi >= 1, "the volume should contain records that straddle block borders"
    assert out[-1]["status"] == "SWEC_ERR_NOT_FOUND"
    tiny = ec.ReadEcShardNeedles(base, [live[0][0]], device=-1, capacity=8)
    assert tiny[0]["status"] == "SWEC_ERR_INVALID_ARG" and tiny[0]["n_bytes"] == len(expected_record(dat, 0, live[0][2]))


def test_mounted_ec_volume_sees_journal_growth(swec, oracle, tmp_path):
    """An EcVolume handle stays open across reads; a needle deleted meanwhile (DeleteNeedleFromEcx appends its
    id to .ecj) reads as deleted on the next call, like the reference's in-memory deleted set."""
    ec = swec.erasure_coding
    base, dat, live = needle_volume(oracle, tmp_path, seed=19)
    vol = ec.EcVolume(base, device=-1)
    ids = [k for k, _, _ in live[:20]]
    first = vol.ReadEcShardNeedles(ids)
    assert all(r["status"] == "SWEC_OK" for r in first)
    with open(base + ".ecj", "ab") as f:
        f.write(ids[5].to_bytes(8, "big"))
    second = vol.ReadEcShardNeedles(ids)
    assert [r["status"] for r in second] == ["SWEC_ERR_DELETED" if i == 5 else "SWEC_OK" for i in range(20)]
    assert all((a["bytes"] == b["bytes"]).all() for i, (a, b) in enumerate(zip(first, second)) if i != 5)
    # DeleteNeedleFromEcx: journal append, idempotent, unknown ids ignored; then the fold sees all of it
    vol.DeleteNeedleFromEcx(ids[7])
    vol.DeleteNeedleFromEcx(ids[7])
    vol.DeleteNeedleFromEcx(ids[5])                                      # journalled by someone else already
    vol.DeleteNeedleFromEcx(0xABCDEF0123)                                # not in the volume
    assert open(base + ".ecj", "rb").read() == ids[5].to_bytes(8, "big") + ids[7].to_bytes(8, "big")
    third = vol.ReadEcShardNeedles(ids)
    assert [i for i, r in enumerate(third) if r["status"] == "SWEC_ERR_DELETED"] == [5, 7]
    vol.close()
    ec.RebuildEcxFile(base)
    assert sum(1 for _, _, sz in rn._entries(open(base + ".ecx", "rb").read()) if sz < 0) == 2
    vol = ec.EcVolume(base, device=-1)                                   # tombstones in .ecx read as deleted too
    assert [r["status"] for r in vol.ReadEcShardNeedles([ids[5], ids[6]])] == ["SWEC_ERR_DELETED", "SWEC_OK"]
    vol.DeleteNeedleFromEcx(ids[5])                                      # already folded: nothing journalled
    assert not os.path.exists(base + ".ecj") or os.path.getsize(base + ".ecj") == 0
    vol.close()
    with pytest.raises(swec.SwecError) as e:
        ec.EcVolume(str(tmp_path / "nothing-here"), device=-1)
    assert e.value.name == "SWEC_ERR_TOO_FEW_SHARDS"


def test_ecx_search_on_reference_fixture_389(swec, tmp_path):
    """TestPositioning (ec_volume_test.go:14-58): SearchNeedleFromSortedIndex on a 2048-entry sample of the
    reference's 389.ecx (485,098 entries) finds the needles of its table at the listed offsets and sizes.  The
    fixture has no shard files, so the reads themselves stop at "too few shards" — offset and size are reported
    all the same."""
    fixture = os.path.join(FIXTURES, "389_sample.ecx")
    ec = swec.erasure_coding
    base = str(tmp_path / "389")
    os.symlink(fixture, base + ".ecx")
    open(base + ".ec00", "wb").write(b"\x03" + b"\x00" * 7)           # a mounted volume needs one local shard
    table = [(0x0F0EDB92, 31300679656, 1167), (0x0EF7D7F8, 11513014944, 66044)]
    out = ec.ReadEcShardNeedles(base, [t[0] for t in table] + [0x0F087622, 1], device=-1)
    for (nid, offset, size), r in zip(table, out):
        assert (r["offset"], r["size"]) == (offset, size), hex(nid)
        assert r["status"] == "SWEC_ERR_TOO_FEW_SHARDS"
    assert out[2]["status"] == "SWEC_ERR_TOO_FEW_SHARDS" and out[2]["offset"] > 0      # found, like the Go test asserts
    assert out[3]["status"] == "SWEC_ERR_NOT_FOUND"


def test_read_ec_needles_old_volume_without_vif(swec, oracle, tmp_path):
    """No .vif ⇒ needle version 3 and shard size = shard file size - 1 (ec_volume.go:408-413)."""
    ec = swec.erasure_coding
    base, dat, live = needle_volume(oracle, tmp_path, seed=23, with_vif=False)
    out = ec.ReadEcShardNeedles(base, [k for k, _, _ in live[:40]], device=-1)
    for (key, off, size), r in zip(live, out):
        assert r["status"] == "SWEC_OK" and (r["bytes"] == expected_record(dat, off * 8, size)).all()


def test_read_ec_needles_recovery_is_loud_without_gpu(swec, oracle, tmp_path):
    ec = swec.erasure_coding
    base, dat, live = needle_volume(oracle, tmp_path, seed=29)
    os.remove(base + ".ec00")
    with pytest.raises(swec.SwecError) as e:
        ec.ReadEcShardNeedles(base, [k for k, _, _ in live], device=-1)
    assert e.value.name == "SWEC_ERR_NO_DEVICE"


# ------------------------------------------------------------------------------------------ GPU

@pytest.mark.gpu
@pytest.mark.parametrize("lost", [(0,), (2, 5), (0, 1, 2, 3), (1, 9, 10, 13)])
def test_read_ec_needles_degraded(cuda, swec, oracle, tmp_path, lost):
    """Degraded reads: the shard files in `lost` are gone; every record is still returned byte-exactly, the
    intervals that lived on lost shards being rebuilt by one batched ReconstructData on the GPU."""
    ec = swec.erasure_coding
    base, dat, live = needle_volume(oracle, tmp_path, seed=41 + len(lost))
    other = tmp_path / "disk2"
    other.mkdir()
    os.rename(base + ".ec06", str(other / "7.ec06"))                      # one healthy shard lives on another disk
    for i in lost:
        os.remove(base + ".ec%02d" % i)
    before = swec.lib().swec_kernel_launches()
    out = ec.ReadEcShardNeedles(base, [k for k, _, _ in live], additional_dirs=[str(other)])
    recovered = 0
    for (key, off, size), r in zip(live, out):
        assert r["status"] == "SWEC_OK", (key, r["status"])
        assert (r["bytes"] == expected_record(dat, off * 8, size)).all(), key
        recovered += r["recovered_intervals"]
    data_lost = [i for i in lost if i < 10]
    assert (recovered > 0) == bool(data_lost)
    launches = swec.lib().swec_kernel_launches() - before
    assert launches <= 8 if data_lost else launches == 0, launches       # batched: not one launch per interval


@pytest.mark.gpu
def test_mounted_ec_volume_degraded_reads_reuse_the_encoder(cuda, swec, oracle, tmp_path):
    """One needle per call on a mounted volume (the shape of today's read path): the handle's encoder, staging
    ring and kernels are created once, so a lone degraded read costs one small launch, not a re-initialisation."""
    import time
    ec = swec.erasure_coding
    base, dat, live = needle_volume(oracle, tmp_path, seed=53)
    for i in (0, 1, 2, 3):
        os.remove(base + ".ec%02d" % i)
    vol = ec.EcVolume(base)
    vol.ReadEcShardNeedles([live[0][0]], capacity=1 << 16)
    t0, n, recovered = time.perf_counter(), 0, 0
    for key, off, size in live[:200]:
        r = vol.ReadEcShardNeedles([key], capacity=1 << 17)[0]
        assert r["status"] == "SWEC_OK" and (r["bytes"] == expected_record(dat, off * 8, size)).all()
        recovered += r["recovered_intervals"]
        n += 1
    per_call = (time.perf_counter() - t0) / n
    assert recovered > 20
    assert per_call < 0.02, f"{per_call * 1e3:.1f} ms per single-needle read: the encoder is not being reused"
    vol.close()


@pytest.mark.gpu
def test_read_ec_needles_too_few_shards(cuda, swec, oracle, tmp_path):
    ec = swec.erasure_coding
    base, dat, live = needle_volume(oracle, tmp_path, seed=47)
    for i in (0, 1, 2, 3, 4):
        os.remove(base + ".ec%02d" % i)
    out = ec.ReadEcShardNeedles(base, [k for k, _, _ in live])
    kinds = {r["status"] for r in out}
    assert kinds == {"SWEC_OK", "SWEC_ERR_TOO_FEW_SHARDS"}               # records wholly on shards 5-9 still read
    for (key, off, size), r in zip(live, out):
        if r["status"] == "SWEC_OK":
            assert r["recovered_intervals"] == 0 and (r["bytes"] == expected_record(dat, off * 8, size)).all()


@pytest.mark.gpu
@pytest.mark.parametrize("volume", ["fixture", "synthetic"])
def test_volume_encode_rebuild_decode_cycle(cuda, swec, oracle, kat, tmp_path, volume):
    """ec.encode → lose shards → ec.rebuild → ec.decode through the three handler-level calls; every file
    is compared with the oracle's (and the fixture's shards with the committed golden digests)."""
    import hashlib
    ec = swec.erasure_coding
    if volume == "fixture":
        dat, idx = np.fromfile(FIXTURE_DAT, dtype=np.uint8), open(FIXTURE_IDX, "rb").read()
    else:
        dat, idx = synthetic_volume(seed=21, needles=400)          # ≈8 MiB: one ragged small row
    base = str(tmp_path / "1")
    dat.tofile(base + ".dat")
    open(base + ".idx", "wb").write(idx)

    ec.VolumeEcShardsGenerate(base, expire_at_sec=1234)
    want = oracle.encode_dat_image(dat)
    for i in range(14):
        got = np.fromfile(base + ec.ToExt(i), dtype=np.uint8)
        assert got.shape == want[i].shape and (got == want[i]).all(), f"shard {i}"
    if volume == "fixture":
        golden = kat["K8"]["production"]["sha256"]
        for i in range(14):
            assert hashlib.sha256(open(base + ec.ToExt(i), "rb").read()).hexdigest() == golden[i]
    ecx = rn.sorted_ecx_from_idx(idx)
    assert open(base + ".ecx", "rb").read() == ecx
    vif = read_vif(base + ".vif")
    assert vif == {"version": int(dat[0]), "datFileSize": len(dat), "expireAtSec": 1234, "ds": 10, "ps": 4,
                   "files": [], "readOnly": False, "replication": "", "bytesOffset": 0}

    # a server dies: four shards gone (two data, two parity); some needles deleted meanwhile
    for i in (0, 7, 10, 13):
        os.remove(base + ec.ToExt(i))
    keys = [k for k, _, _ in rn._entries(ecx)]
    ecj = b"".join(k.to_bytes(8, "big") for k in keys[:2])
    open(base + ".ecj", "wb").write(ecj)
    assert ec.VolumeEcShardsRebuild(base) == [0, 7, 10, 13]
    for i in range(14):
        assert (np.fromfile(base + ec.ToExt(i), dtype=np.uint8) == want[i]).all(), f"rebuilt shard {i}"
    folded = rn.fold_ecj_into_ecx(ecx, ecj)
    assert open(base + ".ecx", "rb").read() == folded

    os.remove(base + ".dat")
    os.remove(base + ".idx")
    size = ec.VolumeEcShardsToVolume(base)
    assert size == rn.find_dat_file_size(folded, int(dat[0]))
    assert (np.fromfile(base + ".dat", dtype=np.uint8) == dat[:size]).all()
    assert open(base + ".idx", "rb").read() == rn.idx_from_ec_index(folded, b"")


@pytest.mark.gpu
def test_volume_generate_keeps_ratio_of_existing_vif(cuda, swec, oracle, tmp_path):
    """Regeneration keeps the EC ratio recorded in an existing .vif (volume_grpc_erasure_coding.go:61-77);
    an invalid recorded ratio falls back to 10+4."""
    ec = swec.erasure_coding
    dat, idx = synthetic_volume(seed=31, needles=50)
    base = str(tmp_path / "3")
    dat.tofile(base + ".dat")
    open(base + ".idx", "wb").write(idx)
    json.dump({"version": 3, "ecShardConfig": {"dataShards": 5, "parityShards": 2}}, open(base + ".vif", "w"))
    ec.VolumeEcShardsGenerate(base)
    want = oracle.encode_dat_image(dat, k=5, m=2)
    for i in range(7):
        assert (np.fromfile(base + ec.ToExt(i), dtype=np.uint8) == want[i]).all()
    assert not os.path.exists(base + ec.ToExt(7))
    vif = read_vif(base + ".vif")
    assert (vif["ds"], vif["ps"], vif["datFileSize"]) == (5, 2, len(dat))

    json.dump({"version": 3, "ecShardConfig": {"dataShards": 30, "parityShards": 9}}, open(base + ".vif", "w"))
    ec.VolumeEcShardsGenerate(base)
    assert os.path.exists(base + ec.ToExt(13)) and read_vif(base + ".vif")["ds"] == 10


def test_read_ec_needle_spanning_many_blocks(swec, oracle, tmp_path):
    """A 66 MiB record crosses 67 one-MiB blocks on all ten data shards: the interval list grows with the record."""
    ec = swec.erasure_coding
    rng = np.random.default_rng(3)
    size = 66 * MIB + 12345
    fixed = 16 + size + 4 + 8
    actual = fixed + (8 - fixed % 8)
    dat = np.concatenate([np.array([3, 0, 0, 0, 0, 0, 0, 0], dtype=np.uint8), rng.integers(0, 256, actual + 4096, dtype=np.uint8)])
    idx = rn._entry(77, 1, size)
    base, _ = lay_down_ec_volume(oracle, tmp_path, dat, idx)
    json.dump({"version": 3, "datFileSize": str(len(dat)), "ecShardConfig": {"dataShards": 10, "parityShards": 4}},
              open(base + ".vif", "w"))
    r = ec.ReadEcShardNeedles(base, [77], device=-1)[0]
    want = expected_record(dat, 8, size)
    assert r["status"] == "SWEC_OK" and r["n_bytes"] == len(want) and (r["bytes"] == want).all()


def test_scrub_local_finds_short_shards(swec, oracle, tmp_path):
    """ScrubLocal (ec_volume_scrub.go:27-118): a healthy volume walks clean; a truncated shard file is reported broken
    with the reference's wording; a shard that is not local is skipped."""
    ec = swec.erasure_coding
    base, dat, live = needle_volume(oracle, tmp_path, seed=61)
    n_entries = len(live)
    vol = ec.EcVolume(base, device=-1)
    assert vol.ScrubLocal() == (n_entries, [], [])
    vol.close()
    os.remove(base + ".ec09")                                             # not local: its chunks are skipped
    size0 = os.path.getsize(base + ".ec00")                               # two small rows: 2 MiB
    os.truncate(base + ".ec00", size0 // 2)                               # the second row's block of shard 0 is gone
    vol = ec.EcVolume(base, device=-1)
    count, broken, findings = vol.ScrubLocal()
    # like the reference, the walk stops at the first record that could not be read completely
    assert 0 < count <= n_entries and broken == [0]
    assert findings[0].startswith("local shard 0 for needle ") and f"is too short ({size0 // 2})" in findings[0]
    assert findings[-1].startswith("expected ") and " bytes for needle " in findings[-1]
    vol.close()
