"""Index files either side of the RS path (.idx → .ecx, .ecj fold, .ecx → .idx, FindDatFileSize):
host-only twins in libswec against the oracle's restatement, on the reference's fixture index
(tests/golden/fixtures/1.idx, 110 of its entries) and on synthetic indexes with overwrites/deletions."""
import os

import numpy as np
import pytest

from oracle import rs_numpy as rn

FIXTURES = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "fixtures")
FIXTURE_IDX = os.path.join(FIXTURES, "1.idx")
FIXTURE_DAT = os.path.join(FIXTURES, "1.dat")


def synthetic_idx(seed=4, n=500):
    rng = np.random.default_rng(seed)
    raw = b""
    offset = 1
    for _ in range(n):
        key = int(rng.integers(1, 200))
        kind = rng.integers(0, 10)
        size = int(rng.integers(1, 5000))
        if kind == 0:
            raw += rn._entry(key, 0, size)                 # zero offset ⇒ delete
        elif kind == 1:
            raw += rn._entry(key, offset, rn.TOMBSTONE)    # tombstone ⇒ delete
        else:
            raw += rn._entry(key, offset, size)
        offset += (size + 31) // 8
    return raw


@pytest.mark.parametrize("source", ["fixture", "synthetic"])
def test_ecx_from_idx_and_journal_fold(swec, tmp_path, source):
    ec = swec.erasure_coding
    if source == "fixture":
        idx = open(FIXTURE_IDX, "rb").read()
    else:
        idx = synthetic_idx()
    base = str(tmp_path / "1")
    open(base + ".idx", "wb").write(idx)
    ec.WriteSortedFileFromIdx(base, ".ecx")
    ecx = open(base + ".ecx", "rb").read()
    assert ecx == rn.sorted_ecx_from_idx(idx)
    keys = [k for k, _, _ in rn._entries(ecx)]
    assert keys == sorted(set(keys)) and len(keys) > 10
    assert ec.HasLiveNeedles(base)

    # journal some deletions (one unknown id, one duplicate), fold them in
    victims = [keys[0], keys[len(keys) // 2], keys[-1], keys[len(keys) // 2], 0xDEADBEEF]
    ecj = b"".join(v.to_bytes(8, "big") for v in victims)
    open(base + ".ecj", "wb").write(ecj)
    ec.WriteIdxFileFromEcIndex(base)                       # ec.decode side: .ecx + .ecj → .idx
    assert open(base + ".idx", "rb").read() == rn.idx_from_ec_index(ecx, ecj)
    ec.RebuildEcxFile(base)
    folded = open(base + ".ecx", "rb").read()
    assert folded == rn.fold_ecj_into_ecx(ecx, ecj)
    assert not os.path.exists(base + ".ecj")
    assert sum(1 for _, _, s in rn._entries(folded) if s < 0) == 3
    ec.RebuildEcxFile(base)                                # no journal: no-op
    assert open(base + ".ecx", "rb").read() == folded

    # everything deleted ⇒ no live needles (issue 7748 path)
    open(base + ".ecj", "wb").write(b"".join(k.to_bytes(8, "big") for k in keys))
    ec.RebuildEcxFile(base)
    assert not ec.HasLiveNeedles(base)


def test_find_dat_file_size_on_fixture_volume(swec, oracle, tmp_path):
    """FindDatFileSize reads the needle version from the superblock at the start of .ec00 and returns the
    end of the last live needle — for the reference's fixture volume that is the .dat size itself."""
    ec = swec.erasure_coding
    dat = np.fromfile(FIXTURE_DAT, dtype=np.uint8)
    base = str(tmp_path / "1")
    open(base + ".idx", "wb").write(open(FIXTURE_IDX, "rb").read())
    ec.WriteSortedFileFromIdx(base, ".ecx")
    shards = oracle.encode_dat_image(dat, buffer_size=50, large=10000, small=100)
    shards[0].tofile(base + ".ec00")
    version = int(dat[0])
    assert version in (1, 2, 3)
    want = rn.find_dat_file_size(open(base + ".ecx", "rb").read(), version)
    got = ec.FindDatFileSize(base, base)
    assert got == want and got <= len(dat) and got > len(dat) - 64 * 1024
    # every live needle of the fixture lies inside the volume and is addressable through LocateData
    for key, offset, size in rn._entries(open(base + ".ecx", "rb").read()):
        ivs = ec.LocateData(10000, 100, len(dat) // 10, offset * 8, 16 + size)
        assert sum(iv[2] for iv in ivs) == 16 + size


def test_index_errors(swec, tmp_path):
    ec = swec.erasure_coding
    with pytest.raises(swec.SwecError) as e:
        ec.WriteSortedFileFromIdx(str(tmp_path / "nope"), ".ecx")
    assert e.value.name == "SWEC_ERR_IO"
    with pytest.raises(swec.SwecError):
        ec.FindDatFileSize(str(tmp_path / "nope"), str(tmp_path / "nope"))
    ec.RebuildEcxFile(str(tmp_path / "nope"))              # no .ecj ⇒ nil, like the reference


def test_index_conversions_fuzz_against_oracle(swec, tmp_path):
    """Random indexes (duplicate keys, zero offsets, tombstones, negative sizes, ragged tails) through .idx→.ecx,
    the .ecj fold and .ecx→.idx: product == oracle, byte for byte (hypothesis, derandomised)."""
    from hypothesis import HealthCheck, given, settings
    from hypothesis import strategies as st
    ec = swec.erasure_coding
    entry = st.tuples(st.integers(1, 40), st.sampled_from([0, 1, 2, 77, 1 << 20, (1 << 32) - 1]),
                      st.sampled_from([0, 1, 100, 4096, -1, -100, (1 << 31) - 1]))
    case = [0]

    @settings(max_examples=120, deadline=None, derandomize=True, suppress_health_check=list(HealthCheck))
    @given(entries=st.lists(entry, max_size=60), tail=st.integers(0, 15), journal=st.lists(st.integers(0, 45), max_size=12))
    def check(entries, tail, journal):
        case[0] += 1
        base = str(tmp_path / f"c{case[0]}")
        idx = b"".join(rn._entry(k, o, s) for k, o, s in entries) + bytes(tail)
        open(base + ".idx", "wb").write(idx)
        ec.WriteSortedFileFromIdx(base, ".ecx")
        ecx = open(base + ".ecx", "rb").read()
        assert ecx == rn.sorted_ecx_from_idx(idx[:len(idx) - tail] if tail else idx)
        assert ec.HasLiveNeedles(base) == any(s >= 0 for _, _, s in rn._entries(ecx))
        ecj = b"".join(j.to_bytes(8, "big") for j in journal)
        if journal:
            open(base + ".ecj", "wb").write(ecj)
        ec.WriteIdxFileFromEcIndex(base)
        assert open(base + ".idx", "rb").read() == rn.idx_from_ec_index(ecx, ecj)
        ec.RebuildEcxFile(base)
        assert open(base + ".ecx", "rb").read() == rn.fold_ecj_into_ecx(ecx, ecj)
        assert not os.path.exists(base + ".ecj")

    check()
