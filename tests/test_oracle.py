"""The oracle pinned against the reference's own known-answer tests and fixtures (SURVEY §8c).
CPU only.  K-numbers refer to tests/golden/make_golden.py."""
import hashlib
import os

import numpy as np
import pytest

from oracle import rs_numpy as rn

FIXTURE_DAT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "fixtures", "1.dat")


def test_k1_log_table(kat, oracle):
    assert oracle.table("log").tolist() == kat["K1_log_table"]
    assert rn.LOG.tolist() == kat["K1_log_table"]


def test_k2_scalars(kat, oracle):
    L = oracle.lib()
    for a, b, r in kat["K2_mul"]:
        assert L.orc_mul(a, b) == r and rn.gf_mul(a, b) == r
    for a, n, r in kat["K2_exp"]:
        assert L.orc_exp(a, n) == r and rn.gf_exp(a, n) == r


def test_k3_slices(kat, oracle):
    L = oracle.lib()
    k3 = kat["K3"]
    x = np.array(k3["input"], dtype=np.uint8)
    for first, first_key, second, second_key in ((25, "mul_25", 52, "then_xor_52"), (177, "mul_177", 117, "then_xor_117")):
        out = np.zeros_like(x)
        L.orc_mul_slice(first, x.ctypes.data, out.ctypes.data, len(x))
        assert out.tolist() == k3[first_key]
        L.orc_mul_slice_xor(second, x.ctypes.data, out.ctypes.data, len(x))
        assert out.tolist() == k3[second_key]
        assert (rn.MUL[first][x] ^ rn.MUL[second][x]).tolist() == k3[second_key]


def test_k4_inverse(kat, oracle):
    for m, inv in ((kat["K4"]["m"], kat["K4"]["inv"]), (kat["K4"]["m5"], kat["K4"]["inv5"])):
        m = np.array(m, dtype=np.uint8)
        assert oracle.matrix_invert(m).tolist() == inv
        assert rn.mat_inv(m).tolist() == inv


def test_k5_encode_and_verify(kat, oracle):
    data = [np.array(d, dtype=np.uint8) for d in kat["K5"]["data"]]
    assert [p.tolist() for p in oracle.encode(5, 5, data)] == kat["K5"]["parity"]
    assert [p.tolist() for p in rn.encode(5, 5, data)] == kat["K5"]["parity"]
    shards = data + [np.array(p, dtype=np.uint8) for p in kat["K5"]["parity"]]
    ptrs = oracle._ptr_array(shards)
    assert oracle.lib().orc_verify(5, 5, ptrs, 2) == 1
    shards[8][0] += 1
    assert oracle.lib().orc_verify(5, 5, ptrs, 2) == 0


def test_generator_matrix(kat, oracle):
    g = oracle.build_matrix(10, 14)
    assert (g[:10] == np.eye(10, dtype=np.uint8)).all()
    assert g[10:].tolist() == kat["generator_rs10_4_parity_rows"]
    assert (rn.build_matrix(10, 14) == g).all()
    # "evaluate the interpolating polynomial at 10..13": data column [0..9] → parity [10..13]
    data = [np.array([i], dtype=np.uint8) for i in range(10)]
    assert [int(p[0]) for p in oracle.encode(10, 4, data)] == [10, 11, 12, 13]


def test_k6_reference_c_kernel_agrees(kat, oracle):
    """The parity the reference's compiled C kernel gave for seeded inputs (kat.json K6): the restatement, the GFNI
    port and, where oracle/_ref is built, the reference kernel itself all reproduce it."""
    g = oracle.build_matrix(10, 14)
    seed = int(kat["K6"]["seed"], 16)
    for n, want in kat["K6"]["parity_sha256"].items():
        n = int(n)
        ins = [oracle.synth(i * n, n, seed) for i in range(10)]
        got = {"oracle": oracle.encode(10, 4, ins)}
        for kind in ([1] if oracle.gfni_level() else []) + ([0] if oracle.ref_available() else []):
            got[kind] = [np.zeros(n, dtype=np.uint8) for _ in range(4)]
            oracle.cpu_apply(kind, g[10:], ins, got[kind], threads=3, batch=4096)
        for name, par in got.items():
            assert [hashlib.sha256(p.tobytes()).hexdigest() for p in par] == want, (name, n)


def test_k7_locate_data(kat, oracle):
    for case in kat["K7"]:
        want = [tuple(iv) for iv in case["intervals"]]
        assert oracle.locate_data(*case["args"]) == want
        assert rn.locate_data(*case["args"]) == want


def test_locate_data_boundary_sweep(oracle):
    # ec_test.go:259-274 (Issue 8179): every interval across the large→small boundary is non-empty
    large, small, shard = 10000, 100, 259092
    area = (shard // large) * 10 * large
    for off in range(area - 500, area + 500, 7):
        ivs = oracle.locate_data(large, small, shard, off, 200)
        assert ivs == rn.locate_data(large, small, shard, off, 200)
        assert all(iv[2] > 0 for iv in ivs) and sum(iv[2] for iv in ivs) == 200


def test_k8_fixture_digests(kat, oracle):
    dat = np.fromfile(FIXTURE_DAT, dtype=np.uint8)
    assert hashlib.sha256(dat.tobytes()).hexdigest() == kat["K8"]["dat_sha256"]
    for label, bufsz in (("production", 256 * 1024), ("test", 50)):
        g = kat["K8"][label]
        shards = oracle.encode_dat_image(dat, buffer_size=bufsz, large=g["large"], small=g["small"])
        assert [hashlib.sha256(s.tobytes()).hexdigest() for s in shards] == g["sha256"]
        # ec_test.go:49-101 validateFiles: every byte is where LocateData says it is
        for off, size in ((0, 1), (8, 5000), (len(dat) - 1000, 1000), (99000, 5000)):
            got = b""
            for iv in oracle.locate_data(g["large"], g["small"], len(dat) // 10, off, size):
                sid, soff = rn.interval_to_shard(iv, g["large"], g["small"])
                got += shards[sid][soff:soff + iv[2]].tobytes()
            assert got == dat[off:off + size].tobytes()
        back = oracle.write_dat_image(shards, len(dat), large=g["large"], small=g["small"])
        assert (back == dat).all()


def test_k9_patterns(kat, oracle):
    n = 64
    a = [np.full(n, (7 * i) & 255, dtype=np.uint8) for i in range(10)]
    assert [int(p[0]) for p in oracle.encode(10, 4, a)] == kat["K9"]["seven_i"]
    b = [((np.arange(n) + i) & 255).astype(np.uint8) for i in range(10)]
    par = oracle.encode(10, 4, b)
    assert [[int(p[j]) for p in par] for j in range(4)] == kat["K9"]["i_plus_j"]


@pytest.mark.parametrize("erased", [(5,), (0, 1, 2, 3), (10, 11, 12, 13), (0, 1, 10, 11), (3, 9, 12), (9, 13)])
def test_reconstruct_roundtrip(oracle, erased):
    rng = np.random.default_rng(len(erased))
    data = [rng.integers(0, 256, 1000, dtype=np.uint8) for _ in range(10)]
    full = data + oracle.encode(10, 4, data)
    holes = [None if i in erased else s for i, s in enumerate(full)]
    for impl in (oracle.reconstruct, rn.reconstruct):
        got = impl(10, 4, list(holes))
        assert all((g == f).all() for g, f in zip(got, full))
    got = oracle.reconstruct(10, 4, list(holes), data_only=True)
    assert all((got[i] == full[i]).all() for i in range(10))
    # the fused single-pass matrix gives the same bytes
    valid, missing, rows = rn.fused_reconstruct_rows(10, 4, [h is not None for h in holes])
    outs = rn.apply_rows(rows, [full[i] for i in valid])
    assert all((o == full[i]).all() for o, i in zip(outs, missing))


def test_too_few_shards(oracle):
    data = [np.zeros(8, dtype=np.uint8)] * 9 + [None] * 5
    with pytest.raises(ValueError):
        oracle.reconstruct(10, 4, data)


def test_expected_shard_size(oracle):
    G, M = 1 << 30, 1 << 20
    cases = {0: 0, 1: M, 10 * M: M, 10 * M + 1: 2 * M, 30 * G: 3 * G, 30000 * M: 2 * G + 952 * M,
             10 * G - 1: 1024 * M, 10 * G: G, 10 * G + 1: G + M}
    for dat, want in cases.items():
        assert oracle.expected_shard_size(dat) == want == rn.expected_shard_size(dat)


def test_file_level_oracle(oracle, tmp_path):
    rng = np.random.default_rng(3)
    dat = rng.integers(0, 256, 2_345_678, dtype=np.uint8)
    base = str(tmp_path / "7")
    dat.tofile(base + ".dat")
    assert oracle.generate_ec_files(base, 50, 10000, 100) == 0
    want = oracle.encode_dat_image(dat, buffer_size=50, large=10000, small=100)
    for i in range(14):
        assert (np.fromfile(base + ".ec%02d" % i, dtype=np.uint8) == want[i]).all()
    # the reference's rebuild loop needs 1 MiB-multiple shards (ec_encoder.go:351-353): use production sizes
    assert oracle.generate_ec_files(base) == 0
    keep = [np.fromfile(base + ".ec%02d" % i, dtype=np.uint8) for i in range(14)]
    for i in (0, 7, 11, 13):
        os.remove(base + ".ec%02d" % i)
    rc, ids = oracle.rebuild_ec_files(base)
    assert rc == 0 and ids == [0, 7, 11, 13]
    for i in range(14):
        assert (np.fromfile(base + ".ec%02d" % i, dtype=np.uint8) == keep[i]).all()


def test_synth_generators_agree(oracle):
    for off, n in ((0, 64), (5, 1000), (8 * 12345 + 3, 77)):
        assert (oracle.synth(off, n, 0x5EA3EED5F00DCAFE) == rn.synth(off, n, 0x5EA3EED5F00DCAFE)).all()


@pytest.mark.parametrize("size", [0, 13, 40 << 20, (2 * 40 + 30 << 20) + 12345, (10 << 20) + 8, (50 << 20) - 1])
def test_volume_digests_equal_digests_of_the_encoded_image(oracle, size):
    """orc_volume_digests (the whole-volume checker of the 30 GiB GPU runs: nothing held in memory, columns
    regenerated from the seeded generator through encodeDatFile's two-tier layout, ec_encoder.go:280-321) must give
    the digests of the shards orc_encode_dat_image writes for the same volume — for the reference's own C kernel,
    the GFNI port and the scalar tables alike."""
    MIB = 1 << 20
    dat = oracle.synth(0, size, 77)
    want = [oracle.np_digest(w) for w in oracle.encode_dat_image(dat, large=4 * MIB, small=MIB)]
    kinds = [2] + ([1] if oracle.gfni_level() else []) + ([0] if oracle.ref_available() else [])
    for kind in kinds:
        assert oracle.volume_digests(size, 77, large=4 * MIB, small=MIB, threads=3, kind=kind) == want, kind
