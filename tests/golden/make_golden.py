#!/usr/bin/env python
"""tests/golden/make_golden.py — regenerates tests/golden/kat.json and tests/golden/fixtures/ from a SeaweedFS
source tree:  python tests/golden/make_golden.py <seaweedfs-source-tree>
What it writes is committed; the tests read only that, never the source tree.

Sources (paths relative to the source tree; "rse/" = seaweed-volume/vendor/reed-solomon-erasure/):
  K1 log table          rse/src/galois_8.rs:339-364   (parsed from the Rust test source)
  K2 scalar mul/exp     rse/src/galois_8.rs:483-485,549-551
  K3 slice vectors      rse/src/galois_8.rs:487-547   (parsed)
  K4 matrix inverse     rse/src/matrix.rs:382-413
  K5 RS(5,5) encode     rse/src/tests/mod.rs:851-893
  K6 C kernel parity    parity of seeded inputs (pyoracle.synth) through rse/simd_c/reedsolomon.c
                        (oracle/_ref/libref_rs_*.so), as sha256 per parity shard
  K7 LocateData         weed/storage/erasure_coding/ec_test.go:199-274
  K8 fixture digests    fixtures/1.dat (below) encoded by the REFERENCE'S OWN compiled C
                        kernel (rse/simd_c/reedsolomon.c → oracle/_ref/libref_rs_*.so) driven like
                        code_some_slices (rse/src/core.rs:484-512) over the shard layout of
                        encodeDatFile (ec_encoder.go:280-321), production and test block sizes
  K9 patterns           weed/storage/store_ec_recovery_test.go:208-213, ec_encoder.rs:666-674 (inputs;
                        parity bytes computed through the reference kernel as for K8)

fixtures/ (binary test data of the source tree, shrunk to stay small):
  1.dat, 1.idx          weed/storage/erasure_coding/1.{dat,idx} cut down to its first FIXTURE_NEEDLES needle
                        records of at most 64 KiB (this leaves out needle 74, 2 MB), records byte-identical,
                        re-addressed back to back behind the original superblock; .idx = their entries re-addressed
  389_sample.ecx        ECX_SAMPLE entries of weed/storage/erasure_coding/test_files/389.ecx (485,098 entries):
                        the ids TestPositioning (ec_volume_test.go:14-58) looks up plus a seeded sample, in file order
  idx/                  the six files of weed/storage/idx/test_files/, verbatim (TestCheckIndexFile)
"""
import hashlib
import json
import os
import re
import shutil
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
GOLDEN = os.path.dirname(os.path.abspath(__file__))
FIXTURES = os.path.join(GOLDEN, "fixtures")
FIXTURE_NEEDLES = 110
ECX_SAMPLE = 2048
ECX_IDS = (0x0F0EDB92, 0x0EF7D7F8, 0x0F087622)      # TestPositioning's table and its third lookup
K6_SEED = 0x6B36
K6_SIZES = (1, 15, 64, 10_003, 300_000)

from oracle import pyoracle as po  # noqa: E402
from oracle import rs_numpy as rn  # noqa: E402


def ints(text):
    return [int(x, 0) for x in re.findall(r"0x[0-9a-fA-F]+|\d+", text)]


def write_fixtures(ref):
    ec_dir = os.path.join(ref, "weed", "storage", "erasure_coding")
    os.makedirs(os.path.join(FIXTURES, "idx"), exist_ok=True)
    dat = open(os.path.join(ec_dir, "1.dat"), "rb").read()
    idx = open(os.path.join(ec_dir, "1.idx"), "rb").read()
    version = dat[0]
    out_dat, moved = bytearray(dat[:8]), {}
    for _, offset, size in sorted(rn._entries(idx), key=lambda e: e[1]):     # records lie back to back
        n = rn.get_actual_size(size, version)
        if n > 64 * 1024:
            continue
        moved[offset] = len(out_dat) // 8
        out_dat += dat[offset * 8:offset * 8 + n]
        if len(moved) == FIXTURE_NEEDLES:
            break
    out_idx = b"".join(rn._entry(k, moved[o], s) for k, o, s in rn._entries(idx) if o in moved)
    open(os.path.join(FIXTURES, "1.dat"), "wb").write(bytes(out_dat))
    open(os.path.join(FIXTURES, "1.idx"), "wb").write(out_idx)

    ecx = open(os.path.join(ec_dir, "test_files", "389.ecx"), "rb").read()
    keys = np.frombuffer(ecx, dtype=">u8")[::2]
    must = [int(np.searchsorted(keys, k)) for k in ECX_IDS]
    assert all(keys[i] == k for i, k in zip(must, ECX_IDS))
    rest = np.setdiff1d(np.arange(len(keys)), must)
    pick = np.sort(np.concatenate([must, np.random.default_rng(389).choice(rest, ECX_SAMPLE - len(must), replace=False)]))
    open(os.path.join(FIXTURES, "389_sample.ecx"), "wb").write(b"".join(ecx[16 * i:16 * i + 16] for i in pick))

    idx_dir = os.path.join(ref, "weed", "storage", "idx", "test_files")
    for name in sorted(os.listdir(idx_dir)):
        shutil.copyfile(os.path.join(idx_dir, name), os.path.join(FIXTURES, "idx", name))


def main(ref):
    os.environ["REF"] = ref                     # oracle/Makefile builds oracle/_ref from this tree
    po.build(quiet=True)
    assert po.ref_available(), "oracle/_ref missing"
    write_fixtures(ref)
    rse = os.path.join(ref, "seaweed-volume", "vendor", "reed-solomon-erasure")
    g8 = open(rse + "/src/galois_8.rs").read()
    out = {}
    m = re.search(r"BACKBLAZE_LOG_TABLE: \[u8; 256\] = \[(.*?)\];", g8, re.S)
    body = re.sub(r"//.*", "", m.group(1))
    out["K1_log_table"] = ints(body)
    assert len(out["K1_log_table"]) == 256
    out["K2_mul"] = [[3, 4, 12], [7, 7, 21], [23, 45, 41]]
    out["K2_exp"] = [[2, 2, 4], [5, 20, 235], [13, 7, 43]]
    t = g8[g8.index("fn test_galois()"):g8.index("fn test_slice_add()")]
    arrays = [ints(a) for a in re.findall(r"= \[(.*?)\];", t, re.S)]
    assert len(arrays) == 5 and all(len(a) == 34 for a in arrays)
    out["K3"] = {"input": arrays[0], "mul_25": arrays[1], "then_xor_52": arrays[2],
                 "mul_177": arrays[3], "then_xor_117": arrays[4]}
    out["K4"] = {"m": [[56, 23, 98], [3, 100, 200], [45, 201, 123]],
                 "inv": [[175, 133, 33], [130, 13, 245], [112, 35, 126]],
                 "m5": [[1, 0, 0, 0, 0], [0, 1, 0, 0, 0], [0, 0, 0, 1, 0], [0, 0, 0, 0, 1], [7, 7, 6, 6, 1]],
                 "inv5": [[1, 0, 0, 0, 0], [0, 1, 0, 0, 0], [123, 123, 1, 122, 122], [0, 0, 1, 0, 0], [0, 0, 0, 1, 0]]}
    out["K5"] = {"data": [[0, 1], [4, 5], [2, 3], [6, 7], [8, 9]],
                 "parity": [[12, 13], [10, 11], [14, 15], [90, 91], [94, 95]]}
    out["K7"] = [
        {"args": [1 << 30, 1 << 20, 3221225472 - 1, 21479557912, 4194339],
         "intervals": [[4, 527128, 521448, False, 2], [5, 0, 1048576, False, 2], [6, 0, 1048576, False, 2],
                       [7, 0, 1048576, False, 2], [8, 0, 527163, False, 2]]},
        {"args": [1 << 30, 1 << 20, 3221225472 - 1, 30782909808, 112568],
         "intervals": [[8876, 912752, 112568, False, 2]]},
        {"args": [10000, 100, 10001, 100000, 1], "intervals": [[0, 0, 1, False, 1]]},
        {"args": [1 << 30, 1 << 20, 3 << 30, 20 << 30, 1024], "intervals": [[20, 0, 1024, True, 3]]},
    ]

    # K8 / K9 through the reference's own compiled kernel
    gen = rn.build_matrix(10, 14)

    def ref_parity(data):
        n = len(data[0])
        outs = [np.zeros(n, dtype=np.uint8) for _ in range(4)]
        po.cpu_apply(0, gen[10:], [np.ascontiguousarray(d) for d in data], outs, threads=1)
        return outs

    out["K6"] = {"seed": hex(K6_SEED), "parity_sha256": {}}
    for n in K6_SIZES:
        data = [po.synth(i * n, n, K6_SEED) for i in range(10)]
        out["K6"]["parity_sha256"][str(n)] = [hashlib.sha256(p.tobytes()).hexdigest() for p in ref_parity(data)]
    dat = np.fromfile(os.path.join(FIXTURES, "1.dat"), dtype=np.uint8)
    out["K8"] = {"dat_sha256": hashlib.sha256(dat.tobytes()).hexdigest(), "dat_size": int(dat.shape[0])}
    for label, (large, small) in {"production": (1 << 30, 1 << 20), "test": (10000, 100)}.items():
        shards = rn.encode_dat_image(dat, 10, 4, large, small)[:10]  # layout only
        shards += ref_parity(shards)                                  # arithmetic by the reference kernel
        out["K8"][label] = {"large": large, "small": small, "shard_size": int(shards[0].shape[0]),
                            "sha256": [hashlib.sha256(s.tobytes()).hexdigest() for s in shards]}
    n = 64
    pat_a = [np.full(n, (7 * i) & 255, dtype=np.uint8) for i in range(10)]
    pat_b = [((np.arange(n) + i) & 255).astype(np.uint8) for i in range(10)]
    out["K9"] = {"seven_i": [int(p[0]) for p in ref_parity(pat_a)],
                 "i_plus_j": [[int(p[j]) for p in ref_parity(pat_b)] for j in range(4)]}
    out["generator_rs10_4_parity_rows"] = gen[10:].tolist()
    with open(os.path.join(GOLDEN, "kat.json"), "w") as f:
        json.dump(out, f, indent=1)
    print("wrote kat.json")


if __name__ == "__main__":
    if len(sys.argv) != 2:
        sys.exit("usage: make_golden.py <seaweedfs-source-tree>")
    main(os.path.abspath(sys.argv[1]))
