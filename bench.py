#!/usr/bin/env python
"""bench.py — RS(10,4) encode throughput of one (or N) B200 against the HBM roofline, with the
reference's CPU arithmetic timed beside it.

  python bench.py --gpus N --steps K --warmup W            our arm (one rank per GPU under torchrun)
  python bench.py --impl reference --gpus N ...            the reference's CPU implementation of the path

Workload (BASELINE.json configs[1]): RS(10,4) encode of one 30 GiB synthetic volume per GPU,
two-tier striping of encodeDatFile (3 large rows of 10×1 GiB), volume resident in HBM when the
timed region starts.  A step = one whole volume through swec_encode_volume_device.  Weak scaling:
every rank encodes its own volume (volume v → GPU v mod N), no collective on the data path.
`value` = total .dat bytes encoded by all ranks ÷ max-over-ranks device time (GB/s, 1e9).
`e2e` = the same encode through the reference-facing C-ABI call (Encoder.Encode = swec_encode) on
pinned HOST buffers, H2D of the 10 data shards and D2H of the 4 parity shards inside the timed region.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

GIB = 1 << 30
MIB = 1 << 20
SEED0 = 0x5EA3EED5F00DCAFE
METRIC = "rs10_4_encode_input_GBps"
UNIT = "GB/s"
DUMP_BYTES_PER_SHARD = 1 << 21      # --dump-outputs: 4 shards x 2 Mi positions as float32 = 32 MiB
DUMP_SEED = 0x5EED


def load_traffic(dat_size):
    """dram__bytes_read+write per launch from the committed ncu --set full capture (profiles/), scaled
    to this run's volume if it differs; None when no capture is on record."""
    try:
        with open(os.path.join(ROOT, "profiles", "ncu_traffic.json")) as f:
            t = json.load(f)
        return int((t["dram_bytes_read"] + t["dram_bytes_write"]) * (dat_size / t["dat_bytes"])), t["source"]
    except Exception:
        return None, None


def load_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            p = json.load(f)
        return float(p["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """SM clock, power and throttle reasons sampled DURING the timed region: NVML in-process every
    ~5 ms (the timed region of 10 steps lasts ~70 ms), falling back to nvidia-smi polling."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")
    BITS = {0x4: "sw_power_cap", 0x8: "hw_slowdown", 0x20: "sw_thermal_slowdown", 0x40: "hw_thermal_slowdown"}

    def __init__(self, index: int, uuid: str | None = None):
        self.index, self.uuid = index, uuid
        self.samples, self._stop, self._t = [], threading.Event(), None   # (sm_mhz, max_mhz, watts, {reasons})
        self.source = "nvml"
        try:
            import pynvml
            pynvml.nvmlInit()
            self._nv = pynvml
            self._h = None
            if uuid:
                try:
                    self._h = pynvml.nvmlDeviceGetHandleByUUID(("GPU-" + uuid).encode() if not uuid.startswith("GPU-") else uuid.encode())
                except Exception:
                    self._h = None
            if self._h is None:
                self._h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self._max = pynvml.nvmlDeviceGetMaxClockInfo(self._h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self._nv, self.source = None, "nvidia-smi"

    def _run(self):
        while not self._stop.is_set():
            try:
                if self._nv:
                    nv = self._nv
                    sm = nv.nvmlDeviceGetClockInfo(self._h, nv.NVML_CLOCK_SM)
                    mask = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self._h)
                    watts = nv.nvmlDeviceGetPowerUsage(self._h) / 1000.0
                    self.samples.append((sm, self._max, watts, {n for b, n in self.BITS.items() if mask & b}))
                    self._stop.wait(0.005)
                    continue
                out = subprocess.run(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                      "-i", str(self.index)], stdout=subprocess.PIPE, text=True, timeout=5).stdout
                f = [x.strip() for x in out.strip().split(",")]
                if len(f) >= 7:
                    names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
                    self.samples.append((int(float(f[0])), int(float(f[1])), float(f[2]),
                                         {n for n, v in zip(names, f[3:7]) if v.lower().startswith("active")}))
            except Exception:
                pass
            self._stop.wait(0.1)

    def __enter__(self):
        self._t = threading.Thread(target=self._run, daemon=True)
        self._t.start()
        return self

    def __exit__(self, *a):
        self._stop.set()
        self._t.join(timeout=6)

    def summary(self):
        sm = sorted(s[0] for s in self.samples)
        reasons = sorted(set().union(*[s[3] for s in self.samples])) if self.samples else []
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_min_mhz": sm[0] if sm else None,
                "sm_max_mhz": max((s[1] for s in self.samples), default=None),
                "power_w_max": round(max((s[2] for s in self.samples), default=0.0), 1),
                "reasons": reasons, "samples": len(self.samples), "source": self.source}


def _cpu_variants(seconds_each: float, threads: int):
    """Whole-box CPU throughput of the reference's arithmetic (input GB/s), best case for the CPU:
    NUMA-local per-thread buffers, pinned threads (oracle/cpu_baseline.c orc_cpu_bench).
      reference_c_kernel_*  the reference's own vendored SIMD kernel (oracle/_ref), 40 passes per
                            256 KiB batch exactly like code_some_slices / encodeDataOneBatch
      gfni_port_*           fused AVX-512/AVX2+GFNI kernel standing in for klauspost's GFNI path"""
    from oracle import pyoracle as po
    rows = po.build_matrix(10, 14)[10:]
    per_shard = 4 * MIB                       # per thread: 10 x 4 MiB in, 4 x 4 MiB out
    kinds = []
    if po.ref_available():
        kinds.append((0, "reference_c_kernel_" + po.ref_isa()))
    if po.gfni_level():
        kinds.append((1, "gfni_port_" + ("avx512" if po.gfni_level() == 2 else "avx2")))
    res, passes_used = {}, {}
    # hyper-threads do not always help a memory-bound loop: try all logical CPUs and one per core
    counts, _quota = _thread_counts(threads)
    for kind, name in kinds:
        for tc in counts:
            probe = po.cpu_bench(kind, rows, per_shard, tc, 2)
            if probe <= 0:
                continue
            passes = max(4, int(seconds_each / len(counts) * probe * 1e9 / (tc * 10 * per_shard)))
            got = round(po.cpu_bench(kind, rows, per_shard, tc, passes), 3)
            if got > res.get(name, (0, 0))[0]:
                res[name] = (got, tc)
                passes_used[name] = passes
    if not res:
        raise RuntimeError("no CPU baseline available (oracle/_ref missing and no GFNI)")
    return res, passes_used, per_shard


def cpu_baseline(seconds_target: float = 12.0, threads: int | None = None):
    threads = threads or os.cpu_count() or 1
    res, passes, per_shard = _cpu_variants(seconds_target / 2, threads)
    best = max(res, key=lambda k: res[k][0])
    return {"value": res[best][0], "unit": UNIT, "cores": res[best][1],
            "kind": "reference" if best.startswith("reference") else "port",
            "sample": f"{res[best][1]} pinned threads x 10x{per_shard // MIB} MiB NUMA-local data shards, "
                      f"{passes[best]} passes each (in-memory, no disk); best of {list(res)} x thread counts",
            "variants": {k: {"GBps": v[0], "threads": v[1]} for k, v in res.items()},
            "logical_cpus": threads, "cpu_quota_cores": _cpu_quota_cores(), "cpu_model": _cpu_model()}


def _cpu_quota_cores():
    """CPU time this container may actually use (cgroup v2 cpu.max / v1 cfs quota), in cores; None = unlimited.
    The GPU boxes report 128 logical CPUs but run under a 16-core quota — threads beyond it only throttle."""
    try:
        q, per = open("/sys/fs/cgroup/cpu.max").read().split()
        if q != "max":
            return max(1, int(round(int(q) / int(per))))
    except Exception:
        pass
    try:
        q = int(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read())
        per = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
        if q > 0:
            return max(1, int(round(q / per)))
    except Exception:
        pass
    return None


def _thread_counts(logical):
    quota = _cpu_quota_cores()
    cand = {logical, max(1, logical // 2)}
    if quota:
        cand |= {min(logical, quota), min(logical, 2 * quota)}
    return sorted(cand, reverse=True), quota


def _cpu_model():
    try:
        for line in open("/proc/cpuinfo"):
            if line.startswith("model name"):
                return line.split(":", 1)[1].strip()
    except Exception:
        pass
    return "unknown"


def run_reference(args):
    """--impl reference: the reference's CPU implementation of the path on all host threads, rank 0
    only.  A step = 8 passes of every thread over its own 10 x 4 MiB data shards (bounded sample of
    the 30 GiB-volume workload; in-memory, so this is the CPU arithmetic's best case)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle import pyoracle as po
    threads = os.cpu_count() or 1
    rows = po.build_matrix(10, 14)[10:]
    per_shard, passes_per_step = 4 * MIB, 8
    kinds = []
    if po.ref_available():
        kinds.append((0, "reference", "reference_c_kernel_" + po.ref_isa()))
    if po.gfni_level():
        kinds.append((1, "port", "gfni_port_" + ("avx512" if po.gfni_level() == 2 else "avx2")))
    if not kinds:
        print(json.dumps({"impl": "reference", "unavailable": "oracle/_ref not built and CPU has no GFNI"}))
        return
    variants = {}
    for kind, label, name in kinds:
        for tc in _thread_counts(threads)[0]:
            po.cpu_bench(kind, rows, per_shard, tc, max(1, args.warmup))      # untimed warm-up
            got = po.cpu_bench(kind, rows, per_shard, tc, args.steps * passes_per_step)
            if got > variants.get(name, (0, "", 0))[0]:
                variants[name] = (got, label, tc)
    name = max(variants, key=lambda k: variants[k][0])
    value, label, used = variants[name]
    step_bytes = used * passes_per_step * 10 * per_shard
    sample = (f"{used} pinned threads x {passes_per_step} passes over 10x{per_shard // MIB} MiB NUMA-local "
              f"data shards per step ({step_bytes / GIB:.1f} GiB of input per step), {name}")
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": round(value, 3), "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(step_bytes / (value * 1e9) * 1e3, 3),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
        # the same workload name and shape as our own arm's `config` (the arm is compared on it); what the CPU actually
        # ran per step — a bounded in-memory sample of that workload — is spelled out in `sample`
        "config": {"workload": f"RS(10,4) encode of one {args.volume_gib:g} GiB synthetic volume per GPU "
                               "(BASELINE configs[1]); 10x1 GiB large-block rows",
                   "residency": "host memory: every thread's data shards in its own NUMA-local buffers",
                   "dat_bytes_per_gpu": int(args.volume_gib * GIB), "volumes": args.gpus, "seed": hex(SEED0),
                   "sample": sample, "host": _cpu_model()},
        "cpu_baseline": {"value": round(value, 3), "unit": UNIT, "cores": used, "kind": label, "sample": sample,
                         "variants": {k: {"GBps": round(v[0], 3), "threads": v[2]} for k, v in variants.items()},
                         "logical_cpus": threads, "cpu_quota_cores": _cpu_quota_cores()},
        "e2e": {"value": round(value, 3), "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


def oracle_window_check(par, dat_size, shard, seed, offs=None):
    """Parity windows of one encoded volume against the CPU oracle: the data columns are regenerated on the
    CPU from the seeded generator through the two-tier layout of encodeDatFile, encoded by the oracle and
    compared with what the GPU wrote.  Returns the number of windows checked."""
    import numpy as np
    from oracle import pyoracle as po
    G = GIB
    nlarge = dat_size // (10 * G)
    offs = offs or sorted({0, max(0, shard - 4096), (shard // 2) & ~15})
    for off in offs:
        cols = []
        for i in range(10):
            if off < nlarge * G:
                src = (off // G) * 10 * G + i * G + off % G
            else:
                o2 = off - nlarge * G
                src = nlarge * 10 * G + (o2 // MIB) * 10 * MIB + i * MIB + o2 % MIB
            col = np.zeros(4096, dtype=np.uint8)
            have = max(0, min(4096, dat_size - src))
            if have:
                col[:have] = po.synth(src, have, seed)
            cols.append(col)
        want = po.encode(10, 4, cols)
        for p in range(4):
            assert (par[p][off:off + 4096].cpu().numpy() == want[p]).all(), "parity mismatch vs oracle"
    return len(offs)


def dump_outputs(out_dir, par, shard):
    """--dump-outputs: the four parity shards the last timed step wrote, as DIR/ec10.npy … ec13.npy (float32, one
    value per byte).  A shard longer than DUMP_BYTES_PER_SHARD is sampled at the same seeded, sorted positions on
    every run, so two builds given the same arguments can be compared output for output."""
    import numpy as np
    import torch
    os.makedirs(out_dir, exist_ok=True)
    if shard > DUMP_BYTES_PER_SHARD:
        pos = np.sort(np.random.default_rng(DUMP_SEED).choice(shard, DUMP_BYTES_PER_SHARD, replace=False))
    else:
        pos = np.arange(shard)
    idx = torch.from_numpy(pos).to(par[0].device)
    for p in range(4):
        np.save(os.path.join(out_dir, "ec%02d.npy" % (10 + p)), par[p][idx].float().cpu().numpy())


def whole_volume_check(L, local, par_ptrs, par, dat_size, shard, seed, stream):
    """Every byte of the four parity shards of one encoded volume against the CPU oracle: the device digests of the
    shards must equal the digests oracle/cpu_baseline.c::orc_volume_digests computes for the same seeded volume
    (columns regenerated from the generator through encodeDatFile's two-tier layout, encoded by the reference's own
    compiled C kernel when oracle/_ref is shipped, else the GFNI port).  Windows are compared byte for byte too, so a
    failure is localised.  Returns the description for config.check."""
    from oracle import pyoracle as po
    got = []
    for p in range(4):
        one = C.c_uint64(0)
        assert L.swec_digest_device(local, par_ptrs[p], shard, C.byref(one), stream) == 0
        got.append(one.value)
    nwin = oracle_window_check(par, dat_size, shard, seed)
    kind = po.best_cpu_kind()
    t0 = time.perf_counter()
    want = po.volume_digests(dat_size, seed, kind=kind)[10:]
    assert got == want, f"whole-volume parity digests differ from the CPU oracle: {got} vs {want}"
    return (f"whole volume: device digests of all 4 x {shard} B parity shards equal the CPU oracle's "
            f"({['reference C kernel (oracle/_ref)', 'GFNI port', 'scalar tables'][kind]}, "
            f"{time.perf_counter() - t0:.1f} s on the host cores); {nwin} windows byte-identical too")


def host_api_leg(L, enc, local, sizes=(256 * 1024, 1 << 20, 16 << 20), min_s=0.4):
    """The Encoder-level seam from HOST memory at the batch sizes the Go call sites use: 256 KiB per shard in
    encodeDataOneBatch (ec_encoder.go:248-278), 1 MiB in rebuildEcFiles (:340-376) — one synchronous swec_encode /
    swec_reconstruct call per batch, exactly what a cgo reedsolomon.Encoder does.  `pageable` = Go heap memory
    (bounces through the pinned ring, copies spread over the host-copy pool), `pinned` = the 14 slices of one
    swec_alloc_pinned_for_device allocation (DMA'd in place, one strided DMA each way).  Beside them one CPU thread
    of the reference arithmetic on the same buffers (GFNI port, or the reference C kernel without GFNI)."""
    import numpy as np
    from oracle import pyoracle as po
    rows = po.build_matrix(10, 14)[10:]
    kind = 1 if po.gfni_level() else 0
    if kind == 0 and not po.ref_available():
        return {"error": "no CPU arithmetic to compare with"}

    def rate(fn):
        fn()
        fn()
        t0, k = time.perf_counter(), 0
        while time.perf_counter() - t0 < min_s:
            fn()
            k += 1
        return k / (time.perf_counter() - t0)

    out = {"api": "swec_encode / swec_reconstruct(data_only) on host buffers, one synchronous call per batch",
           "cpu": "1 thread, " + ("GFNI port" if kind == 1 else "reference C kernel"), "sizes": {}}
    rng = np.random.default_rng(7)
    for n in sizes:
        res = {}
        page = [rng.integers(0, 256, n, dtype=np.uint8) for _ in range(10)] + [np.zeros(n, dtype=np.uint8) for _ in range(4)]
        arr_page = (C.c_void_p * 14)(*[a.ctypes.data for a in page])
        raw = L.swec_alloc_pinned_for_device(local, 14 * n)
        pinned = np.ctypeslib.as_array(C.cast(raw, C.POINTER(C.c_uint8)), shape=(14, n))
        for i in range(10):
            pinned[i][:] = page[i]
        arr_pin = (C.c_void_p * 14)(*[raw + i * n for i in range(14)])
        want = [np.zeros(n, dtype=np.uint8) for _ in range(4)]
        po.cpu_apply(kind, rows, page[:10], want, threads=1)
        for name, arr, bufs in (("pageable", arr_page, page), ("pinned", arr_pin, list(pinned))):
            def enc_call():
                assert L.swec_encode(enc._h, arr, n) == 0
            r = rate(enc_call)
            for p_ in range(4):
                assert np.array_equal(bufs[10 + p_], want[p_]), f"host-API parity mismatch ({name}, {n})"
            res[name + "_encode_GBps"] = round(r * 10 * n / 1e9, 2)
            res[name + "_encode_us_per_call"] = round(1e6 / r, 1)
            present = (C.c_uint8 * 14)(*([1] * 5 + [0] + [1] * 8))       # shard 5 lost: the degraded-read shape
            keep = bufs[5].copy()

            def rec_call():
                assert L.swec_reconstruct(enc._h, arr, present, n, 1) == 0
            bufs[5][:] = 0
            r2 = rate(rec_call)
            assert np.array_equal(bufs[5], keep), f"host-API reconstruct mismatch ({name}, {n})"
            res[name + "_reconstruct_data_GBps"] = round(r2 * 10 * n / 1e9, 2)
        outs = [np.zeros(n, dtype=np.uint8) for _ in range(4)]
        rc = rate(lambda: po.cpu_apply(kind, rows, page[:10], outs, threads=1))
        res["cpu_1thread_GBps"] = round(rc * 10 * n / 1e9, 2)
        L.swec_free_pinned(raw)
        out["sizes"][str(n)] = res
    out["check"] = "every timed configuration's parity (and the rebuilt shard) byte-identical to the CPU arithmetic"
    return out


def power_state(L, device):
    """(heat_ms, low_power) of the library's auto power policy on `device` (swec_debug_power_state)."""
    heat, lp = C.c_double(0), C.c_int(0)
    L.swec_debug_power_state(device, C.byref(heat), C.byref(lp))
    return heat.value, lp.value


def load_batch_golden(n_volumes, dat_size):
    """CPU-oracle digest of the first n volumes of the configs[3] batch (tests/golden/batch256.json, written by
    tests/golden/make_batch_golden.py: every volume regenerated, striped and encoded on the CPU)."""
    try:
        with open(os.path.join(ROOT, "tests", "golden", "batch256.json")) as f:
            g = json.load(f)
        if g["dat_bytes_per_volume"] == dat_size and g["seed0"] == hex(SEED0):
            return g["prefix_digests"].get(str(n_volumes)), g["cpu_kind"]
    except Exception:
        pass
    return None, None


def batch_leg(n_volumes, L, enc, dat, dat_size, par, shard, stream, local, rank, world, dist, barrier, warmup):
    """BASELINE configs[3]: a batch of independent volumes sharded round-robin over the GPUs (volume v on GPU
    v mod N), no data-path collective.  Per volume: regenerate the synthetic .dat in HBM (untimed), encode (timed
    with CUDA events on the launching stream), digest the four parity shards on the device (untimed).
    value = batch bytes / the slowest rank's summed encode time; `digest` combines the per-volume digests
    independently of placement, so runs at N = 1, 2, 4, 8 must print the same one — and it must equal the digest
    the CPU oracle computed for the same 256 seeded volumes (tests/golden/batch256.json).  Collective on every
    rank; returns the leg's dict on rank 0, None elsewhere."""
    import torch
    from seaweedfs_b200 import sharding
    par_ptrs = [p.data_ptr() for p in par]
    for _ in range(max(3, warmup)):
        enc.encode_volume_device(dat.data_ptr(), dat_size, par_ptrs, stream)
    barrier()
    launches0 = L.swec_kernel_launches()
    last = {}

    def encode_volume(v, seed):
        assert L.swec_synth_fill_device(local, dat.data_ptr(), 0, dat.numel(), seed, stream) == 0
        last["lp"] = last.get("lp", 0) + power_state(L, local)[1]
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        enc.encode_volume_device(dat.data_ptr(), dat_size, par_ptrs, stream)
        b.record()
        d, four = 0, []
        for p in range(4):
            one = C.c_uint64(0)
            assert L.swec_digest_device(local, par_ptrs[p], shard, C.byref(one), stream) == 0   # synchronises
            four.append(one.value)
            d = (d * 0x100000001B3 + one.value) & ((1 << 64) - 1)
        last["v"], last["seed"], last["four"] = v, seed, four
        return d, a.elapsed_time(b)

    device = torch.device("cuda", local)
    with ClockSampler(local, None) as clk:
        res = sharding.run_batch(n_volumes, encode_volume, dist=dist, device=device)
    encode_launches = len(sharding.volumes_for_rank(n_volumes, world, rank))
    barrier()
    if rank != 0:
        return None
    golden, golden_kind = load_batch_golden(n_volumes, dat_size)
    digest = "%016x" % res["digest"]
    if golden is not None:
        assert digest == golden, f"batch digest {digest} differs from the CPU oracle's {golden}"
        check = (f"checksum of the {n_volumes} per-volume parity digests equals the CPU oracle's for the same seeded "
                 f"volumes ({golden_kind}; tests/golden/batch256.json): every byte of all 4 parity shards of every volume")
    elif last:
        from oracle import pyoracle as po
        want = po.volume_digests(dat_size, last["seed"])[10:]
        assert last["four"] == want, "whole-volume parity digests of the last volume differ from the CPU oracle"
        check = (f"all 4 parity shards of rank 0's last volume (v={last['v']}) equal the CPU oracle's whole-volume "
                 "digests; digest = placement-independent checksum of per-volume device digests")
    else:
        check = None
    peak, peak_src = load_peaks()
    ms_max = res["ms_max"]
    per_volume_ms = ms_max / max(1, encode_launches)
    achieved = 1.4 * dat_size / (per_volume_ms / 1e3) / 1e9
    c = clk.summary()
    return {"volumes": n_volumes, "placement": "volume v on GPU v mod N (BASELINE configs[3])", "scaling": "strong",
            "value": round(n_volumes * dat_size / (ms_max / 1e3) / 1e9, 2), "unit": UNIT,
            "volumes_per_gpu": encode_launches, "ms_per_volume": round(per_volume_ms, 4),
            "per_rank_ms": [round(x, 3) for x in res["per_rank_ms"]],
            "roofline_frac": round(achieved / peak, 4), "digest": digest, "check": check,
            "rank0_launches_on_low_power_variant": last.get("lp", 0),
            "sm_mhz": c["sm_mhz"], "sm_mhz_min": c["sm_min_mhz"], "power_w_max": c["power_w_max"], "reasons": c["reasons"],
            "gpu_launches": int(L.swec_kernel_launches() - launches0)}


def run_batch(args, L, enc, dat, dat_size, par, shard, stream, local, rank, world, dist, barrier):
    """--batch-volumes N as the whole run: the batch leg printed as its own line."""
    leg = batch_leg(args.batch_volumes, L, enc, dat, dat_size, par, shard, stream, local, rank, world, dist, barrier,
                    args.warmup)
    if rank == 0:
        peak, peak_src = load_peaks()
        print(json.dumps({
            "metric": METRIC, "value": leg["value"], "unit": UNIT,
            "n_gpus": world, "steps": leg["volumes_per_gpu"], "warmup": max(3, args.warmup),
            "ms_per_step": leg["ms_per_volume"], "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "u8", "data": "synthetic",
            "config": {"workload": f"batch encode of {args.batch_volumes} x {args.volume_gib:g} GiB synthetic volumes, "
                                   "volume v on GPU v mod N (BASELINE configs[3]); HBM-resident, no collective",
                       "volumes": args.batch_volumes, "dat_bytes_per_volume": dat_size,
                       "l2": "every volume (30 GiB) far exceeds the 126 MB L2; no flush needed",
                       "seed": hex(SEED0), "check": leg["check"]},
            "digest": leg["digest"], "per_rank_ms": leg["per_rank_ms"],
            "roofline": {"bound": "hbm", "achieved": round(leg["roofline_frac"] * peak, 1), "peak": peak, "unit": "GB/s",
                         "frac": leg["roofline_frac"], "traffic": load_traffic(dat_size)[0],
                         "peak_source": peak_src, "kernel": "rs10x4_encode_blocked",
                         "algorithmic_bytes_per_launch": int(1.4 * dat_size), "kernel_ms": leg["ms_per_volume"]},
            "clocks": {"sm_mhz": leg["sm_mhz"], "sm_min_mhz": leg["sm_mhz_min"], "power_w_max": leg["power_w_max"],
                       "reasons": leg["reasons"]},
            "gpu_launches": leg["gpu_launches"],
        }))
    if dist:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="swec", choices=["swec", "reference"])
    ap.add_argument("--volume-gib", type=float, default=30.0, help="synthetic .dat size per GPU (GiB)")
    ap.add_argument("--e2e-gib", type=float, default=-1.0, help="host-buffer volume for the e2e leg (GiB); <0 = auto")
    ap.add_argument("--batch-volumes", type=int, default=0,
                    help="BASELINE configs[3]: encode this many volumes (volume v seeded SEED0+v, placed on rank "
                         "v mod N) and print the batch line with a placement-independent checksum of checksums")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-reconstruct", action="store_true")
    ap.add_argument("--no-sustained", action="store_true")
    ap.add_argument("--no-files", action="store_true")
    ap.add_argument("--no-variant", action="store_true", help="skip the 30,000 MiB + ragged leg")
    ap.add_argument("--no-host-api", action="store_true", help="skip the Encoder-level host-buffer leg")
    ap.add_argument("--batch-leg-volumes", type=int, default=256,
                    help="volumes of the configs[3] batch leg inside the default line (0 = skip)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write rank 0's parity shards of the last step to DIR/ec10.npy … "
                         "ec13.npy (float32, a fixed seeded sample of byte positions)")
    args = ap.parse_args()
    args.warmup = max(args.warmup, 3) if args.impl == "swec" else args.warmup
    if args.impl == "reference":
        return run_reference(args)

    import numpy as np
    import torch

    import seaweedfs_b200
    from seaweedfs_b200 import erasure_coding as ec

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device — the engine has no CPU path")
    # Placement: rank r drives the r-th GPU of the library's socket-interleaved order (0,4,1,5,… on this pool's boxes)
    # when the box shows more GPUs than ranks — N = 2 and 4 then use both sockets' memory controllers for the host-fed
    # e2e leg instead of crowding socket 0 (SCALE_r01: 4 GPUs of one socket share ~142 GB/s of H2D).
    rank_local = local
    placement = "cuda:%d (LOCAL_RANK)" % local
    if torch.cuda.device_count() > world and not os.environ.get("SWEC_BENCH_NO_SPREAD"):
        order = (C.c_int * 64)()
        cnt = C.c_int(0)
        if seaweedfs_b200.lib().swec_device_spread_order(order, 64, C.byref(cnt)) == 0 and cnt.value > local:
            local = int(order[local])
            placement = "cuda:%d = entry %d of swec_device_spread_order %s" % (local, rank_local, list(order[:cnt.value]))
    torch.cuda.set_device(local)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    def barrier():
        torch.cuda.synchronize()
        if dist:
            dist.barrier()
        torch.cuda.synchronize()

    L = seaweedfs_b200.lib()
    enc = ec.Encoder(10, 4, device=local)
    stream = torch.cuda.current_stream().cuda_stream
    dat_size = int(args.volume_gib * GIB)
    shard = ec.expected_shard_size(dat_size)
    dat = torch.empty(dat_size + (-dat_size) % 8, dtype=torch.uint8, device="cuda")
    par = [torch.empty(shard, dtype=torch.uint8, device="cuda") for _ in range(4)]
    par_ptrs = [p.data_ptr() for p in par]
    # volume v = rank (round-robin v mod N with one volume per GPU in flight), seeded SEED0 + v
    assert L.swec_synth_fill_device(local, dat.data_ptr(), 0, dat.numel(), SEED0 + rank, stream) == 0

    if args.batch_volumes > 0:
        return run_batch(args, L, enc, dat, dat_size, par, shard, stream, local, rank, world, dist, barrier)

    # Wake-up: from a cold process the first ~8 launches of ANY kernel run on clocks still ramping up from idle
    # (profiles/r01z_warmup_ramp_probe.jsonl: 7.9 -> 7.0 ms over ~70 ms).  Twenty digest passes over the volume
    # (a measurement kernel, ~120 ms of HBM reads, nothing of the path under test) take the GPU out of idle so
    # that the W warm-up steps of each leg do what warm-up is for.  Every leg keeps its own W untimed steps and
    # exactly K timed ones; the `sustained` leg below shows what happens when the boost window is over.
    wake = C.c_uint64(0)
    for _ in range(20):
        assert L.swec_digest_device(local, dat.data_ptr(), dat_size, C.byref(wake), stream) == 0
    # ---- reconstruct, shards 0-3 erased (worst case, BASELINE configs[2]); untimed for `value` --------
    recon = None
    if not args.no_reconstruct:
        S = shard & ~15
        d_ptrs = [dat.data_ptr() + i * S for i in range(10)]        # the image viewed as 10 flat data shards
        enc.encode_device(d_ptrs, par_ptrs, S, stream)              # parity consistent with that view
        scratch = [torch.empty(S, dtype=torch.uint8, device="cuda") for _ in range(4)]
        ptrs = [t.data_ptr() for t in scratch] + d_ptrs[4:] + par_ptrs
        present = [0, 0, 0, 0] + [1] * 10
        for _ in range(args.warmup):                                # first call compiles the decode kernel
            enc.reconstruct_device(ptrs, present, S, False, stream)
        barrier()
        r0, r1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        r0.record()
        for _ in range(args.steps):
            enc.reconstruct_device(ptrs, present, S, False, stream)
        r1.record()
        barrier()
        rt = torch.tensor([r0.elapsed_time(r1)], dtype=torch.float64, device="cuda")
        if dist:
            dist.all_reduce(rt, op=dist.ReduceOp.MAX)
        rms = float(rt.item()) / args.steps
        ok = True
        for i in range(4):
            a, b = C.c_uint64(0), C.c_uint64(0)
            assert L.swec_digest_device(local, scratch[i].data_ptr(), S, C.byref(a), stream) == 0
            assert L.swec_digest_device(local, d_ptrs[i], S, C.byref(b), stream) == 0
            ok = ok and a.value == b.value
        assert ok, "reconstructed shards differ from the originals"
        # one lost shard (what ec.rebuild meets after a single disk died, and every degraded read behind it): the
        # compiled-in single-loss kernel, 10 streams read, 1 written
        one_ptrs = [scratch[0].data_ptr() if i == 5 else (d_ptrs[i] if i < 10 else par_ptrs[i - 10]) for i in range(14)]
        one_present = [0 if i == 5 else 1 for i in range(14)]
        for _ in range(args.warmup):
            enc.reconstruct_device(one_ptrs, one_present, S, False, stream)
        barrier()
        o0, o1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        o0.record()
        for _ in range(args.steps):
            enc.reconstruct_device(one_ptrs, one_present, S, False, stream)
        o1.record()
        barrier()
        ot = torch.tensor([o0.elapsed_time(o1)], dtype=torch.float64, device="cuda")
        if dist:
            dist.all_reduce(ot, op=dist.ReduceOp.MAX)
        oms = float(ot.item()) / args.steps
        a, b = C.c_uint64(0), C.c_uint64(0)
        assert L.swec_digest_device(local, scratch[0].data_ptr(), S, C.byref(a), stream) == 0
        assert L.swec_digest_device(local, d_ptrs[5], S, C.byref(b), stream) == 0
        assert a.value == b.value, "single-loss reconstruct differs from the original shard"
        nvrtc, hits, aot_n, aot_l = C.c_uint64(0), C.c_uint64(0), C.c_int(0), C.c_uint64(0)
        L.swec_jit_stats(C.byref(nvrtc), C.byref(hits), C.byref(aot_n), C.byref(aot_l))
        peak, _ = load_peaks()
        recon = {"value": round(world * 10 * S / (rms / 1e3) / 1e9, 2), "unit": UNIT, "ms_per_step": round(rms, 4),
                 "erased": [0, 1, 2, 3], "shard_bytes": S,
                 "roofline_frac": round(14 * S / (rms / 1e3) / 1e9 / peak, 4),
                 "launches_per_step": 1,
                 "check": "device digests of the 4 rebuilt shards equal the originals",
                 "single_loss": {"erased": [5], "ms_per_step": round(oms, 4),
                                 "value": round(world * 10 * S / (oms / 1e3) / 1e9, 2), "unit": UNIT,
                                 "roofline_frac": round(11 * S / (oms / 1e3) / 1e9 / peak, 4),
                                 "algorithmic_bytes_per_launch": 11 * S,
                                 "check": "device digest of the rebuilt shard equals the original"},
                 "kernel_source": {"compiled_in_matrices": aot_n.value, "compiled_in_launches": aot_l.value,
                                   "nvrtc_compiles": nvrtc.value, "disk_cache_hits": hits.value}}
        del scratch

    def step():
        enc.encode_volume_device(dat.data_ptr(), dat_size, par_ptrs, stream)

    for _ in range(args.warmup):
        step()
    barrier()
    launches0 = L.swec_kernel_launches()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps + 1)]
    try:
        gpu_uuid = str(torch.cuda.get_device_properties(local).uuid)
    except Exception:
        gpu_uuid = None
    with ClockSampler(local, gpu_uuid) as clk:
        ev[0].record()
        for i in range(args.steps):
            step()
            ev[i + 1].record()
        barrier()
    launches = L.swec_kernel_launches() - launches0
    ms_total = ev[0].elapsed_time(ev[-1])
    per_step = [ev[i].elapsed_time(ev[i + 1]) for i in range(args.steps)]
    t = torch.tensor([ms_total], dtype=torch.float64, device="cuda")
    if dist:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_max = float(t.item())
    value = world * args.steps * dat_size / (ms_max / 1e3) / 1e9
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, par, shard)

    # correctness outside the timed region: spot-check the parity against the oracle (rank 0)
    checked = None
    if rank == 0:
        checked = whole_volume_check(L, local, par_ptrs, par, dat_size, shard, SEED0 + rank, stream)

    # ---- BASELINE.md C2's variant: the 30,000 MiB default volume-size limit plus a ragged tail = 2 large rows
    # (BLOCKED launch), 952 full small rows (second BLOCKED launch) and one zero-padded tail row (third launch)
    variant = None
    if not args.no_variant and dat_size >= 30000 * MIB + 123_457:
        vsize = 30000 * MIB + 123_457
        vshard = ec.expected_shard_size(vsize)

        def vstep():
            enc.encode_volume_device(dat.data_ptr(), vsize, par_ptrs, stream)
        for _ in range(args.warmup):
            vstep()
        barrier()
        vl0 = L.swec_kernel_launches()
        v0, v1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        v0.record()
        for _ in range(args.steps):
            vstep()
        v1.record()
        barrier()
        vt = torch.tensor([v0.elapsed_time(v1)], dtype=torch.float64, device="cuda")
        if dist:
            dist.all_reduce(vt, op=dist.ReduceOp.MAX)
        vms = float(vt.item()) / args.steps
        vcheck = whole_volume_check(L, local, par_ptrs, par, vsize, vshard, SEED0 + rank, stream) if rank == 0 else None
        variant = {"dat_bytes": vsize, "rows": "2 large (10x1 GiB) + 952 small (10x1 MiB) + 1 zero-padded tail row",
                   "value": round(world * vsize / (vms / 1e3) / 1e9, 2), "unit": UNIT, "ms_per_step": round(vms, 4),
                   "steps": args.steps, "launches_per_step": (L.swec_kernel_launches() - vl0) // args.steps,
                   "roofline_frac": round((vsize + 4 * vshard) / (vms / 1e3) / 1e9 / load_peaks()[0], 4),
                   "check": vcheck}

    # ---- BASELINE configs[3]: the 256-volume batch, volume v on GPU v mod N (strong scaling inside this leg)
    batch = None
    if args.batch_leg_volumes > 0:
        batch = batch_leg(args.batch_leg_volumes, L, enc, dat, dat_size, par, shard, stream, local, rank, world, dist,
                          barrier, args.warmup)
        # the legs below expect the bench volume back in HBM
        assert L.swec_synth_fill_device(local, dat.data_ptr(), 0, dat.numel(), SEED0 + rank, stream) == 0
        step()
        torch.cuda.synchronize()


    # ---- the same step sustained: 100 more back-to-back volumes.  The timed region above is a burst (K steps
    # after W warm-ups, GPU at boost clocks); a B200 that keeps encoding drops its SM clock within ~0.3 s and
    # reaches its power cap within ~1 s (profiles/r01z_xt_variant_timeline.jsonl) — reported, not hidden.
    sustained = None
    if not args.no_sustained:
        n_sus = 100
        sev = [torch.cuda.Event(enable_timing=True) for _ in range(n_sus + 1)]
        with ClockSampler(local, gpu_uuid) as sclk:
            sev[0].record()
            lp_steps = []
            for i in range(n_sus):
                lp_steps.append(power_state(L, local)[1])          # which variant this launch is about to take
                step()
                sev[i + 1].record()
            barrier()
        sms = [sev[i].elapsed_time(sev[i + 1]) for i in range(n_sus)]
        tail = sum(sms[n_sus // 2:]) / (n_sus - n_sus // 2)
        st = torch.tensor([tail], dtype=torch.float64, device="cuda")
        if dist:
            dist.all_reduce(st, op=dist.ReduceOp.MAX)
        tail = float(st.item())
        sc = sclk.summary()
        sustained = {"steps": n_sus, "ms_per_step_last_half": round(tail, 4),
                     "ms_every_10th_step": [round(x, 3) for x in sms[::10]], "ms_min": round(min(sms), 4),
                     "value": round(world * dat_size / (tail / 1e3) / 1e9, 2), "unit": UNIT,
                     "roofline_frac": round(1.4 * dat_size / (tail / 1e3) / 1e9 / load_peaks()[0], 4),
                     "sm_mhz_min": sc["sm_min_mhz"], "power_w_max": sc["power_w_max"], "reasons": sc["reasons"],
                     "power_mode": "auto: boost-clock kernel variant until the Horner kernels own > 45 % of the last "
                                   "second, the low-power variant from then on",
                     "low_power_variant_from_step": (lp_steps.index(1) if 1 in lp_steps else None),
                     "heat_ms_at_end": round(power_state(L, local)[0], 1)}
    # ---- e2e leg: Encoder.Encode on pinned host buffers (H2D + kernel + D2H timed) -----------------
    e2e = None
    if not args.no_e2e:
        avail = 0
        try:
            for line in open("/proc/meminfo"):
                if line.startswith("MemAvailable"):
                    avail = int(line.split()[1]) * 1024
        except Exception:
            pass
        e2e_gib = args.e2e_gib if args.e2e_gib > 0 else min(args.volume_gib, max(1.0, avail / world * 0.25 / GIB / 1.4))
        n = int(e2e_gib * GIB / 10) & ~4095                     # bytes per shard
        raw = L.swec_alloc_pinned_for_device(local, 14 * n)
        if raw:
            bufs = [raw + i * n for i in range(14)]
            # fill the host data shards from the device generator (not timed)
            host = torch.from_numpy(np.ctypeslib.as_array(C.cast(raw, C.POINTER(C.c_uint8)), shape=(14 * n,)))
            for i in range(10):
                host[i * n:(i + 1) * n].copy_(dat[i * n:(i + 1) * n])
            torch.cuda.synchronize()
            shards_arr = (C.c_void_p * 14)(*bufs)
            e2e_steps = max(2, min(args.steps, 5))
            # the bound of this leg: what one H2D DMA stream reaches from the same pinned buffer (no D2H
            # running, so an upper bound — the parity going back shares the link's control traffic)
            probe_bytes = min(10 * n, 8 * GIB)
            pe0, pe1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            dat[:probe_bytes].copy_(host[:probe_bytes], non_blocking=True)
            torch.cuda.synchronize()
            pe0.record()
            dat[:probe_bytes].copy_(host[:probe_bytes], non_blocking=True)
            pe1.record()
            torch.cuda.synchronize()
            h2d_peak = probe_bytes / (pe0.elapsed_time(pe1) / 1e3) / 1e9
            # (host[:10n] was filled from dat[:10n], so the probe rewrote HBM with the bytes it already held)
            for _ in range(2):
                assert L.swec_encode(enc._h, shards_arr, n) == 0
            barrier()
            t0 = time.perf_counter()
            for _ in range(e2e_steps):
                assert L.swec_encode(enc._h, shards_arr, n) == 0
            torch.cuda.synchronize()
            dt = time.perf_counter() - t0
            tt = torch.tensor([dt], dtype=torch.float64, device="cuda")
            if dist:
                dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            dt = float(tt.item())
            e2e_check = None
            if rank == 0:
                # Whole-volume check outside the timed region: recompute all four parity shards of the
                # host volume with the reference's own compiled C kernel (oracle/_ref; the GFNI port if
                # that is not shipped) on every host core and compare every byte the GPU path wrote.
                from oracle import pyoracle as po
                hnp = host.numpy()
                kind = 0 if po.ref_available() else 1
                rows = po.build_matrix(10, 14)[10:]
                cpu_par = [np.empty(n, dtype=np.uint8) for _ in range(4)]
                po.cpu_apply(kind, rows, [hnp[i * n:(i + 1) * n] for i in range(10)], cpu_par, threads=os.cpu_count() or 1)
                for p_ in range(4):
                    assert np.array_equal(hnp[(10 + p_) * n:(11 + p_) * n], cpu_par[p_]), "e2e parity mismatch vs CPU"
                del cpu_par
                # ... and the device-resident kernel against that now CPU-verified parity, whole volume:
                # `par` still holds encode_device() of the same 10 flat shards (reconstruct leg above)
                if recon is not None and n == (shard & ~15):
                    enc.encode_device([dat.data_ptr() + i * n for i in range(10)], par_ptrs, n, stream)   # flat view again
                    torch.cuda.synchronize()
                    for p_ in range(4):
                        assert torch.equal(par[p_][:n], host[(10 + p_) * n:(11 + p_) * n].cuda()), "device parity mismatch"
                    device_full = True
                else:
                    device_full = False
                e2e_check = (f"all 4 x {n} B host parity shards byte-identical to the "
                             f"{'reference C kernel (oracle/_ref)' if kind == 0 else 'GFNI port'} on the same host data"
                             + ("; device-resident encode of the same shards identical too" if device_full else ""))
            e2e = {"value": round(world * e2e_steps * 10 * n / dt / 1e9, 3), "unit": UNIT,
                   "h2d_bytes_per_step": 10 * n, "d2h_bytes_per_step": 4 * n, "steps": e2e_steps,
                   "api": "swec_encode (Encoder.Encode) on pinned host shards", "volume_gib": round(10 * n / GIB, 3),
                   "roofline": {"bound": "pcie_h2d", "achieved": round(e2e_steps * 10 * n / dt / 1e9, 2),
                                "peak": round(h2d_peak, 2), "unit": "GB/s per GPU",
                                "frac": round(e2e_steps * 10 * n / dt / 1e9 / h2d_peak, 4),
                                "peak_source": "H2D-only DMA of the same pinned buffer, timed in this run",
                                "host_ceiling": "with several GPUs the bound is the socket, not the link: plain cudaMemcpy in "
                                                "both directions at once tops out at ~95 + 95 GB/s per socket on this pool's "
                                                "hosts (profiles/r02d_pcie_probe_thp.jsonl: 23.7 GB/s per direction per GPU with 4 "
                                                "GPUs on a socket); e2e moves 1.4 B of DMA per input byte, so ~136-142 GB/s of "
                                                "input per socket is the ceiling (N=8: ~283)"},
                   "check": e2e_check}
            L.swec_free_pinned(raw)
    barrier()

    host_api = None
    if rank == 0 and world == 1 and not args.no_host_api:
        host_api = host_api_leg(L, enc, local)

    # ---- file level (BASELINE configs[4] in miniature), rank 0 at N=1: WriteEcFiles / RebuildEcFiles on an 8 GiB
    # .dat in RAM-backed storage next to the reference-shaped serial walk with SIMD Encode; shards byte-compared
    files = None
    if rank == 0 and world == 1 and not args.no_files:
        try:
            import shutil
            import types
            sys.path.insert(0, os.path.join(ROOT, "scripts"))
            import bench_files
            fdir = next((d_ for d_ in ("/dev/shm", "/tmp") if os.path.isdir(d_) and shutil.disk_usage(d_).free > (28 << 30)), None)
            if fdir:
                del dat, par
                torch.cuda.empty_cache()
                files = bench_files.run(types.SimpleNamespace(dir=fdir, gib=8.0, cpu_gib=1.0))
        except Exception as ex:                                  # noqa: BLE001
            files = {"error": repr(ex)}

    if rank == 0:
        peak, peak_src = load_peaks()
        ms_step = ms_max / args.steps
        # dominant kernel: rs10x4_encode_blocked — one launch per step covers the whole volume
        kernel_ms = ms_step                                      # mean of the K timed steps (max over ranks)
        algo_bytes = 1.4 * dat_size                              # read 10 streams once, write 4 (SURVEY §8d)
        achieved = algo_bytes / (kernel_ms / 1e3) / 1e9
        clocks = clk.summary()
        traffic, traffic_src = load_traffic(dat_size)
        out = {
            "metric": METRIC, "value": round(value, 2), "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": round(ms_step, 4), "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "u8", "data": "synthetic",
            "config": {"workload": f"RS(10,4) encode of one {args.volume_gib:g} GiB synthetic volume per GPU "
                                   "(BASELINE configs[1]); 10x1 GiB large-block rows",
                       "residency": "volume resident in HBM when the timed region starts",
                       "dat_bytes_per_gpu": dat_size, "shard_bytes": shard, "volumes": world, "rank0_device": placement,
                       "l2": "inputs (30 GiB) far exceed the 126 MB L2; no flush needed",
                       "wake_up": "20 digest passes over the volume (~120 ms) before the legs: the GPU leaves idle clocks",
                       "seed": hex(SEED0), "check": checked},
            "roofline": {"bound": "hbm", "achieved": round(achieved, 1), "peak": peak, "unit": "GB/s",
                         "frac": round(achieved / peak, 4), "traffic": traffic, "traffic_source": traffic_src,
                         "peak_source": peak_src,
                         "kernel": "rs10x4_encode_blocked", "algorithmic_bytes_per_launch": int(algo_bytes),
                         "kernel_ms": round(kernel_ms, 4),
                         "kernel_ms_median_step_rank0": round(sorted(per_step)[len(per_step) // 2], 4),
                         "regime": "burst: K steps after W warm-ups at boost clocks; see `sustained` and `batch` for "
                                   "the power-capped regime"},
            "clocks": clocks, "gpu_launches": int(launches), "e2e": e2e, "reconstruct": recon, "sustained": sustained,
            "variant_30000MiB": variant, "batch": batch, "host_api": host_api, "file_level": files,
        }
        if world == 1 and not args.no_cpu_baseline:
            try:
                out["cpu_baseline"] = cpu_baseline()
            except Exception as ex:                              # noqa: BLE001
                out["cpu_baseline"] = {"error": str(ex)}
        print(json.dumps(out))
    if dist:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
