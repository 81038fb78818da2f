#!/usr/bin/env python3
"""bench.py -- benchmark of the B200 Paillier engine on the BASELINE.json configurations.

Headline ("step"): raw_encrypt of a batch of 2048-bit-key plaintexts followed by raw_decrypt of the resulting
ciphertexts (BASELINE.json configs[1]: 2048-bit key, batch 1M, bit-exact round trip).  `value` is encrypts/s of the
whole job with inputs resident in HBM; the decrypt leg of the same steps is reported under "decrypt".  `e2e` runs the
same step through the host-pointer C ABI with pinned host buffers at the same batch (H2D + kernels + D2H inside the
timed region), `e2e_python` through the Python-int API a phe user calls (list[int] in, list[int] out).

Extra keys of the same JSON line (each leg is outside the headline's timed region and has its own timing):
  config2_add_mul  configs[2]: 1M _raw_add and 1M _raw_mul (64-bit scalars; float-encoded and negative-scalar mixes)
  config3072       configs[3]: 3072-bit key, 4M rows sharded over the ranks (strong scaling), encrypt + decrypt, plus the
                   NCCL all-gather of the ciphertext shards timed separately
  multi_gpu_parity N > 1: every rank encrypts its shard of a seeded vector, the shards are all-gathered and rank 0 checks
                   the gathered rows against the GMP oracle
  federated        configs[4]: one round of the federated-learning example shape (rank 0, N = 1)
  reductions       EncryptedVector.sum / dot (fused kernels) against the launch chains they replace

  python bench.py [--gpus N] [--steps K] [--warmup W] [--batch B] [--impl reference] [--dump-outputs DIR]

Multi-GPU (torchrun, one rank per GPU): the headline batch shards across ranks (weak scaling: `--batch` is the per-GPU
batch), no data-path collective; the key limbs are broadcast from rank 0 over NCCL.
`--impl reference` times the reference's CPU path (oracle port of phe bound to libgmp -- the routine gmpy2.powmod wraps --
fanned over the host cores this process may really use) on a bounded sample of the same workload.
"""
import argparse
import json
import math
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

KEY_BITS = 2048
DEFAULT_BATCH = 1 << 20
ROWS_3072 = 1 << 22
DUMP_ROWS = 1 << 14
NOMINAL_MAC_PER_CLK_SM = 32.0     # IMAD.WIDE is a half-rate fmaheavy instruction: 4 SMSPs x 16 lanes / 2


# --------------------------------------------------------------------------------------------- MAC accounting
def sliding_counts(e, w):
    """(squarings, multiplications) of the engine's sliding-window program for the public exponent e (pai_engine.cu
    sliding_program: left to right, windows of at most w bits that start and end on a 1 bit)."""
    bits = bin(e)[2:]
    i, nsq, nmul, first = 0, 0, 0, True
    while i < len(bits):
        if bits[i] == "0":
            nsq += 1
            i += 1
            continue
        l = min(w, len(bits) - i)
        while bits[i + l - 1] == "0":
            l -= 1
        if first:
            first = False
        else:
            nsq += l
            nmul += 1
        i += l
    return nsq, nmul


def executed_macs(kb, n=None, scalar_bits=64, enc_path="digit", dec_path="digit", mul_path=None):
    """32x32->64 MACs the kernels really issue on the INTEGER pipe per op, counted from the loops.
    digit family (pai_digit.cuh): dsqr<T> = T(T+1)/2 + 3 T^2 tile products, dmul<T> = 5 T^2, a tile product = 64 MACs,
    plus 2T truncated quotient products (mul_lo8, 36 MACs) per dsqr/dmul (2048-bit: 228 + 16 and 320 + 16).
    tc family (pai_tc.cuh): the reductions run on the tensor cores, what is left is dsqr = T(T+1)/2 + T^2 (100 at 2048 bit),
    dmul = 3 T^2 (192), no quotient products; `tensor` counts the u8 x u8 MACs of the four [128 x D] x [D x D] GEMMs
    per product and ciphertext.  mont_mul<T> = 2 T^2 + T tiles + T mul_lo8; big_mul T x T = T^2 tiles."""
    def mont(t):
        return 64 * (2 * t * t + t) + 36 * t

    def ops(t, path):
        if path == "tc":
            return 64 * (t * (t + 1) // 2 + t * t), 64 * 3 * t * t, 4 * (32 * t) ** 2
        return 64 * (t * (t + 1) // 2 + 3 * t * t) + 36 * 2 * t, 64 * 5 * t * t + 36 * 2 * t, 0
    th = kb // 256                       # tiles of n
    tp = kb // 512                       # tiles of p, q
    if n is None:
        n = (1 << kb) - 1
    nsq, nmul = sliding_counts(n, 6)
    dsqr, dmul, tens = ops(th, enc_path)
    n_sq, n_mul = nsq + 1, nmul + 31 + 2                                         # table: 1 sqr + 31 mul; entry, exit
    enc = n_sq * dsqr + n_mul * dmul + 64 * th * th                              # + Z0 + n Z1
    enc_tensor = (n_sq + n_mul) * tens
    nwin = -(-(kb // 2) // 5)
    dsq, dmu, tens_d = ops(tp, dec_path)
    s_sq, s_mul = 1 + 5 * (nwin - 1), 4 + 29 + (nwin - 1) + 1
    side = s_sq * dsq + s_mul * dmu + mont(tp)
    dec = 2 * side + mont(tp) + 64 * tp * tp
    dec_tensor = 2 * (s_sq + s_mul) * tens_d
    add = 2 * mont(2 * th)
    nw = -(-scalar_bits // 4)
    dsqr_i, dmul_i, _ = ops(th, mul_path or enc_path)          # raw_mul runs on the same kernel family as encrypt
    mul = 2 * dmul_i + dsqr_i + 13 * dmul_i + (nw - 1) * (4 * dsqr_i + dmul_i) + dmul_i + 64 * th * th
    return {"encrypt": enc, "decrypt": dec, "add": add, "mul": mul, "mont_full": mont(2 * th),
            "encrypt_tensor_u8_macs": enc_tensor, "decrypt_tensor_u8_macs": dec_tensor}


def canonical_macs(kb, scalar_bits=64):
    """SURVEY.md section 8(d): canonical 32x32->64 MAC counts (schoolbook CIOS, window 5, no squaring credit)."""
    def modmul(L):
        return 2 * L * L + L

    def modexp(e, L):
        return (e + -(-e // 5) + 30 + 2) * modmul(L)
    enc = modexp(kb, kb // 16) + 2 * modmul(kb // 16) + (kb // 32) ** 2
    dec = 2 * modexp(kb // 2, kb // 32)
    return {"encrypt": enc, "decrypt": dec, "add": 2 * modmul(kb // 16),
            "mul": (scalar_bits + scalar_bits // 4 + 14 + 2) * modmul(kb // 16)}


# --------------------------------------------------------------------------------------------- clocks
class ClockSampler:
    """nvidia-smi clocks + throttle reasons during the timed region."""

    def __init__(self, index):
        self.index = index
        self.samples = []
        self.proc = None

    def start(self):
        q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
            "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q, "--format=csv,noheader,nounits",
                                          "-lms", "200"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.samples.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for s in self.samples:
            f = [x.strip() for x in s.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1]))
            except ValueError:
                continue
            for nm, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


# --------------------------------------------------------------------------------------------- CPU side
def host_cores():
    """Cores this process may really use: the scheduler affinity mask, clamped by the cgroup CPU quota
    (os.cpu_count() sees neither; round 1 counted 128 'cores' on a lease that delivered about 11)."""
    try:
        aff = len(os.sched_getaffinity(0))
    except (AttributeError, OSError):
        aff = os.cpu_count() or 1
    info = {"affinity": aff, "cpu_count": os.cpu_count(), "cgroup_quota": None}
    quota = None
    try:
        with open("/sys/fs/cgroup/cpu.max") as f:                        # cgroup v2
            q, p = f.read().split()[:2]
            if q != "max":
                quota = float(q) / float(p)
    except (OSError, ValueError):
        try:                                                             # cgroup v1
            with open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us") as f:
                q = float(f.read())
            with open("/sys/fs/cgroup/cpu/cpu.cfs_period_us") as f:
                p = float(f.read())
            if q > 0:
                quota = q / p
        except (OSError, ValueError):
            pass
    info["cgroup_quota"] = quota
    cores = aff if quota is None else max(1, min(aff, int(math.ceil(quota))))
    return cores, info


def _oracle(backend_gmp=True):
    from oracle import paillier_oracle as orc
    orc.BACKEND = "gmp" if (backend_gmp and orc.have_gmp()) else "python"
    return orc


def _cpu_worker(args):
    """Encrypt+decrypt `count` elements with the oracle port bound to libgmp.  Returns (enc_s, dec_s, backend)."""
    n, p, q, seed, count = args
    import random
    orc = _oracle()
    pub = orc.PublicConsts(n)
    priv = orc.PrivateConsts(pub, p, q)
    rng = random.Random(seed)
    ms = [rng.randrange(n) for _ in range(count)]
    rs = [rng.randrange(1, n) for _ in range(count)]
    t0 = time.perf_counter()
    cs = [orc.raw_encrypt(pub, m, r) for m, r in zip(ms, rs)]
    t1 = time.perf_counter()
    ds = [orc.raw_decrypt(priv, c) for c in cs]
    t2 = time.perf_counter()
    assert ds == ms
    return t1 - t0, t2 - t1, orc.BACKEND


def _check_worker(args):
    """Parity checker: oracle results for a slice of sampled rows.  kind: 'enc' (m, r) -> c, 'dec' c -> m,
    'add' (a, b), 'mul' (c, k)."""
    kind, n, p, q, rows = args
    orc = _oracle()
    pub = orc.PublicConsts(n)
    if kind == "enc":
        return [orc.raw_encrypt(pub, m, r) for m, r in rows]
    if kind == "dec":
        priv = orc.PrivateConsts(pub, p, q)
        return [orc.raw_decrypt(priv, c) for c in rows]
    if kind == "add":
        return [orc.raw_add(pub, a, b) for a, b in rows]
    if kind == "mul":
        return [orc.raw_mul(pub, c, k) for c, k in rows]
    raise ValueError(kind)


class CpuPool:
    """One spawn pool for the whole run (CPU baseline legs and the oracle side of the parity checks)."""

    def __init__(self, cores):
        import multiprocessing as mp
        self.cores = cores
        self.pool = mp.get_context("spawn").Pool(cores)

    def close(self):
        self.pool.terminate()
        self.pool.join()

    def oracle(self, kind, key, rows):
        n, p, q = key
        if not rows:
            return []
        per = max(1, -(-len(rows) // (4 * self.cores)))
        parts = [rows[i:i + per] for i in range(0, len(rows), per)]
        out = self.pool.map(_check_worker, [(kind, n, p, q, part) for part in parts])
        return [x for part in out for x in part]

    def sample(self, key, per_core, label):
        """All counted cores, `per_core` elements each."""
        n, p, q = key
        t0 = time.perf_counter()
        res = self.pool.map(_cpu_worker, [(n, p, q, 1000 + i, per_core) for i in range(self.cores)], chunksize=1)
        wall = time.perf_counter() - t0
        total = per_core * self.cores
        # whole-host throughput = sum of the per-process rates (one process per counted core)
        return {"enc_per_s": sum(per_core / r[0] for r in res), "dec_per_s": sum(per_core / r[1] for r in res),
                "cores": self.cores, "backend": res[0][2], "wall_s": wall,
                "sample": "%d encrypt + %d decrypt (%s) over %d processes" % (total, total, label, self.cores)}

    def single(self, key, count):
        r = self.pool.apply(_cpu_worker, ((key[0], key[1], key[2], 77, count),))
        return {"enc_per_s": count / r[0], "dec_per_s": count / r[1]}


def cpu_baseline(pool, key, per_core, label, info):
    c = pool.sample(key, per_core, label)
    one = pool.single(key, 64)
    per_core_rate = c["enc_per_s"] / c["cores"]
    out = {"value": c["enc_per_s"], "unit": "encrypts/s", "decrypts_per_s": c["dec_per_s"], "cores": c["cores"], "kind": "port",
           "sample": c["sample"], "single_process": {"encrypts_per_s": one["enc_per_s"], "decrypts_per_s": one["dec_per_s"]},
           "encrypts_per_s_per_counted_core": per_core_rate, "effective_cores": c["enc_per_s"] / one["enc_per_s"],
           "core_count_source": info,
           "engine": "oracle port of phe bound to libgmp mpz_powm (what gmpy2.powmod wraps)" if c["backend"] == "gmp"
                     else "oracle port of phe, Python pow"}
    if per_core_rate < 50 and c["backend"] == "gmp" and KEY_BITS == 2048:
        out["flag"] = ("CPU-starved box: %.1f encrypts/s per counted core (libgmp does ~110/s on one real core): the host "
                       "delivers fewer cores than it reports; effective_cores is the honest count" % per_core_rate)
    return out


def run_reference(args, key):
    """--impl reference: the reference's CPU path on this box's host cores, same metric/config."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores, info = host_cores()
    pool = CpuPool(cores)
    per_core = max(4, args.ref_per_core)
    for _ in range(args.warmup):
        pool.sample(key, 2, "2048-bit")
    t = [pool.sample(key, per_core, "2048-bit") for _ in range(args.steps)]
    one = pool.single(key, 64)
    pool.close()
    enc = sum(x["enc_per_s"] for x in t) / len(t)
    dec = sum(x["dec_per_s"] for x in t) / len(t)
    total = per_core * cores
    last = t[-1]
    line = {
        "impl": "reference", "metric": "paillier_raw_encrypts_per_sec_2048", "value": enc, "unit": "encrypts/s",
        "decrypt": {"value": dec, "unit": "decrypts/s"},
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1e3 * total / enc, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "u32 limbs (exact integer)", "data": "synthetic",
        "config": {"workload": "configs[1]: 2048-bit key raw_encrypt + raw_decrypt; each step is a bounded sample of %d elements "
                               "(rate-based: the CPU rate does not depend on the batch size)" % total, "key_bits": KEY_BITS},
        "cpu_baseline": {"value": enc, "unit": "encrypts/s", "decrypts_per_s": dec, "cores": cores, "kind": "port",
                         "sample": last["sample"], "core_count_source": info,
                         "single_process": {"encrypts_per_s": one["enc_per_s"], "decrypts_per_s": one["dec_per_s"]},
                         "effective_cores": enc / one["enc_per_s"],
                         "engine": "oracle port of phe bound to libgmp mpz_powm (what gmpy2.powmod wraps)"
                         if last["backend"] == "gmp" else "oracle port of phe, Python pow"},
        "e2e": {"value": enc, "unit": "encrypts/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    if enc / cores < 50 and last["backend"] == "gmp":
        line["cpu_baseline"]["flag"] = "CPU-starved box: %.1f encrypts/s per counted core" % (enc / cores)
    _emit(line)


# --------------------------------------------------------------------------------------------- GPU side helpers
def measured_int_peak():
    """Peak 32x32->64 MAC rate of the integer pipe, measured by bench_micro/imad_peak (IMAD.WIDE.U32.X chains)."""
    exe = os.path.join(ROOT, "bench_micro", "imad_peak")
    fallback = {"mac_per_clk_sm": 25.1, "source": "profiles/r01_imad_peak.json (earlier measurement on this pool)"}
    if not os.path.exists(exe):
        return fallback
    try:
        out = subprocess.run([exe], capture_output=True, text=True, timeout=120).stdout
        js = json.loads(out)
        best = max((r for r in js["results"] if "wide_chain" in r["op"]), key=lambda r: r["thread_ops_per_clk_per_sm"])
        res = {"mac_per_clk_sm": best["thread_ops_per_clk_per_sm"], "op": best["op"], "mhz": best["eff_mhz"], "sms": js["sms"],
               "source": "bench_micro/imad_peak run inside this bench"}
        noadd = [r for r in js["results"] if r["op"] == "mul_wide_no_addend"]
        if noadd:
            res["mul_wide_no_addend_per_clk_sm"] = max(r["thread_ops_per_clk_per_sm"] for r in noadd)
        return res
    except Exception as e:     # noqa: BLE001
        fallback["error"] = str(e)[:100]
        return fallback


def _ncu_traffic(name):
    """DRAM bytes (read + write) per row of the named kernel from the committed `ncu --set full` capture summary
    (profiles/r02c_ncu_traffic.json: the final build; falling back to earlier captures)."""
    for fn in ("r02c_ncu_traffic.json", "r02_ncu_traffic.json", "r01_ncu_traffic.json"):
        try:
            with open(os.path.join(ROOT, "profiles", fn)) as f:
                t = json.load(f)
            t = t.get(name, t) if isinstance(t.get(name), dict) else t
            return {"bytes_per_ciphertext": t["bytes_per_ciphertext"], "algorithmic_bytes_per_ciphertext": 1024,
                    "source": "profiles/" + fn + ": " + t.get("source", "")}
        except (OSError, KeyError, ValueError, AttributeError):
            continue
    return None


_OUT = None


def _emit(obj):
    out = _OUT or sys.stdout
    out.write(json.dumps(obj) + "\n")
    out.flush()


def _log(*a):
    sys.stderr.write(" ".join(str(x) for x in a) + "\n")
    sys.stderr.flush()


class Dev:
    """Per-rank device state shared by the legs."""

    def __init__(self, args):
        import torch
        self.torch = torch
        self.rank = int(os.environ.get("RANK", "0"))
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.local = int(os.environ.get("LOCAL_RANK", "0"))
        torch.cuda.set_device(self.local)
        self.dist = None
        if self.world > 1:
            os.environ.setdefault("NCCL_DEBUG", "WARN")          # keep stdout to the one JSON line
            import torch.distributed as dist
            dist.init_process_group("nccl", device_id=torch.device("cuda", self.local))
            self.dist = dist
        self.l2_flush = torch.empty(256 << 20, dtype=torch.int8, device="cuda")

    def barrier(self):
        self.torch.cuda.synchronize()
        if self.dist is not None:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def max_over_ranks(self, values):
        t = self.torch.tensor(values, dtype=self.torch.float64, device="cuda")
        if self.dist is not None:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return t.tolist()

    def timed(self, fn, steps, flush=True):
        """Average device time (ms) of fn over `steps` launches, CUDA events on the current stream (the engine calls of
        bench.py pass that stream), L2 flushed before every timed launch."""
        torch = self.torch
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
        for a, b in ev:
            if flush:
                self.l2_flush.zero_()
            a.record()
            fn()
            b.record()
        torch.cuda.synchronize()
        return sum(a.elapsed_time(b) for a, b in ev) / steps


def broadcast_key(dev, pb, np, key, kb):
    if dev.world == 1:
        return key
    kl = dev.torch.from_numpy(pb.ints_to_limbs(list(key), kb // 32).view(np.int32).copy()).cuda()
    dev.dist.broadcast(kl, 0)
    return tuple(pb.limbs_to_ints(kl.cpu().numpy().view(np.uint32)))


def uniform_rows(dev, pub, rows, seed, nonce):
    """[rows, n_limbs] uniform in [1, n) on the device (pai_random_lt_n: ChaCha20 + rejection sampling)."""
    t = dev.torch.empty((rows, pub.n_limbs), dtype=dev.torch.int32, device="cuda")
    pub.random_lt_n_dev(t, rows, seed=bytes([seed]) * 32, nonce=nonce, stream=cur_stream(dev))
    return t


def cur_stream(dev):
    return int(dev.torch.cuda.current_stream().cuda_stream)


def to_ints(pb, np, t):
    return pb.limbs_to_ints(t.cpu().numpy().view(np.uint32))


def sample_indices(B, count, seed):
    import random
    rng = random.Random(seed)
    idx = {0, 1, B // 2, B - 1} if B > 3 else set(range(B))
    while len(idx) < min(count, B):
        idx.add(rng.randrange(B))
    return sorted(idx)


def dump_outputs(out_dir, dev, np, B, outputs):
    """--dump-outputs: the same seeded sample of rows of each [B, limbs] int32 output every run, written as
    out_dir/<name>.npy in float64 (u32 limbs are exact there), with the sampled row numbers in out_dir/rows.npy.
    DUMP_ROWS rows of the 2048-bit outputs (128 + 64 limbs) come to 25 MB."""
    os.makedirs(out_dir, exist_ok=True)
    idx = sample_indices(B, DUMP_ROWS, 2024)
    ti = dev.torch.tensor(idx, device="cuda")
    np.save(os.path.join(out_dir, "rows.npy"), np.asarray(idx, dtype=np.float64))
    for name, t in outputs.items():
        np.save(os.path.join(out_dir, name + ".npy"), t[ti].cpu().numpy().view(np.uint32).astype(np.float64))


# --------------------------------------------------------------------------------------------- legs
def leg_headline(dev, args, pb, np, key, pool):
    torch = dev.torch
    n, p, q = key
    pub = pb.PublicContext(n, device=dev.local)
    priv = pb.PrivateContext(p, q, device=dev.local)
    ln, lc = pub.n_limbs, pub.c_limbs
    B = args.batch
    d_m = uniform_rows(dev, pub, B, 11, 2 * dev.rank)               # m, r uniform in [1, n)
    d_r = uniform_rows(dev, pub, B, 11, 2 * dev.rank + 1)
    d_c = torch.empty((B, lc), dtype=torch.int32, device="cuda")
    d_d = torch.empty((B, ln), dtype=torch.int32, device="cuda")
    eng = pb.get_engine()
    st = cur_stream(dev)

    for _ in range(args.warmup):
        pub.encrypt_dev(d_m, d_r, d_c, B, stream=st)
        priv.decrypt_dev(d_c, d_d, B, stream=st)
    dev.barrier()
    assert bool((d_d == d_m).all().item()), "decrypt(encrypt(m)) != m on device"
    parity = None
    if dev.rank == 0 and pool is not None:
        t0 = time.perf_counter()
        idx = sample_indices(B, args.parity_rows, 99)
        ti = torch.tensor(idx, device="cuda")
        mi, ri, ci, di = (to_ints(pb, np, t[ti]) for t in (d_m, d_r, d_c, d_d))
        assert ci == pool.oracle("enc", key, list(zip(mi, ri))), "device ciphertexts differ from the oracle"
        assert di == pool.oracle("dec", key, ci), "device plaintexts differ from the oracle"
        parity = {"rows_checked_vs_gmp_oracle": len(idx), "encrypt": "bit-exact", "decrypt": "bit-exact",
                  "full_batch_roundtrip_on_device": True, "seconds": time.perf_counter() - t0}

    sampler = ClockSampler(dev.local)
    if dev.rank == 0:
        sampler.start()
    launches0 = eng.launch_count()
    ev = [[torch.cuda.Event(enable_timing=True) for _ in range(3)] for _ in range(args.steps)]
    dev.barrier()
    t_wall0 = time.perf_counter()
    for i in range(args.steps):
        dev.l2_flush.zero_()                       # flush L2 between timed iterations (256 MiB > 126 MB L2)
        ev[i][0].record()
        pub.encrypt_dev(d_m, d_r, d_c, B, stream=st)
        ev[i][1].record()
        priv.decrypt_dev(d_c, d_d, B, stream=st)
        ev[i][2].record()
    dev.barrier()
    t_wall = time.perf_counter() - t_wall0
    launches = eng.launch_count() - launches0
    enc_each = sorted(e[0].elapsed_time(e[1]) for e in ev)
    dec_each = sorted(e[1].elapsed_time(e[2]) for e in ev)
    spread = {"encrypt_ms": {"min": enc_each[0], "median": enc_each[len(enc_each) // 2], "max": enc_each[-1]},
              "decrypt_ms": {"min": dec_each[0], "median": dec_each[len(dec_each) // 2], "max": dec_each[-1]},
              "note": "per-step device times of rank 0 (the reported value is the mean over the K steps, max over ranks)"}
    enc_ms = sum(enc_each) / args.steps
    dec_ms = sum(dec_each) / args.steps
    enc_ms, dec_ms = dev.max_over_ranks([enc_ms, dec_ms])
    clocks = sampler.stop() if dev.rank == 0 else None
    if args.dump_outputs and dev.rank == 0:
        dump_outputs(args.dump_outputs, dev, np, B, {"ciphertexts": d_c, "plaintexts": d_d})

    # ---- end to end through the host-pointer C ABI, pinned host buffers, same batch
    e2e = None
    if not args.no_e2e:
        h_m = torch.empty((B, ln), dtype=torch.int32).pin_memory(); h_m.copy_(d_m)
        h_r = torch.empty((B, ln), dtype=torch.int32).pin_memory(); h_r.copy_(d_r)
        h_c = torch.empty((B, lc), dtype=torch.int32).pin_memory()
        h_d = torch.empty((B, ln), dtype=torch.int32).pin_memory()
        reps = max(1, min(args.steps, args.e2e_steps))

        def e2e_step():
            eng.check(eng.lib.pai_encrypt_host(pub.h, h_m.data_ptr(), h_r.data_ptr(), h_c.data_ptr(), B))
            t1 = time.perf_counter()
            eng.check(eng.lib.pai_decrypt_host(priv.h, h_c.data_ptr(), h_d.data_ptr(), B))
            return t1
        e2e_step()
        dev.barrier()
        te, td = 0.0, 0.0
        for _ in range(reps):
            t0 = time.perf_counter()
            t1 = e2e_step()
            t2 = time.perf_counter()
            te += t1 - t0; td += t2 - t1
        assert bool((h_d == h_m).all().item())
        te, td = dev.max_over_ranks([te / reps, td / reps])
        e2e = {"value": dev.world * B / te, "unit": "encrypts/s", "decrypts_per_s": dev.world * B / td, "steps": reps,
               "batch_per_gpu": B, "h2d_bytes_per_step": B * (2 * ln + lc) * 4, "d2h_bytes_per_step": B * (lc + ln) * 4,
               "api": "pai_encrypt_host / pai_decrypt_host (C ABI, limb matrices in pinned host buffers)"}
        del h_c, h_d, h_r, h_m

    # ---- end to end through the Python-int API of the drop-in (what a phe user calls)
    e2e_py = None
    if not args.no_e2e and dev.rank == 0 and dev.world == 1:
        Bp = min(B, args.python_rows)
        pk = pb.PaillierPublicKey(n)
        sk = pb.PaillierPrivateKey(pk, p, q)
        pk._ctx, sk._ctx = pub, priv
        ml, rl = to_ints(pb, np, d_m[:Bp]), to_ints(pb, np, d_r[:Bp])
        t0 = time.perf_counter()
        cl = pk.raw_encrypt_batch(ml, rl)
        t1 = time.perf_counter()
        dl = sk.raw_decrypt_batch(cl)
        t2 = time.perf_counter()
        assert dl == ml and cl[:64] == to_ints(pb, np, d_c[:64])
        e2e_py = {"encrypts_per_s": Bp / (t1 - t0), "decrypts_per_s": Bp / (t2 - t1), "batch": Bp, "unit": "ops/s",
                  "api": "PaillierPublicKey.raw_encrypt_batch / PaillierPrivateKey.raw_decrypt_batch: list[int] -> list[int] "
                         "(int<->limb conversion pipelined against the kernels in wave-sized chunks)",
                  "vs_limb_e2e": None if e2e is None else {"encrypt": Bp / (t1 - t0) / e2e["value"],
                                                           "decrypt": Bp / (t2 - t1) / e2e["decrypts_per_s"]}}
        del ml, rl, cl, dl
    res = {"enc_ms": enc_ms, "dec_ms": dec_ms, "spread": spread, "t_wall": t_wall, "launches": launches, "clocks": clocks, "e2e": e2e,
           "e2e_python": e2e_py, "parity": parity, "ln": ln, "lc": lc, "wave_enc": pub.wave(), "wave_dec": priv.wave(),
           "enc_path": pub.kernel_path(), "dec_path": priv.kernel_path()}
    return res, (pub, priv, d_m, d_r, d_c, d_d)


def leg_add_mul(dev, args, pb, np, key, pool, state, peak_mac_s):
    """configs[2]: 1M ciphertext pairs, _raw_add and _raw_mul."""
    torch = dev.torch
    pub, priv, d_m, d_r, d_c, d_d = state
    n = key[0]
    B = d_c.shape[0]
    st = cur_stream(dev)
    d_r2 = uniform_rows(dev, pub, B, 12, dev.rank)
    d_c2 = torch.empty_like(d_c)
    pub.encrypt_dev(d_m, d_r2, d_c2, B, stream=st)                 # second ciphertext of the same plaintexts, other r stream
    d_o = torch.empty_like(d_c)
    status = torch.zeros((B,), dtype=torch.int32, device="cuda")
    out = {"batch_per_gpu": B}
    steps = max(1, min(args.steps, 3))
    pub.raw_add_dev(d_c, d_c2, d_o, B, stream=st)
    add_ms = dev.timed(lambda: pub.raw_add_dev(d_c, d_c2, d_o, B, stream=st), steps)
    priv.decrypt_dev(d_o, d_d, B, stream=st)
    # homomorphism on the whole batch: dec(c * c2) == 2 m mod n, checked on the device through a second add of plaintext limbs
    add_o = d_o.clone()

    def scalars(kind):
        s = torch.zeros((B, pub.n_limbs), dtype=torch.int32, device="cuda")
        if kind == "u64":
            s[:, :2] = d_m[:, :2]
        elif kind == "float":
            vec = __import__("importlib").import_module("python-paillier_b200.vector")
            vals = np.random.RandomState(5).randn(B) * 0.1
            pk = pb.PaillierPublicKey(n); pk._ctx = pub
            limbs, _ = vec.encode_batch(pk, vals)                 # EncodedNumber.encode of float64: 53-56-bit mantissas,
            s = torch.from_numpy(limbs.view(np.int32).copy()).cuda()   # negative values wrap to n - |x| (invert branch)
        elif kind == "neg":
            vec = __import__("importlib").import_module("python-paillier_b200.vector")
            k = (d_m[:, :2].cpu().numpy().view(np.uint32).astype(np.int64))
            k = (k[:, 0] | (k[:, 1] << 32)) & (2 ** 62 - 1)
            limbs = vec._limbs_from_signed(-k, n, pub.n_limbs)      # n - k: the encoding of the negative scalar -k
            s = torch.from_numpy(limbs.view(np.int32).copy()).cuda()
        return s.contiguous()
    mul = {}
    kept = {}
    for kind in ("u64", "float", "neg"):
        d_s = scalars(kind)
        pub.raw_mul_dev(d_c, d_s, d_o, status, B, stream=st)
        ms = dev.timed(lambda: pub.raw_mul_dev(d_c, d_s, d_o, status, B, stream=st), steps if kind == "u64" else 1)
        assert not bool(status.any().item())
        mul[kind] = ms
        kept[kind] = (d_s, d_o.clone() if kind == "u64" else None)
        if kind != "u64":
            # parity on a few rows for the secondary mixes
            if dev.rank == 0 and pool is not None:
                idx = sample_indices(B, 64, 5)
                ti = torch.tensor(idx, device="cuda")
                assert to_ints(pb, np, d_o[ti]) == pool.oracle("mul", key, list(zip(to_ints(pb, np, d_c[ti]), to_ints(pb, np, d_s[ti]))))
    add_ms, mul_u64, mul_f, mul_n = dev.max_over_ranks([add_ms, mul["u64"], mul["float"], mul["neg"]])
    if dev.rank == 0 and pool is not None:
        idx = sample_indices(B, args.parity_rows_small, 7)
        ti = torch.tensor(idx, device="cuda")
        a, b = to_ints(pb, np, d_c[ti]), to_ints(pb, np, d_c2[ti])
        assert to_ints(pb, np, add_o[ti]) == pool.oracle("add", key, list(zip(a, b))), "raw_add differs from the oracle"
        ks = to_ints(pb, np, kept["u64"][0][ti])
        assert to_ints(pb, np, kept["u64"][1][ti]) == pool.oracle("mul", key, list(zip(a, ks))), "raw_mul differs from the oracle"
        out["parity"] = {"rows_checked_vs_gmp_oracle": len(idx), "add": "bit-exact", "mul": "bit-exact (u64: %d rows; float / negative mixes: 64 rows each)" % len(idx)}
    W = dev.world
    ex, ca = executed_macs(KEY_BITS, n, enc_path=pub.kernel_path()), canonical_macs(KEY_BITS)
    add_s, mul_s = W * B / (add_ms * 1e-3), W * B / (mul_u64 * 1e-3)
    hbm = _hbm_peak()
    out.update({
        "raw_add": {"value": add_s, "unit": "adds/s", "ms": add_ms, "kernel": "k_body<MulBody<16>> (2 full-width Montgomery products mod n^2)",
                    "roofline": {"bound": "int_pipe", "frac": add_s / W * ex["add"] / peak_mac_s, "canonical_frac": add_s / W * ca["add"] / peak_mac_s,
                                 "executed_macs_per_op": ex["add"], "hbm_gbs": add_s / W * 1536 / 1e9, "hbm_frac": add_s / W * 1536 / 1e9 / hbm[0]}},
        "raw_mul_u64": {"value": mul_s, "unit": "muls/s", "ms": mul_u64,
                        "kernel": "rawmul_prep + k_body<InvBatchBody<16>> (copy rows) + " + ("k_body<TcPowBody<8,4>>" if pub.kernel_path() == "tc" else "k_body<PowDigitBody<8,4>>"),
                        "roofline": {"bound": "int_pipe", "frac": mul_s / W * ex["mul"] / peak_mac_s,
                                     "canonical_frac": mul_s / W * ca["mul"] / peak_mac_s, "executed_macs_per_op": ex["mul"]}},
        "raw_mul_float_encoded": {"value": W * B / (mul_f * 1e-3), "unit": "muls/s", "ms": mul_f,
                                  "note": "EncodedNumber.encode(N(0, 0.1) float64): 53-56-bit exponents, half of them negative -> invert + powmod"},
        "raw_mul_negative": {"value": W * B / (mul_n * 1e-3), "unit": "muls/s", "ms": mul_n, "note": "k = n - u64: every row takes invert(c, n^2) first (amortised: one extended gcd per segment of rows, cta_invert_batch)"},
    })
    return out


def _hbm_peak():
    peaks_file = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(peaks_file):
        return json.load(open(peaks_file))["hbm_gbs"], "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def leg_3072(dev, args, pb, np, pool, peak_mac_s, H, load_golden):
    """configs[3]: 3072-bit key (the reference's DEFAULT_KEYSIZE, phe/paillier.py:34), total rows sharded over the ranks
    (strong scaling), NCCL key broadcast, encrypt + decrypt, and the all-gather of the ciphertext shards timed apart."""
    torch = dev.torch
    par = __import__("importlib").import_module("python-paillier_b200.parallel")
    fx = load_golden("vectors_3072.json")
    t0 = time.perf_counter()
    key = broadcast_key(dev, pb, np, (H(fx["n"]), H(fx["p"]), H(fx["q"])), 3072)
    torch.cuda.synchronize()
    bcast_ms = (time.perf_counter() - t0) * 1e3
    n, p, q = key
    pub = pb.PublicContext(n, device=dev.local)
    priv = pb.PrivateContext(p, q, device=dev.local)
    total = args.rows3072
    lo, hi = par.shard_range(total, dev.rank, dev.world)
    rows = hi - lo
    st = cur_stream(dev)
    d_m = uniform_rows(dev, pub, rows, 13, 2 * dev.rank)
    d_r = uniform_rows(dev, pub, rows, 13, 2 * dev.rank + 1)
    d_c = torch.empty((rows, pub.c_limbs), dtype=torch.int32, device="cuda")
    d_d = torch.empty((rows, pub.n_limbs), dtype=torch.int32, device="cuda")
    w = min(rows, pub.wave())
    pub.encrypt_dev(d_m[:w], d_r[:w], d_c[:w], w, stream=st)      # warm-up: one wave (contexts, tables, clocks)
    priv.decrypt_dev(d_c[:w], d_d[:w], w, stream=st)
    dev.barrier()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
    ev[0].record()
    pub.encrypt_dev(d_m, d_r, d_c, rows, stream=st)
    ev[1].record()
    priv.decrypt_dev(d_c, d_d, rows, stream=st)
    ev[2].record()
    dev.barrier()
    enc_ms, dec_ms = dev.max_over_ranks([ev[0].elapsed_time(ev[1]), ev[1].elapsed_time(ev[2])])
    assert bool((d_d == d_m).all().item()), "3072-bit: decrypt(encrypt(m)) != m"
    out = {"key_bits": 3072, "total_rows": total, "rows_per_rank": rows, "scaling": "strong", "waves_per_rank": rows / max(1, pub.wave()),
           "encrypts_per_s": total / (enc_ms * 1e-3), "decrypts_per_s": total / (dec_ms * 1e-3), "enc_ms": enc_ms, "dec_ms": dec_ms,
           "key_broadcast_ms": bcast_ms if dev.world > 1 else None, "steps": 1,
           "note": "one timed pass over the whole vector after a one-wave warm-up; inputs uniform in [1, n) (pai_random_lt_n)"}
    ex, ca = executed_macs(3072, n, enc_path=pub.kernel_path(), dec_path=priv.kernel_path()), canonical_macs(3072)
    out["kernel_family"] = {"encrypt": pub.kernel_path(), "decrypt": priv.kernel_path()}
    per_gpu_enc = total / dev.world / (enc_ms * 1e-3)
    per_gpu_dec = total / dev.world / (dec_ms * 1e-3)
    out["roofline"] = {"bound": "int_pipe", "kernel": "k_body<TcEncBody<12>>" if pub.kernel_path() == "tc" else "k_body<EncDigitBody<12>>", "frac": per_gpu_enc * ex["encrypt"] / peak_mac_s,
                       "canonical_frac": per_gpu_enc * ca["encrypt"] / peak_mac_s, "executed_macs_per_encrypt": ex["encrypt"],
                       "decrypt": {"frac": per_gpu_dec * ex["decrypt"] / peak_mac_s, "canonical_frac": per_gpu_dec * ca["decrypt"] / peak_mac_s}}
    if dev.rank == 0 and pool is not None:
        idx = sample_indices(rows, args.parity_rows_small, 3)
        ti = torch.tensor(idx, device="cuda")
        mi, ri, ci = (to_ints(pb, np, t[ti]) for t in (d_m, d_r, d_c))
        assert ci == pool.oracle("enc", key, list(zip(mi, ri))), "3072-bit ciphertexts differ from the oracle"
        assert mi == pool.oracle("dec", key, ci)
        out["parity"] = {"rows_checked_vs_gmp_oracle": len(idx), "encrypt": "bit-exact", "decrypt": "bit-exact", "full_shard_roundtrip_on_device": True}
    if dev.world > 1:
        del d_d, d_r
        g = par.all_gather_rows(d_c, total)                        # warm-up (NCCL channels, allocator)
        del g
        dev.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        g = par.all_gather_rows(d_c, total)
        e1.record()
        dev.barrier()
        (ag_ms,) = dev.max_over_ranks([e0.elapsed_time(e1)])
        assert g.shape[0] == total and bool((g[lo:hi] == d_c).all().item())
        recv = (total - rows) * pub.c_limbs * 4
        out["allgather"] = {"ms": ag_ms, "bytes_received_per_gpu": recv, "gbs_per_gpu": recv / (ag_ms * 1e-3) / 1e9,
                            "api": "parallel.all_gather_rows (NCCL all_gather of padded shards + concat)",
                            "share_of_encrypt_time": ag_ms / enc_ms}
        del g
    return out


def leg_multi_parity(dev, args, pb, np, pool, H, load_golden):
    """N > 1 correctness inside the bench (GPUTEST boxes have one GPU): a seeded vector is sharded, every rank encrypts its
    rows, the shards are all-gathered and rank 0 compares gathered rows of EVERY shard with the GMP oracle."""
    if dev.world == 1:
        return None
    torch = dev.torch
    par = __import__("importlib").import_module("python-paillier_b200.parallel")
    fx = load_golden("vectors_3072.json")
    key = broadcast_key(dev, pb, np, (H(fx["n"]), H(fx["p"]), H(fx["q"])), 3072)
    pub = pb.PublicContext(key[0], device=dev.local)
    priv = pb.PrivateContext(key[1], key[2], device=dev.local)
    total = 4096 * dev.world + 37                                   # ragged split
    lo, hi = par.shard_range(total, dev.rank, dev.world)
    st = cur_stream(dev)
    d_m = uniform_rows(dev, pub, hi - lo, 21, 2 * dev.rank)
    d_r = uniform_rows(dev, pub, hi - lo, 21, 2 * dev.rank + 1)
    d_c = torch.empty((hi - lo, pub.c_limbs), dtype=torch.int32, device="cuda")
    pub.encrypt_dev(d_m, d_r, d_c, hi - lo, stream=st)
    gm, gr, gc = (par.all_gather_rows(t, total) for t in (d_m, d_r, d_c))
    d_d = torch.empty((total, pub.n_limbs), dtype=torch.int32, device="cuda")
    priv.decrypt_dev(gc, d_d, total, stream=st)                     # every rank decrypts the WHOLE gathered vector
    ok = bool((d_d == gm).all().item())
    res = None
    if dev.rank == 0:
        import random
        rng = random.Random(17)
        idx = []
        for r in range(dev.world):
            a, b = par.shard_range(total, r, dev.world)
            idx += [a, b - 1] + [rng.randrange(a, b) for _ in range(max(2, 640 // dev.world))]
        idx = sorted(set(idx))
        ti = torch.tensor(idx, device="cuda")
        mi, ri, ci = (to_ints(pb, np, t[ti]) for t in (gm, gr, gc))
        if pool is not None:
            assert ci == pool.oracle("enc", key, list(zip(mi, ri))), "gathered ciphertexts differ from the oracle"
        res = {"world": dev.world, "vector_rows": total, "gathered_rows_checked_vs_gmp_oracle": len(idx) if pool is not None else 0,
               "shards_covered": dev.world, "result": "bit-exact" if pool is not None else "oracle check skipped (--no-cpu): device round trip only",
               "decrypt_of_gathered_vector_on_every_rank": None}
    (allok,) = dev.max_over_ranks([0.0 if ok else 1.0])
    assert allok == 0.0, "a rank failed to decrypt the gathered vector"
    if res:
        res["decrypt_of_gathered_vector_on_every_rank"] = True
    return res


def leg_reductions(dev, args, pb, np, key, pool, state):
    """SURVEY 8(f2): homomorphic sum / dot of a 1e5-element encrypted vector, fused kernels vs the launch chains."""
    torch = dev.torch
    vec = __import__("importlib").import_module("python-paillier_b200.vector")
    if not hasattr(vec.EncryptedVector, "sum_chain"):
        return None
    pub, priv, d_m, d_r, d_c, d_d = state
    n, p, q = key
    pk = pb.PaillierPublicKey(n); pk._ctx = pub
    sk = pb.PaillierPrivateKey(pk, p, q); sk._ctx = priv
    R = min(args.reduce_rows, d_c.shape[0])
    v = vec.EncryptedVector(pk, d_c[:R].contiguous(), np.zeros(R, dtype=np.int64))
    eng = pb.get_engine()
    out = {"rows": R}

    def wall(fn, reps=3):
        fn()
        torch.cuda.synchronize()
        l0 = eng.launch_count()
        t0 = time.perf_counter()
        for _ in range(reps):
            r = fn()
        torch.cuda.synchronize()
        return (time.perf_counter() - t0) / reps * 1e3, (eng.launch_count() - l0) // reps, r
    f_ms, f_l, s_f = wall(v.sum)
    c_ms, c_l, s_c = wall(v.sum_chain)
    assert s_f.ciphertext(False) == s_c.ciphertext(False)
    ms_sum = sum(to_ints(pb, np, d_m[:R])) % n
    assert sk.raw_decrypt(s_f.ciphertext(False)) == ms_sum
    out["sum"] = {"fused_ms": f_ms, "fused_launches": f_l, "chain_ms": c_ms, "chain_launches": c_l, "speedup": c_ms / f_ms,
                  "check": "equal to the chain and to sum(m) mod n after decryption"}
    ks = (np.random.RandomState(9).randint(1, 2 ** 62, size=R)).astype(np.int64)
    f_ms, f_l, d_f = wall(lambda: v.dot(ks), reps=2)
    c_ms, c_l, d_c2 = wall(lambda: v.dot_chain(ks), reps=2)
    assert d_f.ciphertext(False) == d_c2.ciphertext(False)
    out["dot_u62"] = {"fused_ms": f_ms, "fused_launches": f_l, "chain_ms": c_ms, "chain_launches": c_l, "speedup": c_ms / f_ms,
                      "check": "equal to mul + sum chain"}
    return out


def leg_federated(dev, args, pb, np, key, cores):
    """configs[4]: one round of examples/federated_learning_with_encryption.py's protocol shape (5 clients, D float64
    gradients each): encrypt, ring sum with exponent alignment, decrypt, average.  CPU side: the same round on ONE core with
    the oracle port on a D' sub-vector, scaled (stated as such), and its ideal fan-out over the counted cores."""
    torch = dev.torch
    n, p, q = key
    pk = pb.PaillierPublicKey(n)
    sk = pb.PaillierPrivateKey(pk, p, q)
    D, C = args.fed_dim, 5
    grads = [np.random.RandomState(43 + i).randn(D) * 0.1 for i in range(C)]
    # warm-up: one small round through every call of the protocol (context creation, workspace allocation of this key's
    # contexts -- a fresh key pair, as a client would have -- are not part of a round)
    w = [pk.encrypt_batch(g[:D // 2 + 7]) for g in grads[:2]]
    sk.decrypt_batch(w[0] + w[1])
    del w
    torch.cuda.synchronize()
    t = {}
    t0 = time.perf_counter()
    enc = [pk.encrypt_batch(g) for g in grads]
    torch.cuda.synchronize()
    t["encrypt_s"] = time.perf_counter() - t0
    t0 = time.perf_counter()
    acc = enc[0]
    for e in enc[1:]:
        acc = acc + e
    torch.cuda.synchronize()
    t["sum_s"] = time.perf_counter() - t0
    t0 = time.perf_counter()
    agg = np.array(sk.decrypt_batch(acc)) / C
    t["decrypt_s"] = time.perf_counter() - t0
    t["round_s"] = sum(t.values())
    ok = bool(np.allclose(agg, np.mean(grads, axis=0), rtol=0, atol=1e-12))
    assert ok
    import random
    orc = _oracle()
    opub = orc.PublicConsts(n)
    opriv = orc.PrivateConsts(opub, p, q)
    S = args.fed_cpu_sample
    rng = random.Random(1)
    t0 = time.perf_counter()
    encs = [[pb.EncodedNumber.encode(pk, float(x)) for x in g[:S]] for g in grads]
    cts = [[orc.raw_encrypt(opub, e.encoding, rng.randrange(1, n)) for e in row] for row in encs]
    accc, acce = cts[0], [e.exponent for e in encs[0]]
    for row, erow in zip(cts[1:], encs[1:]):
        nxt, nxe = [], []
        for a, ea, b, eb in zip(accc, acce, row, erow):
            ex = min(ea, eb.exponent)
            if ea > ex:
                a = orc.raw_mul(opub, a, 16 ** (ea - ex))
            if eb.exponent > ex:
                b = orc.raw_mul(opub, b, 16 ** (eb.exponent - ex))
            nxt.append(orc.raw_add(opub, a, b)); nxe.append(ex)
        accc, acce = nxt, nxe
    dec = [orc.raw_decrypt(opriv, c) for c in accc]
    cpu_s = time.perf_counter() - t0
    cpu_vals = [pb.EncodedNumber(pk, d, e).decode() / C for d, e in zip(dec, acce)]
    assert np.allclose(cpu_vals, agg[:S], rtol=0, atol=1e-12)
    scaled = cpu_s * D / S
    return {"workload": "configs[4]: 5 clients x %d float64 gradients, 2048-bit key" % D, "gpu": t, "aggregate_matches_plaintext_mean": ok,
            "cpu_reference": {"one_core_round_s_scaled": scaled, "sample_elements_per_client": S, "cores": cores,
                              "all_cores_round_s_ideal": scaled / cores,
                              "note": "oracle port on libgmp, measured on one core over a %d-element sub-vector and scaled to D; "
                                      "the reference itself is single-threaded" % S},
            "speedup_vs_one_core": scaled / t["round_s"], "speedup_vs_all_counted_cores_ideal": scaled / cores / t["round_s"]}


# --------------------------------------------------------------------------------------------- main
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=2)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--batch", type=int, default=DEFAULT_BATCH, help="elements per GPU per step (headline leg)")
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--ref-per-core", type=int, default=48)
    ap.add_argument("--cpu-per-core", type=int, default=48)
    ap.add_argument("--no-cpu", action="store_true", help="skip the CPU baseline AND the oracle parity checks")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="headline leg only")
    ap.add_argument("--rows3072", type=int, default=ROWS_3072, help="total rows of the 3072-bit leg (all ranks together)")
    ap.add_argument("--parity-rows", type=int, default=4096)
    ap.add_argument("--parity-rows-small", type=int, default=512)
    ap.add_argument("--python-rows", type=int, default=DEFAULT_BATCH)
    ap.add_argument("--e2e-steps", type=int, default=2)
    ap.add_argument("--reduce-rows", type=int, default=100000)
    ap.add_argument("--fed-dim", type=int, default=100000)
    ap.add_argument("--fed-cpu-sample", type=int, default=60)
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write a fixed sample of rows of the last step's ciphertexts and decrypted "
                         "plaintexts to DIR/*.npy (rank 0's shard when --gpus > 1)")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of the b200 headline leg")
    # the contract is ONE JSON line on stdout: native libraries (NCCL's version banner, ...) write to fd 1 as well, so
    # everything but the final line is sent to stderr
    global _OUT
    sys.stdout.flush()
    _OUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)

    import importlib
    H, load_golden = (lambda m: (m.H, m.load_golden))(importlib.import_module("python-paillier_b200.fixtures"))
    fx = load_golden("vectors_%d.json" % KEY_BITS)
    key = (H(fx["n"]), H(fx["p"]), H(fx["q"]))
    if args.impl == "reference":
        run_reference(args, key)
        return

    import numpy as np
    import paillier_b200 as pb

    dev = Dev(args)
    # key limbs travel from rank 0 to every rank over NCCL (a few hundred bytes); batches never move
    key = broadcast_key(dev, pb, np, key, KEY_BITS)
    cores, core_info = host_cores()
    pool = None
    if dev.rank == 0 and not args.no_cpu:
        pool = CpuPool(cores)                                      # spawn pool: oracle side of the parity checks + CPU baseline
    t_all = time.perf_counter()
    head, state = leg_headline(dev, args, pb, np, key, pool)
    _log("headline done", time.perf_counter() - t_all)

    enc_ms, dec_ms = head["enc_ms"], head["dec_ms"]
    B, world, ln, lc = args.batch, dev.world, head["ln"], head["lc"]
    enc_per_s = world * B / (enc_ms * 1e-3)
    dec_per_s = world * B / (dec_ms * 1e-3)
    clocks = head["clocks"]
    peak = measured_int_peak() if dev.rank == 0 else {"mac_per_clk_sm": 25.1}
    sm_mhz = (clocks or {}).get("sm_mhz") or peak.get("mhz") or 1965.0
    (pk_mac, sm_mhz) = dev.max_over_ranks([peak["mac_per_clk_sm"] if dev.rank == 0 else 0.0, sm_mhz if dev.rank == 0 else 0.0])
    peak_mac_s = pk_mac * 148 * sm_mhz * 1e6
    nominal_mac_s = NOMINAL_MAC_PER_CLK_SM * 148 * sm_mhz * 1e6

    extras = {}
    if not args.no_extras:
        for name, fn in (("config2_add_mul", lambda: leg_add_mul(dev, args, pb, np, key, pool, state, peak_mac_s)),
                         ("reductions", lambda: leg_reductions(dev, args, pb, np, key, pool, state) if dev.world == 1 else None)):
            t0 = time.perf_counter()
            extras[name] = fn()
            _log(name, "done", time.perf_counter() - t0)
    pub, priv = state[0], state[1]
    del state
    dev.torch.cuda.empty_cache()
    if not args.no_extras:
        for name, fn in (("config3072", lambda: leg_3072(dev, args, pb, np, pool, peak_mac_s, H, load_golden)),
                         ("multi_gpu_parity", lambda: leg_multi_parity(dev, args, pb, np, pool, H, load_golden)),
                         ("federated", lambda: leg_federated(dev, args, pb, np, key, cores) if (dev.world == 1 and not args.no_cpu) else None)):
            t0 = time.perf_counter()
            extras[name] = fn()
            dev.torch.cuda.empty_cache()
            _log(name, "done", time.perf_counter() - t0)

    if dev.rank != 0:
        if dev.dist is not None:
            dev.dist.destroy_process_group()
        return

    ex, ca = executed_macs(KEY_BITS, key[0], enc_path=head["enc_path"], dec_path=head["dec_path"]), canonical_macs(KEY_BITS)
    hbm_peak, hbm_src = _hbm_peak()
    ach = enc_per_s / world * ex["encrypt"]
    kern = {"tc": "k_body<TcEncBody<8>> (raw_encrypt: digit products on the integer pipe, Montgomery reductions as tcgen05 kind::i8 GEMMs)",
            "digit": "k_body<EncDigitBody<8>> (raw_encrypt, r^n mod n^2 on base-n digits)", "full": "k_body<EncBody<16>>"}
    kern_d = {"tc": "k_body<TcDecBody<4,5>>", "digit": "k_body<DecDigitBody<4,5>>", "full": "k_body<DecBody<4,5>>"}
    tensor_peak = 2 * json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["bf16_tflops"] / 2 if os.path.exists(os.path.join(ROOT, "MEASURED_PEAKS.json")) else 1590.0
    roofline = {
        "bound": "int_pipe", "kernel": kern[head["enc_path"]], "kernel_family": head["enc_path"],
        "achieved": ach / 1e12, "peak": peak_mac_s / 1e12, "unit": "TMAC/s (32x32->64 MACs the kernel executes, per GPU)",
        "frac": ach / peak_mac_s,
        "frac_of_nominal_pipe": ach / nominal_mac_s, "peak_nominal": nominal_mac_s / 1e12,
        "canonical_frac": enc_per_s / world * ca["encrypt"] / peak_mac_s,
        "executed_macs_per_encrypt": ex["encrypt"], "canonical_macs_per_encrypt": ca["encrypt"],
        "note": "frac = MACs executed on the integer pipe / measured IMAD.WIDE.U32 peak.  canonical_frac uses SURVEY 8(d)'s schoolbook count; the "
                "base-n digit arithmetic halves it and the tensor-core reductions halve it again (algorithmic savings, not throughput) -- "
                "it exceeds 1.  peak_nominal = 32 MAC/clk/SM "
                "(half-rate fmaheavy instruction); the measured peak is ~25: an IMAD.WIDE with a 64-bit addend issues every 5th cycle "
                "per SM sub-partition, not every 4th (bench_micro/imad_peak: the same instruction without an addend, "
                "mul_wide_no_addend, is reported beside it), so ~0.78 of nominal is the ceiling of this instruction and ncu's "
                "sm__pipe_fmaheavy_cycles_active tops out near 80 %",
        "peak_source": "measured IMAD.WIDE.U32.X rate %.1f MAC/clk/SM (%s) x 148 SMs x %.0f MHz (SM clock sampled under load)"
                       % (pk_mac, peak.get("source"), sm_mhz),
        "peak_micro": peak,
        "decrypt": {"kernel": kern_d[head["dec_path"]], "kernel_family": head["dec_path"], "frac": dec_per_s / world * ex["decrypt"] / peak_mac_s,
                    "canonical_frac": dec_per_s / world * ca["decrypt"] / peak_mac_s, "executed_macs_per_decrypt": ex["decrypt"]},
        "tensor": {"u8_macs_per_encrypt": ex["encrypt_tensor_u8_macs"], "achieved_tmacs": enc_per_s / world * ex["encrypt_tensor_u8_macs"] / 1e12,
                   "peak_tmacs_int8_dense": tensor_peak, "frac": enc_per_s / world * ex["encrypt_tensor_u8_macs"] / 1e12 / tensor_peak,
                   "note": "the reductions' GEMMs ([128 x D] x Toeplitz, u8 x u8 -> s32); peak = measured dense bf16 TFLOP/s x 2 (int8) / 2 (MAC = 2 ops); "
                           "the tensor pipe is a helper here, not the bound"},
        "hbm": {"achieved_gbs": enc_per_s / world * (ln * 2 + lc) * 4 / 1e9, "peak_gbs": hbm_peak, "peak_source": hbm_src,
                "frac": enc_per_s / world * (ln * 2 + lc) * 4 / 1e9 / hbm_peak},
        "traffic": _ncu_traffic("encrypt"),
    }
    cpu = None
    if pool is not None and world == 1:
        cpu = cpu_baseline(pool, key, args.cpu_per_core, "2048-bit", core_info)
    if pool is not None:
        pool.close()
    line = {
        "metric": "paillier_raw_encrypts_per_sec_2048", "value": enc_per_s, "unit": "encrypts/s",
        "decrypt": {"value": dec_per_s, "unit": "decrypts/s", "ms_per_step": dec_ms},
        "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": enc_ms,
        "step_ms_enc_plus_dec": enc_ms + dec_ms, "step_ms_spread": head["spread"], "wall_s_timed_region": head["t_wall"],
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "u32 limbs (exact integer)", "data": "synthetic",
        "config": {"workload": "configs[1]: 2048-bit key, raw_encrypt + raw_decrypt, batch %d per GPU" % B, "key_bits": KEY_BITS,
                   "batch_per_gpu": B, "parallelism": "batch sharded over %d GPU(s), no data-path collective" % world,
                   "inputs": "m, r uniform in [1, n) (pai_random_lt_n, seeded)",
                   "rows_per_wave": {"encrypt": head["wave_enc"], "decrypt": head["wave_dec"]},
                   "l2": "256 MiB flush between timed iterations; inputs (%.0f MB) exceed L2" % (B * (2 * ln + lc) * 4 / 1e6)},
        "roofline": roofline, "cpu_baseline": cpu, "e2e": head["e2e"], "e2e_python": head["e2e_python"], "parity": head["parity"],
        "gpu_launches": head["launches"], "clocks": clocks,
        "targets": {"encrypts_per_s_1gpu": 1e5, "decrypts_per_s_1gpu": 2e5},
        "wall_s_total": time.perf_counter() - t_all,
    }
    line.update(extras)
    _emit(line)
    if dev.dist is not None:
        dev.dist.destroy_process_group()


if __name__ == "__main__":
    main()
