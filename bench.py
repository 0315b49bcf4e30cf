#!/usr/bin/env python
"""bench.py — create_proof-schedule benchmark for the B200 back end (BASELINE.json metric:
"create_proof ms + MSM G1-pairs/s at k=19 ECDSA").

One "step" = one pass of the prover hot path for ONE proof of a halo2-lib benchmark circuit: the witness-column
assignment (`assign_witnesses` / `LookupAnyManager::assign_raw`), every MSM of size 2^k and every (coset) NTT
create_proof issues for that constraint system (SURVEY.md §3.3 / §8 table, restated — the prover crate is not
vendored).  The headline workload is BASELINE.json configs[2] (secp256k1 ECDSA, k=19, 1 advice / q_lookup / 1 fixed,
halo2-ecc/configs/secp256k1/bench_ecdsa.config:1); the other four BASELINE configs are run as a short sweep and
reported under `extra.configs` of the same JSON line.  `value` is the MSM throughput of the whole step (G1 pairs /
step time); `ms_per_step` is the create_proof-schedule time.

Every line proves its own outputs (outside the timed regions): all commitments of the resident step and of the
end-to-end step are compared with the closed form  sum_i s_i * (a0 + d*i) mod r * G  (the bases are that arithmetic
progression of multiples of G; SURVEY.md §8(c) L1) computed with Python integers, at every N after the all-reduce;
one polynomial is taken through lagrange_to_coeff -> coeff_to_extended -> extended_to_coeff and checked against
Horner evaluations at domain points.  A mismatch exits with status 3 and prints no JSON line.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--config 1..5] [--sweep 1,2,4,5|none]
                    [--dump-outputs DIR]

`--steps` is the number of timed steps of each step timing of the headline config (resident step in both transform
placements, resident proof, host-buffer step); the per-op timings take 3 repetitions and the sweep extras 2-3 steps each.
`--dump-outputs DIR` writes what the last timed resident step computed to DIR/<name>.npy (see `Workload.outputs`).
"""
from __future__ import annotations
import argparse
import atexit
import json
import math
import os
import shutil
import subprocess
import sys
import tempfile
import threading
import time

sys.dont_write_bytecode = True  # the tree may be read-only: nothing is cached next to the sources
ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import numpy as np

R_MOD = 0x30644E72E131A029B85045B68181585D2833E84879B9709143E1F593F0000001  # Fr
P_MOD = 0x30644E72E131A029B85045B68181585D97816A916871CA8D3C208C16D87CFD47  # Fq
ZETA = 0x30644E72E131A029048B6E193FD84104CC37A73FEC2BC5E9B8CA0B2D36636F23   # Fr cube root of unity (coset generator)
ROOT_OF_UNITY = pow(7, (R_MOD - 1) >> 28, R_MOD)
MONT_RINV_R = pow(1 << 256, -1, R_MOD)
MONT_RINV_P = pow(1 << 256, -1, P_MOD)
UNUSABLE_ROWS = 20  # the benches call calculate_params(Some(20)) (halo2-base/benches/*.rs, secp256k1/tests/ecdsa.rs:122)
BASES = {"monomial": (3, 5), "lagrange": (7, 11)}  # basis -> (a0, d): P_i = (a0 + d*i) * G

# ---- the five BASELINE.json configs: column shapes from the reference's config files (SURVEY.md §8 table)
CONFIGS = {
    1: dict(name="halo2-base inner_product bench", k=14, A=1, L=0, F=1, n_lk=0, d=3,
            src="halo2-base/benches/inner_product.rs:23-49"),
    2: dict(name="halo2-ecc fp_mul bench (BN254 Fq non-native mul)", k=16, A=8, L=2, F=1, n_lk=2, d=4,
            src="halo2-ecc/benches/fp_mul.rs:29-45 (shape by analogy with configs/secp256k1/bench_ecdsa.config:4)"),
    3: dict(name="halo2-ecc secp256k1 ECDSA verify circuit", k=19, A=1, L=0, F=1, n_lk=1, d=5,
            src="halo2-ecc/configs/secp256k1/bench_ecdsa.config:1"),
    4: dict(name="halo2-ecc variable-base MSM circuit (100 BN254 G1 points)", k=20, A=11, L=2, F=1, n_lk=2, d=4,
            src="halo2-ecc/configs/bn254/bench_msm.config:5"),
    5: dict(name="halo2-ecc BN254 pairing circuit", k=23, A=1, L=0, F=1, n_lk=1, d=5,
            src="halo2-ecc/configs/bn254/bench_pairing.config:9 (k=22 row extrapolated)"),
}


class Schedule:
    """The restated create_proof schedule of one constraint system (SURVEY.md §3.3): which MSMs / transforms exist,
    in which transcript phase, over which basis, with which scalar class (witness-like columns are dominated by 0/1
    bits and <= 88-bit limbs, SURVEY.md §8d)."""

    def __init__(self, cfg_id: int, k: int | None = None):
        c = dict(CONFIGS[cfg_id])
        if k is not None:
            c["k"] = k
        self.cfg_id, self.cfg = cfg_id, c
        self.k, self.A, self.L, self.F, self.n_lk, self.d = c["k"], c["A"], c["L"], c["F"], c["n_lk"], c["d"]
        self.n = 1 << self.k
        self.c_adv = self.A + self.L                                   # committed advice columns (gate + lookup advice)
        self.n_pm = -(-(self.A + self.L + self.F) // (self.d - 2))     # permutation product columns, chunks of d - 2
        self.ext_k = self.k + max(1, math.ceil(math.log2(self.d - 1)))  # EvaluationDomain::new(j = d, k)
        ph = [
            [("lagrange", "witness", "advice")] * self.c_adv,                                  # step 2
            [("lagrange", "witness", "permuted")] * (2 * self.n_lk),                           # step 3
            [("lagrange", "uniform", "product")] * (self.n_pm + self.n_lk) + [("monomial", "uniform", "random")],  # 4, 5
            [("monomial", "uniform", "h")] * (self.d - 1),                                     # step 6
            [("monomial", "uniform", "shplonk")],                                              # step 8
            [("monomial", "uniform", "shplonk")],
        ]
        self.msm, self.phases = [], []
        for p in ph:
            if not p:
                continue
            self.phases.append(list(range(len(self.msm), len(self.msm) + len(p))))
            self.msm.extend(p)
        # polynomials that go through lagrange_to_coeff + coeff_to_extended: advice, permuted, products (step 6);
        # ntt_ready[phase] = polynomials that exist when that commitment phase starts
        self.n_poly = self.c_adv + 2 * self.n_lk + self.n_pm + self.n_lk
        self.ntt_ready, pos = {}, 0
        for tag, cnt in (("advice", self.c_adv), ("permuted", 2 * self.n_lk), ("product", self.n_pm + self.n_lk)):
            if cnt:  # index in self.phases of the commitment phase that carries these polynomials
                ph_idx = next(i for i, p in enumerate(self.phases) if self.msm[p[0]][2] == tag)
                self.ntt_ready[ph_idx] = list(range(pos, pos + cnt))
            pos += cnt
        self.h_phase = next(i for i, p in enumerate(self.phases) if self.msm[p[0]][2] == "h")
        self.pairs = len(self.msm) * self.n

    def describe(self, gpus):
        c = self.cfg
        lk = "q_lookup on the gate column" if (self.L == 0 and self.n_lk) else f"{self.L} lookup advice"
        return {
            "workload": f"{c['name']}, k={self.k} (BASELINE.json configs[{self.cfg_id - 1}]; {c['src']}): create_proof schedule restated in SURVEY.md §3.3/§8",
            "k": self.k, "columns": f"{self.A} advice / {lk} / {self.F} fixed", "degree": self.d,
            "msm": f"{len(self.msm)} x 2^{self.k} ({sum(1 for b, _, _ in self.msm if b == 'lagrange')} lagrange + {sum(1 for b, _, _ in self.msm if b == 'monomial')} monomial basis) in phases {[len(p) for p in self.phases]}",
            "ntt": f"{self.n_poly} x iNTT(2^{self.k}) + {self.n_poly} x coeff_to_extended(2^{self.ext_k}) + 1 x extended_to_coeff(2^{self.ext_k})",
            "assignment": f"{self.A} gate column(s) with break points + {self.L} lookup column(s) x 2^{self.k} rows (the commitments of phase 0 read the assigned columns)",
            "scalars": f"{sum(1 for _, c2, _ in self.msm if c2 == 'witness')} witness-like + {sum(1 for _, c2, _ in self.msm if c2 == 'uniform')} uniform columns (SURVEY.md §8d)",
            "overlap": ("the MSMs of a transcript phase share grouped sort / accumulate / bucket-reduction pipelines on up to 3 lanes (bucket reductions on high-priority streams); "
                        + ("the iNTT + coset NTT of a polynomial run on a side stream from the moment the polynomial exists and are joined before extended_to_coeff / the h(X) commitments"
                           if (self.n // max(gpus, 1)) >= (1 << 18) else
                           "MSM shards below 2^18 points are latency-bound chains, so the transforms run in one block before extended_to_coeff / the h(X) commitments instead of beside the phases")),
            "parallelism": (f"msm point-range sharded x{gpus} + fused NVLink peer all-reduce of the partial sums (one kernel per phase); NTT one polynomial per device" if gpus > 1 else "single GPU"),
            "l2_policy": "inputs larger than L2: distinct scalar columns + two multi-level base tables + NTT buffers per step exceed the 126 MB L2 (k >= 16); smaller configs are sweep extras, not the headline",
        }


def witness_like(rng, n):
    """canonical ints: 35% zero, 25% one, 30% < 2^88, 10% uniform Fr (SURVEY.md §8d distribution W)"""
    cls = rng.random(n)
    out = np.zeros((n, 4), dtype=np.uint64)
    one = (cls >= 0.35) & (cls < 0.60)
    small = (cls >= 0.60) & (cls < 0.90)
    full = cls >= 0.90
    out[one, 0] = 1
    k = int(small.sum())
    out[small, 0] = rng.integers(0, 1 << 63, size=k, dtype=np.int64).astype(np.uint64) * np.uint64(2) + rng.integers(0, 2, size=k, dtype=np.int64).astype(np.uint64)
    out[small, 1] = rng.integers(0, 1 << 24, size=k, dtype=np.int64).astype(np.uint64)
    k = int(full.sum())
    out[full] = uniform_residues(rng, k)
    return out


def uniform_residues(rng, n):
    """n uniform values < 2^252 < r as 4 x u64 limbs (valid Montgomery residues and valid canonical values)"""
    a = rng.integers(0, 1 << 63, size=(n, 4), dtype=np.int64).astype(np.uint64)
    a[:, :3] = a[:, :3] * np.uint64(2) + rng.integers(0, 2, size=(n, 3), dtype=np.int64).astype(np.uint64)
    a[:, 3] &= np.uint64((1 << 60) - 1)
    return a


# ------------------------------------------------------------------------------------------------ self-verification
# Independent of the library and of oracle/: plain Python integers and numpy sums.
def limbs_to_int(l):
    return sum(int(v) << (64 * i) for i, v in enumerate(l))


def progression_dot(mont_limbs: np.ndarray, a0: int, d: int, begin: int) -> int:
    """sum_i m_i * (a0 + d * (begin + i)) as an exact integer, m_i the 256-bit values held in the limbs (numpy: 16-bit
    limb columns, S0 = sum m, S1 = sum i*m; every partial sum stays below 2^63 for n <= 2^23)"""
    a = np.ascontiguousarray(mont_limbs, dtype=np.uint64).reshape(-1, 4)
    n = len(a)
    assert begin + n <= (1 << 23) + 1, "progression_dot: index range would overflow the u64 partial sums"
    s0 = np.zeros(16, dtype=np.uint64)
    s1 = np.zeros(16, dtype=np.uint64)
    step = 1 << 18
    for lo in range(0, n, step):
        chunk = a[lo:lo + step].view(np.uint16).reshape(-1, 16).astype(np.uint64)
        idx = np.arange(begin + lo, begin + lo + len(chunk), dtype=np.uint64)
        s0 += chunk.sum(axis=0, dtype=np.uint64)
        s1 += (chunk * idx[:, None]).sum(axis=0, dtype=np.uint64)
    return sum((a0 * int(s0[j]) + d * int(s1[j])) << (16 * j) for j in range(16))


def ec_mul_g(s: int):
    """s * G on y^2 = x^3 + 3 over Fq, G = (1, 2); Jacobian double-and-add on Python ints; returns affine or None"""
    s %= R_MOD
    if s == 0:
        return None
    X, Y, Z = 1, 2, 1
    for bit in bin(s)[3:]:
        # double (a = 0)
        A = X * X % P_MOD; B = Y * Y % P_MOD; C = B * B % P_MOD
        D = 2 * ((X + B) * (X + B) - A - C) % P_MOD
        E = 3 * A % P_MOD
        X3 = (E * E - 2 * D) % P_MOD
        Y3 = (E * (D - X3) - 8 * C) % P_MOD
        Z3 = 2 * Y * Z % P_MOD
        X, Y, Z = X3, Y3, Z3
        if bit == "1":  # mixed add of (1, 2); the doubling / cancellation cases cannot occur for 0 < s < r mid-ladder
            Z2 = Z * Z % P_MOD
            U2 = Z2 % P_MOD; S2 = 2 * Z * Z2 % P_MOD
            H = (U2 - X) % P_MOD; Rr = (S2 - Y) % P_MOD
            if H == 0:
                raise ArithmeticError("ec_mul_g: unexpected doubling inside the ladder")
            H2 = H * H % P_MOD; H3 = H * H2 % P_MOD; V = X * H2 % P_MOD
            X3 = (Rr * Rr - H3 - 2 * V) % P_MOD
            Y3 = (Rr * (V - X3) - Y * H3) % P_MOD
            Z3 = Z * H % P_MOD
            X, Y, Z = X3, Y3, Z3
    zi = pow(Z, -1, P_MOD)
    return (X * zi * zi % P_MOD, Y * zi * zi * zi % P_MOD)


def point_matches(xyz_limbs, expect) -> bool:
    """xyz_limbs: 12 u64 (Jacobian, Montgomery) as the library returns them; expect: affine ints or None"""
    v = np.asarray(xyz_limbs, dtype=np.uint64).reshape(3, 4)
    X, Y, Z = (limbs_to_int(v[i]) * MONT_RINV_P % P_MOD for i in range(3))
    if expect is None:
        return Z == 0
    if Z == 0:
        return False
    z2 = Z * Z % P_MOD
    return X == expect[0] * z2 % P_MOD and Y == expect[1] * z2 * Z % P_MOD


def horner_mont(coeff_limbs: np.ndarray, x: int) -> int:
    """sum_j c_j x^j mod r for Montgomery-limb coefficients; returns the canonical value"""
    acc = 0
    for row in coeff_limbs[::-1]:
        acc = (acc * x + (int(row[0]) | (int(row[1]) << 64) | (int(row[2]) << 128) | (int(row[3]) << 192))) % R_MOD
    return acc * MONT_RINV_R % R_MOD


# ------------------------------------------------------------------------------------------------ --dump-outputs
# Outputs are written as canonical integers (out of Montgomery form, points in affine form), so that two builds that
# represent the same values differently still compare equal.  Each 256-bit value is 8 little-endian 32-bit limbs, held
# exactly in float64.
DUMP_ROWS = 8192         # rows per column / polynomial: a fixed, seeded sample of the longer ones
DUMP_LIMIT = 64 << 20    # bytes in all (config 4, the widest schedule, writes about 32 MB)


def dump_rows(n: int) -> np.ndarray:
    """the sorted row indices written for an output of n rows (the same on every run)"""
    if n <= DUMP_ROWS:
        return np.arange(n)
    return np.sort(np.random.default_rng(0xD0D0).choice(n, DUMP_ROWS, replace=False))


def ints_to_limbs32(vals) -> np.ndarray:
    return np.frombuffer(b"".join(v.to_bytes(32, "little") for v in vals), dtype=np.uint32).astype(np.float64).reshape(-1, 8)


def fr_canonical(mont_limbs: np.ndarray) -> np.ndarray:
    """Montgomery Fr elements (m x 4 u64) -> their values, m x 8 limbs"""
    buf = np.ascontiguousarray(mont_limbs, dtype=np.uint64).tobytes()
    return ints_to_limbs32([int.from_bytes(buf[i:i + 32], "little") * MONT_RINV_R % R_MOD for i in range(0, len(buf), 32)])


def g1_affine(xyz_limbs) -> np.ndarray:
    """one G1 point as the library returns it (12 u64, Jacobian, Montgomery) -> affine (x, y), 16 limbs; the identity
    is all zeros ((0, 0) is not on the curve)"""
    X, Y, Z = (limbs_to_int(r) * MONT_RINV_P % P_MOD for r in np.asarray(xyz_limbs, dtype=np.uint64).reshape(3, 4))
    if Z == 0:
        return ints_to_limbs32([0, 0]).reshape(16)
    zi = pow(Z, -1, P_MOD)
    return ints_to_limbs32([X * zi * zi % P_MOD, Y * zi * zi * zi % P_MOD]).reshape(16)


def write_outputs(outputs: dict, d: str):
    total = sum(a.nbytes for a in outputs.values())
    assert total <= DUMP_LIMIT, f"--dump-outputs: {total} bytes exceed the {DUMP_LIMIT}-byte limit"
    os.makedirs(d, exist_ok=True)
    for name, a in outputs.items():
        np.save(os.path.join(d, name + ".npy"), a)


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""

    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, gpu_index):
        self.rows, self.proc, self.idx = [], None, gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-i", str(self.idx), "-lms", "50"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, smax, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0]))
                smax = float(f[1])
            except ValueError:
                continue
            for nm, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": smax, "samples": len(sm), "reasons": sorted(reasons)}


def measured_hbm_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


# ------------------------------------------------------------------------------------------------ CPU arm
def host_cpu_info(threads):
    """what the CPU arm could actually use: affinity mask, cgroup quota, OpenMP placement (VERDICT r1 weak #7)"""
    info = {"nproc_affinity": threads, "os_cpu_count": os.cpu_count()}
    try:
        txt = open("/sys/fs/cgroup/cpu.max").read().split()
        info["cgroup_cpu_max"] = " ".join(txt)
        if txt[0] != "max":
            info["cgroup_cpus"] = float(txt[0]) / float(txt[1])
    except Exception:
        info["cgroup_cpu_max"] = None
    for v in ("OMP_PLACES", "OMP_PROC_BIND", "OMP_NUM_THREADS"):
        info[v] = os.environ.get(v)
    try:
        for line in open("/proc/cpuinfo"):
            if line.startswith("model name"):
                info["cpu_model"] = line.split(":", 1)[1].strip()
                break
    except Exception:
        pass
    return info


def cpu_sample(sched: Schedule, threads: int | None = None, reps: int = 3):
    """Times the CPU restatement (oracle/, OpenMP, all host threads) on one op of each class of the schedule and
    composes the step time: sum(count_i * t_i).  Every op is repeated `reps` times per thread count; the minimum is
    used, min / median are reported.  ~10-30 s of CPU work on a typical host at k=19."""
    from oracle import oracle as orc
    try:  # a -march=native build for the host it runs on (the shipped .so is x86-64-v3), outside the (possibly read-only) tree
        tmp = tempfile.mkdtemp(prefix="h2b_oracle_")
        atexit.register(shutil.rmtree, tmp, True)
        so = os.path.join(tmp, "liboracle_native.so")
        subprocess.check_call(["make", "-C", os.path.join(ROOT, "oracle"), "-s", "MARCH=native", f"OUT={so}"], stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)
        orc._lib = None
        orc._SO = so
    except Exception:
        pass
    if threads is None:  # all host cores this process may use (torchrun exports OMP_NUM_THREADS=1: ignore it)
        try:
            threads = len(os.sched_getaffinity(0))
        except Exception:
            threads = os.cpu_count() or 1
    info = host_cpu_info(threads)
    if info.get("cgroup_cpus"):
        threads = max(1, min(threads, int(math.ceil(info["cgroup_cpus"]))))
    # SMT siblings hurt this integer code on some hosts: every op is timed with all logical CPUs and with half of
    # them, and the faster one is kept (a tuned CPU run would do the same)
    cand = sorted({threads, max(1, threads // 2)}, reverse=True)
    orc.set_threads(threads)
    orc.use_fast_ntt(True)  # many-core four-step NTT (oracle/bn254_oracle.c: orc_ntt_fast)
    k, n, ext_k = sched.k, sched.n, sched.ext_k
    rng = np.random.default_rng(0xB2000000 + k)
    # bases: any valid curve points time the same; build n points a_i * G cheaply with the oracle itself
    from util import affine_to_limbs
    from oracle import pyref
    g = affine_to_limbs([pyref.G1])[0]
    small = np.zeros((n, 4), dtype=np.uint64)
    small[:, 0] = np.arange(3, 3 + 5 * n, 5, dtype=np.uint64)  # canonical small scalars
    t0 = time.perf_counter()
    bases = orc.g1_fixed_base_mul(orc.to_mont(orc.FR, small), g)
    t_setup = time.perf_counter() - t0
    s_uni = uniform_residues(rng, n)
    s_wit = orc.to_mont(orc.FR, witness_like(rng, n))
    # warm the OpenMP pool and the code paths on a tiny instance before timing anything
    orc.msm_pippenger(s_uni[:256], bases[:256], threads)
    orc.extended_to_coeff(orc.coeff_to_extended(orc.lagrange_to_coeff(s_uni[:256], 8, threads), 10, threads), 10, threads)
    times, used, samples = {}, {}, {}
    a = uniform_residues(rng, n)

    def best(name, fn, reps=reps):
        res = None
        for th in cand:
            for _ in range(reps):
                t0 = time.perf_counter(); r = fn(th); dt = time.perf_counter() - t0
                samples.setdefault(name, {}).setdefault(th, []).append(dt)
                if name not in times or dt < times[name]:
                    times[name], used[name] = dt, th
                res = r
        return res
    msm_fn = getattr(orc, "msm_best", None) or orc.msm_pippenger  # fastest CPU variant the oracle offers
    best("msm_uniform", lambda th: msm_fn(s_uni, bases, th))
    best("msm_witness", lambda th: msm_fn(s_wit, bases, th))
    coeffs = best("intt", lambda th: orc.lagrange_to_coeff(a, k, th))
    ext = best("coset_ntt", lambda th: orc.coeff_to_extended(coeffs, ext_k, th))
    best("coset_intt", lambda th: orc.extended_to_coeff(ext, ext_k, th))
    best("assign", lambda th: orc.assign_witnesses(a[: n - UNUSABLE_ROWS], np.zeros(0, dtype=np.uint64), k, 1))
    orc.use_fast_ntt(False)
    n_wit = sum(1 for _, c, _ in sched.msm if c == "witness")
    n_uni = len(sched.msm) - n_wit
    step_s = (n_uni * times["msm_uniform"] + n_wit * times["msm_witness"] + sched.n_poly * (times["intt"] + times["coset_ntt"])
              + times["coset_intt"] + (sched.A + sched.L) * times["assign"])
    # achieved multi-thread scaling of the MSM: best time at the larger thread count vs at half of it
    scal = None
    if len(cand) == 2:
        tm = {th: min(v) for th, v in samples["msm_uniform"].items()}
        scal = {"threads": cand, "msm_uniform_speedup_full_vs_half": tm[cand[1]] / tm[cand[0]]}
    return {
        "value": sched.pairs / step_s,
        "unit": "G1 pairs/s",
        "cores": threads,
        "threads_used": used,
        "kind": "port",
        "sample": (f"oracle/bn254_oracle.c (restated CPU path, OpenMP, best of {cand} threads per op, min of {reps} repetitions; the Rust reference cannot be built here): one MSM(2^{k}) per scalar "
                   f"class + one iNTT(2^{k}) + one coeff_to_extended/extended_to_coeff(2^{ext_k}) + one assignment, composed by the schedule counts"),
        "step_ms": step_s * 1e3,
        "op_ms": {kk: v * 1e3 for kk, v in times.items()},
        "op_ms_median": {kk: float(np.median([x for lst in v.values() for x in lst])) * 1e3 for kk, v in samples.items()},
        "host": info,
        "thread_scaling": scal,
        "setup_s": t_setup,
    }


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    sched = Schedule(args.config, args.k)
    vals, last = [], None
    for i in range(args.warmup + args.steps):
        last = cpu_sample(sched, reps=1 if args.steps + args.warmup > 2 else 3)
        if i >= args.warmup:
            vals.append(last)
    step_ms = float(np.mean([v["step_ms"] for v in vals]))
    value = sched.pairs / (step_ms / 1e3)
    cb = dict(last)
    cb["value"] = value
    print(json.dumps({
        "impl": "reference", "metric": metric_name(sched), "value": value, "unit": "G1 pairs/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": step_ms, "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "u32x8 (254-bit Montgomery integers)", "data": "synthetic",
        "config": sched.describe(args.gpus), "cpu_baseline": cb,
        "e2e": {"value": value, "unit": "G1 pairs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "create_proof_schedule_ms": step_ms,
    }))


def metric_name(sched):
    names = {1: "inner_product", 2: "fp_mul", 3: "ECDSA", 4: "MSM circuit", 5: "pairing"}
    return "msm_g1_pairs_per_s (create_proof schedule, %s k=%d)" % (names[sched.cfg_id], sched.k)


# ------------------------------------------------------------------------------------------------ GPU arm
# experiment switch: small shards run their transforms in the BACKGROUND of the commitment phases with this many CTAs per SM
BENCH_BG_NTT = int(os.environ.get("H2B_BENCH_BG_NTT", "0"))


class Rig:
    """process-wide GPU plumbing shared by every workload of one bench.py run"""

    def __init__(self, args):
        import torch
        import halo2_lib_b200 as h
        self.torch, self.h = torch, h
        self.rank = int(os.environ.get("RANK", "0"))
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.local_rank = int(os.environ.get("LOCAL_RANK", "0"))
        assert self.world == args.gpus, f"--gpus {args.gpus} but WORLD_SIZE={self.world}"
        torch.cuda.set_device(self.local_rank)
        self.dev = torch.device("cuda", self.local_rank)
        self.dist = None
        if self.world > 1:
            import torch.distributed as dist
            self.dist = dist
            # NCCL prints its version banner to stdout when the communicator is created: keep stdout for the ONE JSON line
            sys.stdout.flush()
            saved_fd = os.dup(1)
            os.dup2(2, 1)
            try:
                dist.init_process_group("nccl", device_id=self.dev)
                dist.barrier()
                torch.cuda.synchronize()
            finally:
                sys.stdout.flush()
                os.dup2(saved_fd, 1)
                os.close(saved_fd)
        self.ctx = h.Context(self.local_rank)
        # a dedicated non-default stream: the library treats a NULL stream as "use the context's own stream", and the
        # CUDA events below must be recorded on the stream the kernels are launched on
        # (higher priority than the transform stream below: the transforms fill the bubbles the MSM pipeline leaves)
        self.stream = torch.cuda.Stream(device=self.dev, priority=-1 if os.environ.get("H2B_BENCH_PRIORITY", "1") != "0" else 0)
        torch.cuda.set_stream(self.stream)
        assert self.stream.cuda_stream != 0
        self.ctx.set_stream(self.stream.cuda_stream)
        # second context + stream on the same GPU: the polynomial transforms of a column run beside the commitment
        # phases that do not depend on them (see step_resident)
        self.ctx_ntt = h.Context(self.local_rank)
        self.stream_ntt = torch.cuda.Stream(device=self.dev)
        self.ctx_ntt.set_stream(self.stream_ntt.cuda_stream)
        if BENCH_BG_NTT:
            self.ctx_ntt.set_option("ntt.max_ctas_per_sm", BENCH_BG_NTT)
        if self.world > 1:
            h.connect_peers(self.ctx)  # NVLink mailboxes for the fused all-reduce of partial commitments (csrc/peer.cu)

    def barrier(self):
        if self.dist:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def launches(self):
        return self.ctx.kernel_launches + self.ctx_ntt.kernel_launches

    def timed(self, fn, steps, warmup, prof=None):
        torch = self.torch
        for _ in range(warmup):
            fn()
        self.barrier()
        if prof:
            self.ctx.profile_reset()
            self.ctx.profile_enable(prof)
        l0 = self.launches()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(self.stream)
        for _ in range(steps):
            fn()
        e1.record(self.stream)
        self.barrier()
        ms = e0.elapsed_time(e1)
        if prof:
            self.ctx.profile_enable(None)
        t = torch.tensor([ms], dtype=torch.float64, device=self.dev)
        if self.dist:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item()) / steps, self.launches() - l0

    def time_op(self, fn, reps=3):
        torch = self.torch
        fn(); torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(self.stream)
        for _ in range(reps):
            fn()
        b.record(self.stream); torch.cuda.synchronize()
        return a.elapsed_time(b) / reps

    def all_true(self, ok: bool) -> bool:
        if not self.dist:
            return ok
        t = self.torch.tensor([1 if ok else 0], dtype=self.torch.int32, device=self.dev)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MIN)
        return bool(t.item())

    def sum_ints(self, vals: list[int]) -> list[int]:
        """element-wise sum over ranks of a list of (huge) Python ints"""
        if not self.dist:
            return vals
        got = [None] * self.world
        self.dist.all_gather_object(got, [hex(v) for v in vals])
        return [sum(int(g[j], 16) for g in got) for j in range(len(vals))]


class Workload:
    """device- and host-resident inputs of one schedule + the two step functions"""

    def __init__(self, rig: Rig, sched: Schedule, want_e2e: bool, fault: str | None = None):
        import ctypes as C
        torch, h = rig.torch, rig.h
        from halo2_lib_b200._capi import lib
        self.rig, self.s, self.lib, self.C, self.fault = rig, sched, lib, C, fault
        self.want_e2e = want_e2e
        ctx, dev, world, rank = rig.ctx, rig.dev, rig.world, rig.rank
        k, n, ext_k = sched.k, sched.n, sched.ext_k
        self.begin, self.n_loc = h.shard_range(n, rank, world)
        begin, n_loc = self.begin, self.n_loc
        rng = np.random.default_rng(0xB2000000 + 97 * sched.cfg_id + k)
        vp = C.c_void_p

        def dev_u64(arr):
            return torch.from_numpy(arr.view(np.int64)).to(dev)

        # ---- setup (untimed): SRS-like bases on the GPU, this rank's shard only: P_i = (a0 + d*i) * G
        gbase = np.array([0xd35d438dc58f0d9d, 0x0a78eb28f5c70b3d, 0x666ea36f7879462c, 0x0e0a77c19a07df2f,  # x = 1 (Montgomery)
                          0xa6ba871b8b1e1b3a, 0x14f1d651eb8e167b, 0xccdd46def0f28c58, 0x1c14ef83340fbe5e], dtype=np.uint64)  # y = 2
        tables = {}
        for name, (a0, d) in BASES.items():
            sc = np.zeros((n_loc, 4), dtype=np.uint64)
            sc[:, 0] = (a0 + d * (begin + np.arange(n_loc, dtype=np.uint64))).astype(np.uint64)
            sc_m = ctx.field_op(1, 5, sc)  # to Montgomery form on the GPU
            d_sc = dev_u64(sc_m)
            d_pts = torch.empty((n_loc, 8), dtype=torch.int64, device=dev)
            ctx.check(lib.h2b_g1_fixed_base_mul_dev(ctx.h, vp(gbase.ctypes.data), vp(d_sc.data_ptr()), n_loc, vp(d_pts.data_ptr())))
            tables[name] = d_pts
        torch.cuda.synchronize()
        self.params = h.ParamsKZG(ctx, k, g=tables["monomial"].data_ptr(), g_lagrange=tables["lagrange"].data_ptr(), begin=begin, count=n_loc, device_ptrs=True)
        del tables

        # ---- witness: the virtual column V of the gate advice (A columns, break points as keygen would pin them:
        # every column is filled to within 3 rows of the usable region, SURVEY.md App. A.1) and the looked-up cells
        usable = n - UNUSABLE_ROWS
        A, L = sched.A, sched.L
        self.break_points = np.array([usable - 1 - (c % 3) for c in range(A - 1)], dtype=np.uint64)
        last_len = usable - 5
        n_cells = int(self.break_points.sum()) + last_len
        self.n_cells = n_cells
        v_host = ctx.field_op(1, 5, witness_like(rng, n_cells))  # Montgomery limbs
        self.vcol_host = torch.from_numpy(v_host.view(np.int64)).pin_memory()
        self.vcol_dev = self.vcol_host.to(dev)
        self.n_lookup = (usable - 7) * L
        if L:
            lk_host = ctx.field_op(1, 5, witness_like(rng, self.n_lookup))
            self.lk_host = torch.from_numpy(lk_host.view(np.int64)).pin_memory()
            self.lk_dev = self.lk_host.to(dev)
        self.acols_dev = torch.zeros((A, n, 4), dtype=torch.int64, device=dev)
        self.lcols_dev = torch.zeros((max(L, 1), n, 4), dtype=torch.int64, device=dev)
        # the columns the assignment must produce, restated on the host with numpy slicing (App. A.2 / A.3)
        exp_cols = []
        starts = np.concatenate([[0], np.cumsum(self.break_points)]).astype(np.int64)
        for c in range(A):
            ln = int(self.break_points[c]) + 1 if c < A - 1 else n_cells - int(starts[c])
            col = np.zeros((n, 4), dtype=np.uint64)
            col[:ln] = v_host[int(starts[c]): int(starts[c]) + ln]
            exp_cols.append(col)
        for c in range(L):
            col = np.zeros((n, 4), dtype=np.uint64)
            part = lk_host[c::L]
            col[: len(part)] = part
            exp_cols.append(col)

        # ---- scalar columns of every MSM.  Advice commitments read the assigned columns; the others get their own
        # synthetic column.  expect_dot[j] = this rank's share of sum_i m_i * (a0 + d*i)  (closed form, Python ints)
        self.cols_host, self.cols_dev, self.col_ptr = [], [], []
        expect_dot = []
        self.basis_id = [0 if b == "monomial" else 1 for b, _, _ in sched.msm]
        for j, (basis, cls, tag) in enumerate(sched.msm):
            a0, d = BASES[basis]
            if tag == "advice":
                full = exp_cols[j]
                if j < A:
                    self.col_ptr.append(self.acols_dev[j].data_ptr() + begin * 32)
                else:
                    self.col_ptr.append(self.lcols_dev[j - A].data_ptr() + begin * 32)
                self.cols_host.append(None)
                self.cols_dev.append(None)
            else:
                full = uniform_residues(rng, n) if cls == "uniform" else ctx.field_op(1, 5, witness_like(rng, n))
                shard = np.ascontiguousarray(full[begin:begin + n_loc])
                th = torch.from_numpy(shard.view(np.int64))
                th = th.pin_memory() if want_e2e else th
                self.cols_host.append(th)
                td = th.to(dev)
                self.cols_dev.append(td)
                self.col_ptr.append(td.data_ptr())
            expect_dot.append(progression_dot(full[begin:begin + n_loc], a0, d, begin))
        del exp_cols
        tot = rig.sum_ints(expect_dot)
        self.expect_scalar = [t * MONT_RINV_R % R_MOD for t in tot]
        self.expect_point = [ec_mul_g(s) for s in self.expect_scalar]

        # ---- polynomials of the transforms (own buffers: the in-place iNTT runs beside the commitments)
        # one polynomial per device: transform i in [0, n_poly) is the iNTT of column i over 2^k, n_poly + i its coset NTT over
        # 2^ext_k, 2 * n_poly the extended_to_coeff; whole transforms are dealt by cost (longest first) so that no device
        # gets two of the 4x larger ones while another has none
        npoly = sched.n_poly
        owners = h.ntt_owners_balanced([1.0] * npoly + [float(1 << (ext_k - k))] * (npoly + 1), world)
        self.my_ntt = lambda i: owners[i] == rank
        mine = [i for i in range(npoly) if self.my_ntt(i) or self.my_ntt(npoly + i)]
        if not mine:  # a rank that owns no column transform (8 GPUs: six own one large transform each) still times the ops
            mine = [0]
        self.polys_dev = {i: dev_u64(uniform_residues(rng, n)) for i in mine}
        self.ext_dev = {i: torch.empty((1 << ext_k, 4), dtype=torch.int64, device=dev) for i in mine}
        if 0 not in self.ext_dev:
            self.ext_dev[0] = torch.empty((1 << ext_k, 4), dtype=torch.int64, device=dev)
        if want_e2e:
            self.polys_host = {i: self.polys_dev[i].cpu().pin_memory() for i in mine}
            self.ext_host = {i: torch.empty((1 << ext_k, 4), dtype=torch.int64).pin_memory() for i in set(mine) | {0}}
            self.acols_host = torch.empty((A, n, 4), dtype=torch.int64).pin_memory()
            self.lcols_host = torch.empty((max(L, 1), n, 4), dtype=torch.int64).pin_memory()
        self.outs_dev = torch.zeros((len(sched.msm), 12), dtype=torch.int64, device=dev)
        self.outs_host = np.zeros((len(sched.msm), 12), dtype=np.uint64)
        self.ev_fork = [torch.cuda.Event() for _ in range(len(sched.phases))]
        self.ev_join = torch.cuda.Event()
        self.bp_arr = (C.c_uint64 * max(1, len(self.break_points)))(*[int(b) for b in self.break_points])
        self.side_pool = None
        self.trace = None

    # -------------------------------------------------------------------------------------------- resident step
    def _ntt_pair_dev(self, ctx, i):
        s, lib, vp = self.s, self.lib, self.C.c_void_p
        if self.my_ntt(i):
            ctx.check(lib.h2b_lagrange_to_coeff_dev(ctx.h, vp(self.polys_dev[i].data_ptr()), s.k))
        if self.my_ntt(s.n_poly + i):
            ctx.check(lib.h2b_coeff_to_extended_dev(ctx.h, vp(self.polys_dev[i].data_ptr()), s.n, s.ext_k, vp(self.ext_dev[i].data_ptr())))

    def assign_dev(self):
        s, lib, vp, ctx = self.s, self.lib, self.C.c_void_p, self.rig.ctx
        nbp = len(self.break_points)
        ctx.check(lib.h2b_assign_columns_dev(ctx.h, vp(self.vcol_dev.data_ptr()), self.n_cells, self.bp_arr if nbp else None, nbp,
                                             s.k, s.A, vp(self.acols_dev.data_ptr())))
        if s.L:
            ctx.check(lib.h2b_assign_lookups_dev(ctx.h, vp(self.lk_dev.data_ptr()), self.n_lookup, s.k, s.L, vp(self.lcols_dev.data_ptr())))

    def step_resident(self, overlap=None):
        """overlap=None: the schedule's own rule — the transforms of a column run beside the next commitment phase when the
        MSM shards are large enough to be throughput-bound (>= 2^18 points per GPU); with small shards the commitment phases
        are chains of latency-bound kernels and a transform beside them only delays every link, so the transforms run in
        one block before the h(X) phase instead."""
        rig, s, lib, vp = self.rig, self.s, self.lib, self.C.c_void_p
        if overlap is None:
            overlap = self.n_loc >= (1 << 18) or BENCH_BG_NTT > 0
        ctx, stream, stream_ntt = rig.ctx, rig.stream, rig.stream_ntt
        # every rank assigns the full columns (it commits its own row range of each of them)
        self.assign_dev()
        for pi, phase in enumerate(s.phases):
            if pi in s.ntt_ready:
                if overlap:
                    self.ev_fork[pi].record(stream)
                    stream_ntt.wait_event(self.ev_fork[pi])
                    for i in s.ntt_ready[pi]:
                        self._ntt_pair_dev(rig.ctx_ntt, i)
            elif pi == s.h_phase:
                if overlap:
                    self.ev_join.record(stream_ntt)
                    stream.wait_event(self.ev_join)
                else:
                    for i in range(s.n_poly):
                        self._ntt_pair_dev(ctx, i)
                if self.my_ntt(2 * s.n_poly):
                    ctx.check(lib.h2b_extended_to_coeff_dev(ctx.h, vp(self.ext_dev[0].data_ptr()), s.ext_k))
            j0 = phase[0]
            self.params.commit_batch_dev([self.basis_id[j] for j in phase], [self.col_ptr[j] for j in phase], self.n_loc, self.outs_dev[j0].data_ptr())
            if rig.world > 1 and not (self.fault == "skip_allreduce" and pi == 1):
                # all-reduce under EC addition: one fused kernel over NVLink peer memory, no NCCL call
                for lo in range(0, len(phase), 16):
                    rig.h.allreduce_points(ctx, self.outs_dev[j0 + lo].data_ptr(), min(16, len(phase) - lo))

    # -------------------------------------------------------------------------------------------- end-to-end step
    def _ntt_side_host(self, polys):
        """h2b_lagrange_to_coeff_and_extended_batch on the second context: pinned host buffers in and out, the
        coefficients stay on the device between the two transforms, PCIe legs pipelined against the kernels"""
        s, lib, C, ctx_ntt = self.s, self.lib, self.C, self.rig.ctx_ntt
        npoly = s.n_poly
        both = [i for i in polys if self.my_ntt(i) and self.my_ntt(npoly + i)]
        if both:
            pa = (C.c_void_p * len(both))(*[self.polys_host[i].data_ptr() for i in both])
            pe = (C.c_void_p * len(both))(*[self.ext_host[i].data_ptr() for i in both])
            ctx_ntt.check(lib.h2b_lagrange_to_coeff_and_extended_batch(ctx_ntt.h, pa, len(both), s.k, s.ext_k, pe))
        a = [i for i in polys if self.my_ntt(i) and i not in both]
        if a:
            ptrs = (C.c_void_p * len(a))(*[self.polys_host[i].data_ptr() for i in a])
            ctx_ntt.check(lib.h2b_lagrange_to_coeff_batch(ctx_ntt.h, ptrs, len(a), s.k))
        b = [i for i in polys if self.my_ntt(npoly + i) and i not in both]
        if b:
            pin = (C.c_void_p * len(b))(*[self.polys_host[i].data_ptr() for i in b])
            pout = (C.c_void_p * len(b))(*[self.ext_host[i].data_ptr() for i in b])
            ctx_ntt.check(lib.h2b_coeff_to_extended_batch(ctx_ntt.h, pin, len(b), s.n, s.ext_k, pout))

    def _mark(self, label):
        if self.trace is not None:
            self.trace.append((label, time.perf_counter()))

    def step_e2e(self, overlap=True):
        """the same step through the host-pointer C ABI: pinned host buffers in, host buffers out.  With `overlap` a second
        host thread drives the transforms of the polynomials that already exist (same dependency model as step_resident)
        through a second context, so their PCIe traffic runs beside the commitment phases."""
        rig, s, lib, C = self.rig, self.s, self.lib, self.C
        vp, ctx = C.c_void_p, rig.ctx
        if self.side_pool is None:
            from concurrent.futures import ThreadPoolExecutor
            self.side_pool = ThreadPoolExecutor(max_workers=1)  # drives the transform context (ctypes drops the GIL)
        self._mark("start")
        nbp = len(self.break_points)
        ctx.check(lib.h2b_assign_columns(ctx.h, vp(self.vcol_host.data_ptr()), self.n_cells, self.bp_arr if nbp else None, nbp,
                                         s.k, s.A, vp(self.acols_host.data_ptr())))
        if s.L:
            ctx.check(lib.h2b_assign_lookups(ctx.h, vp(self.lk_host.data_ptr()), self.n_lookup, s.k, s.L, vp(self.lcols_host.data_ptr())))
        self._mark("assign")
        pending = []
        for pi, phase in enumerate(s.phases):
            if pi in s.ntt_ready:
                if overlap:
                    pending.append(self.side_pool.submit(self._ntt_side_host, s.ntt_ready[pi]))
            elif pi == s.h_phase:
                if overlap:
                    for f in pending:
                        f.result()
                else:
                    self._ntt_side_host(list(range(s.n_poly)))
                self._mark("join_side")
                if self.my_ntt(2 * s.n_poly):
                    ctx.check(lib.h2b_extended_to_coeff(ctx.h, vp(self.ext_host[0].data_ptr()), s.ext_k))
                self._mark("ext_to_coeff")
            m = len(phase)
            host_ptr = []
            for j in phase:
                if self.cols_host[j] is not None:
                    host_ptr.append(self.cols_host[j].data_ptr())
                elif j < s.A:
                    host_ptr.append(self.acols_host[j].data_ptr() + self.begin * 32)
                else:
                    host_ptr.append(self.lcols_host[j - s.A].data_ptr() + self.begin * 32)
            ptrs = (C.c_void_p * m)(*host_ptr)
            bs = (C.c_int * m)(*[self.basis_id[j] for j in phase])
            out = np.empty((m, 12), dtype=np.uint64)
            # host buffers in, the full commitments out: with peers connected the partial sums of all GPUs are combined
            # by the fused NVLink all-reduce kernel before the one device-to-host copy
            ctx.check(lib.h2b_msm_g1_batch_reduced(ctx.h, self.params.h, bs, ptrs, m, self.n_loc, vp(out.ctypes.data)))
            self.outs_host[phase] = out
            self._mark("phase%d" % pi)

    # -------------------------------------------------------------------------------------------- resident prover (e2e)
    def setup_prover(self):
        """the resident prover path (halo2-lib_b200/prover.py): a SATISFIED synthetic halo2-base circuit of this config's
        shape (A gate-advice / L lookup-advice columns, selector lookup or none); host side = pinned witness cells (virtual
        column + looked-up cells) + pinned random polynomial, everything else lives behind h2b_poly handles"""
        rig, s = self.rig, self.s
        torch, h = rig.torch, rig.h
        rng = np.random.default_rng(0xB2002000 + s.k)
        sel = s.n_lk > 0 and s.L == 0
        inst = h.synthetic_circuit(rig.ctx, s.k, rng, A=s.A, L=s.L, selector_lookup=sel)
        self.pr_circuit = h.Circuit(rig.ctx, s.k, inst["fixed"], inst["sigma"], A=s.A, L=s.L, selector_lookup=sel)
        assert self.pr_circuit.degree == s.d and self.pr_circuit.n_sets == s.n_pm and self.pr_circuit.n_lookups == s.n_lk
        self.pr_session = h.ProverSession(rig.ctx, self.params, self.pr_circuit)
        if rig.world > 1:
            self.pr_session.shard(self.begin, self.n_loc, lambda ptr, m: h.allreduce_points(rig.ctx, ptr, m))
        pin = lambda a: torch.from_numpy(np.ascontiguousarray(a).view(np.int64)).pin_memory()
        self.pr_witness = pin(inst["virtual"])
        self.pr_lookup = pin(inst["lookup"]) if len(inst["lookup"]) else None
        self.pr_random = pin(uniform_residues(rng, s.n))
        self.pr_bp = inst["break_points"]
        self.pr_sel = sel
        self.pr_last = None

    def _prove(self):
        lk = self.pr_lookup
        return self.pr_session.prove(self.pr_witness.data_ptr(), len(self.pr_witness), self.pr_random.data_ptr(), seed=1, break_points=self.pr_bp,
                                     lookup_ptr=lk.data_ptr() if lk is not None else 0, n_lookup=len(lk) if lk is not None else 0)

    def step_e2e_prover(self):
        self.pr_last = self._prove()

    def verify_prover(self) -> dict:
        """one untimed proof with the committed polynomials kept: every commitment against the closed form of its
        polynomial, and the quotient identity at the challenge point (tests/prover_check.py, Python integers)"""
        import prover_check as pc
        s, sess = self.s, self.pr_session
        sess.keep = {}
        res = self._prove()
        kept, sess.keep = sess.keep["committed"], None
        ok = 0
        for cm, (basis, poly) in zip(res["commitments"], kept):
            a0, d = BASES["monomial" if basis == 0 else "lagrange"]
            scalar = progression_dot(poly, a0, d, 0) * MONT_RINV_R % R_MOD
            ok += 1 if point_matches(cm, ec_mul_g(scalar)) else 0
        left, right = pc.quotient_identity(res, s.k, self.pr_circuit.bf, s.A, s.L, self.pr_sel)
        return {"commitments": ok, "of": len(kept), "expected": len(s.msm), "quotient_identity": left == right,
                "h2d_bytes": res["h2d_bytes"], "d2h_bytes": res["d2h_bytes"]}

    def close_prover(self):
        if getattr(self, "pr_session", None) is not None:
            self.pr_session.free()
            self.pr_circuit.free()
            self.pr_session = None

    # -------------------------------------------------------------------------------------------- verification
    def verify_commitments(self, arr) -> int:
        """number of the schedule's commitments in `arr` (len(msm) x 12 limbs) that equal the closed form"""
        arr = np.asarray(arr, dtype=np.uint64).reshape(-1, 12)
        return sum(1 for j in range(len(self.s.msm)) if point_matches(arr[j], self.expect_point[j]))

    def verify_ntt(self) -> dict:
        """one polynomial through the three transforms, each checked against Horner evaluations (Python ints)"""
        rig, s, lib, vp = self.rig, self.s, self.lib, self.C.c_void_p
        torch, ctx = rig.torch, rig.ctx
        rng = np.random.default_rng(0xB2001000 + s.k)
        x = uniform_residues(rng, s.n)
        d_x = torch.from_numpy(x.view(np.int64)).to(rig.dev)
        d_e = torch.empty((1 << s.ext_k, 4), dtype=torch.int64, device=rig.dev)
        ctx.check(lib.h2b_lagrange_to_coeff_dev(ctx.h, vp(d_x.data_ptr()), s.k))
        ctx.check(lib.h2b_coeff_to_extended_dev(ctx.h, vp(d_x.data_ptr()), s.n, s.ext_k, vp(d_e.data_ptr())))
        torch.cuda.synchronize()
        coeffs = d_x.cpu().numpy().view(np.uint64)
        ext = d_e.cpu().numpy().view(np.uint64)
        ctx.check(lib.h2b_extended_to_coeff_dev(ctx.h, vp(d_e.data_ptr()), s.ext_k))
        torch.cuda.synchronize()
        back = d_e.cpu().numpy().view(np.uint64)
        w = pow(ROOT_OF_UNITY, 1 << (28 - s.k), R_MOD)
        we = pow(ROOT_OF_UNITY, 1 << (28 - s.ext_k), R_MOD)
        pts = [1, s.n // 3 + 1] if s.k <= 20 else [s.n // 3 + 1]
        ok_intt = all(horner_mont(coeffs, pow(w, i, R_MOD)) == limbs_to_int(x[i]) * MONT_RINV_R % R_MOD for i in pts)
        i = (1 << s.ext_k) // 5 + 2
        ok_coset = horner_mont(coeffs, ZETA * pow(we, i, R_MOD) % R_MOD) == limbs_to_int(ext[i]) * MONT_RINV_R % R_MOD
        ok_back = bool(np.array_equal(back[: s.n], coeffs)) and not back[s.n:].any()
        return {"lagrange_to_coeff": ok_intt, "coeff_to_extended": ok_coset, "extended_to_coeff_roundtrip": ok_back,
                "points_checked": len(pts) + 1}

    def outputs(self) -> dict:
        """what the last step_resident computed, as its caller receives it (for --dump-outputs):
        commitments       every commitment of the schedule, after the all-reduce (len(msm) x 16)
        assigned_columns  the gate columns, then the lookup columns (A + L, rows, 8)
        coefficients      lagrange_to_coeff of each polynomial whose iNTT this rank runs (rows, 8 each)
        extended          coeff_to_extended of each polynomial whose coset NTT this rank runs, except polynomial 0
        extended_to_coeff extended_to_coeff of polynomial 0's coset evaluations
        The transforms work in place on buffers that persist across steps, so these depend on warmup + steps."""
        torch, s = self.rig.torch, self.s
        torch.cuda.synchronize()

        def rows(t, n):  # (..., n, 4) int64 on the device -> (..., dump rows, 8)
            idx = torch.from_numpy(dump_rows(n)).to(t.device)
            sample = t.index_select(t.dim() - 2, idx).cpu().numpy().view(np.uint64)
            return fr_canonical(sample).reshape(*t.shape[:-2], len(idx), 8)

        npoly, ext_n = s.n_poly, 1 << s.ext_k
        to_coeff = self.my_ntt(2 * npoly) and self.my_ntt(npoly)  # ext_dev[0] holds this rank's coset NTT of polynomial 0
        out = {"commitments": np.stack([g1_affine(c) for c in self.outs_dev.cpu().numpy().view(np.uint64)]),
               "assigned_columns": rows(self.acols_dev, s.n) if not s.L else np.concatenate([rows(self.acols_dev, s.n), rows(self.lcols_dev, s.n)])}
        coeffs = [rows(self.polys_dev[i], s.n) for i in sorted(self.polys_dev) if self.my_ntt(i)]
        ext = [rows(self.ext_dev[i], ext_n) for i in sorted(self.ext_dev) if i in self.polys_dev and self.my_ntt(npoly + i) and not (i == 0 and to_coeff)]
        if coeffs:
            out["coefficients"] = np.stack(coeffs)
        if ext:
            out["extended"] = np.stack(ext)
        if to_coeff:
            out["extended_to_coeff"] = rows(self.ext_dev[0], ext_n)
        return out

    def close(self):
        if self.side_pool:
            self.side_pool.shutdown()
        if getattr(self, "pr_session", None) is not None:
            self.pr_session.free()
            self.pr_circuit.free()
        self.params.close()


def run_config(rig: Rig, sched: Schedule, steps: int, warmup: int, headline: bool, args):
    """times one schedule; returns (result dict, workload)"""
    torch = rig.torch
    wl = Workload(rig, sched, want_e2e=headline, fault=args.inject_fault)
    res = {"k": sched.k, "config": sched.describe(rig.world), "pairs_per_step": sched.pairs}
    prof = "k_accumulate" if headline else None
    ms_step, launches = rig.timed(wl.step_resident, steps, warmup, prof=prof)
    res["ms_per_step"], res["gpu_launches"] = ms_step, launches
    if headline:
        res["acc"] = rig.ctx.profile_read("k_accumulate")
        res["bred"] = rig.ctx.profile_read("k_batch_affine")
        if args.dump_outputs and rig.rank == 0:
            write_outputs(wl.outputs(), args.dump_outputs)
    torch.cuda.synchronize()
    res["verified_resident"] = wl.verify_commitments(wl.outs_dev.cpu().numpy().view(np.uint64))
    if headline:
        # the other placement of the transforms, for the record (the rule in step_resident picks by shard size)
        dflt_overlap = wl.n_loc >= (1 << 18) or BENCH_BG_NTT > 0
        ms_alt, _ = rig.timed(lambda: wl.step_resident(not dflt_overlap), steps, 1)
        res["ms_per_step_seq"] = ms_alt if dflt_overlap else ms_step
        res["ms_per_step_ovl"] = ms_step if dflt_overlap else ms_alt
        res["transform_placement"] = "beside the commitment phases (side stream)" if dflt_overlap else "one block before the h(X) phase"
    return res, wl


def run_b200(args):
    rig = Rig(args)
    torch, ctx, rank, world = rig.torch, rig.ctx, rig.rank, rig.world
    lib, C = None, None
    sched = Schedule(args.config, args.k)
    k, n, ext_k = sched.k, sched.n, sched.ext_k

    sampler = ClockSampler(rig.local_rank)
    if rank == 0:
        sampler.start()
    res, wl = run_config(rig, sched, args.steps, args.warmup, True, args)
    clocks = sampler.stop() if rank == 0 else None
    lib, C, vp = wl.lib, wl.C, wl.C.c_void_p
    ms_step, launches, ms_step_seq = res["ms_per_step"], res["gpu_launches"], res["ms_per_step_seq"]
    acc_ms, acc_cnt = res["acc"]

    # ---- end to end (the headline): the resident prover path — witness cells and the random polynomial go up from pinned
    # host memory, commitments and evaluations come down, every column stays in HBM behind h2b_poly handles in between,
    # and the step contains the quotient / product-column / opening work create_proof does between the commitments
    wl.setup_prover()
    ms_e2e, e2e_launches = rig.timed(wl.step_e2e_prover, args.steps, 2)
    torch.cuda.synchronize()
    prover_check = wl.verify_prover()
    # ---- the round-1 end-to-end path for continuity: every call takes and returns HOST buffers (h2b_* without _dev)
    if os.environ.get("H2B_E2E_TRACE"):
        wl.trace = []
    ms_e2e_ovl, _ = rig.timed(wl.step_e2e, args.steps, 1)
    ms_e2e_seq, _ = rig.timed(lambda: wl.step_e2e(False), args.steps, 1)
    torch.cuda.synchronize()
    verified_e2e = wl.verify_commitments(wl.outs_host)
    if wl.trace is not None and rank == 0:
        wl.trace.clear()
        wl.step_e2e(True)
        torch.cuda.synchronize()
        t0 = wl.trace[0][1]
        print("e2e trace (ms since start): " + ", ".join("%s=%.2f" % (l, 1e3 * (t - t0)) for l, t in wl.trace[1:]), file=sys.stderr)
    ms_e2e_host = min(ms_e2e_ovl, ms_e2e_seq)
    ntt_check = wl.verify_ntt()

    # per-op device timings (context for the headline; same CUDA-event method, 3 reps each)
    iu = next(j for j, (_, c, _) in enumerate(sched.msm) if c == "uniform")
    iw = next(j for j, (_, c, t) in enumerate(sched.msm) if c == "witness" and t != "advice")
    p0 = next(iter(wl.polys_dev))
    op_ms = {
        "msm_uniform": rig.time_op(lambda: wl.params.commit_dev(wl.basis_id[iu], wl.col_ptr[iu], wl.n_loc, wl.outs_dev[iu].data_ptr())),
        "msm_witness": rig.time_op(lambda: wl.params.commit_dev(wl.basis_id[iw], wl.col_ptr[iw], wl.n_loc, wl.outs_dev[iw].data_ptr())),
        "intt": rig.time_op(lambda: ctx.check(lib.h2b_lagrange_to_coeff_dev(ctx.h, vp(wl.polys_dev[p0].data_ptr()), k))),
        "coset_ntt": rig.time_op(lambda: ctx.check(lib.h2b_coeff_to_extended_dev(ctx.h, vp(wl.polys_dev[p0].data_ptr()), n, ext_k, vp(wl.ext_dev[p0].data_ptr())))),
        "coset_intt": rig.time_op(lambda: ctx.check(lib.h2b_extended_to_coeff_dev(ctx.h, vp(wl.ext_dev[p0].data_ptr()), ext_k))),
        "assign": rig.time_op(wl.assign_dev),
    }

    # the same columns once more, one MSM at a time (no lane overlap): the accumulation kernels timed alone
    ctx.profile_reset()
    ctx.profile_enable("k_")
    for j in range(len(sched.msm)):
        wl.params.commit_dev(wl.basis_id[j], wl.col_ptr[j], wl.n_loc, wl.outs_dev[j].data_ptr())
    torch.cuda.synchronize()
    iso_ms, iso_cnt = ctx.profile_read("k_accumulate")
    iso_aff_ms, iso_aff_cnt = ctx.profile_read("k_batch_affine")
    ctx.profile_enable(None)
    windows = wl.params.windows
    n_cells_total = wl.n_cells + wl.n_lookup
    window_bits = wl.params.window_bits
    wl.close()
    del wl
    torch.cuda.empty_cache()

    # ---- the other BASELINE configs (short runs; resident step + verification only)
    sweep = {}
    for cid in args.sweep_ids:
        if cid == args.config:
            continue
        s2 = Schedule(cid)
        st = 2 if s2.k >= 22 else 3
        try:
            r2, w2 = run_config(rig, s2, st, 2, False, args)
            ntt2 = w2.verify_ntt()
            iu2 = next(j for j, (_, c, _) in enumerate(s2.msm) if c == "uniform")
            p2 = next(iter(w2.polys_dev))
            t_msm = rig.time_op(lambda: w2.params.commit_dev(w2.basis_id[iu2], w2.col_ptr[iu2], w2.n_loc, w2.outs_dev[iu2].data_ptr()))
            t_ntt = rig.time_op(lambda: ctx.check(lib.h2b_coeff_to_extended_dev(ctx.h, vp(w2.polys_dev[p2].data_ptr()), s2.n, s2.ext_k, vp(w2.ext_dev[p2].data_ptr()))))
            t_asg = rig.time_op(w2.assign_dev)
            ok = r2["verified_resident"] == len(s2.msm) and all(v for kk, v in ntt2.items() if kk != "points_checked")
            # the resident proof of this shape (multi-column / lookup-advice / lookup-less circuits included), verified
            e2e2 = None
            if s2.k <= 20:
                w2.setup_prover()
                ms_p, _ = rig.timed(w2.step_e2e_prover, st, 1)
                torch.cuda.synchronize()
                chk = w2.verify_prover()
                e2e2 = {"ms_per_proof": ms_p, "pairs_per_s": s2.pairs / (ms_p / 1e3), "commitments_verified": chk["commitments"], "of": chk["of"],
                        "quotient_identity": chk["quotient_identity"], "h2d_bytes": chk["h2d_bytes"], "d2h_bytes": chk["d2h_bytes"]}
                ok = ok and chk["commitments"] == chk["of"] == len(s2.msm) and chk["quotient_identity"]
                w2.close_prover()
            sweep[f"config{cid}"] = {
                "workload": r2["config"]["workload"], "k": s2.k, "columns": r2["config"]["columns"], "msm": r2["config"]["msm"], "ntt": r2["config"]["ntt"],
                "create_proof_schedule_ms": r2["ms_per_step"], "msm_pairs_per_s": s2.pairs / (r2["ms_per_step"] / 1e3),
                "msm_only_ms": t_msm, "msm_only_pairs_per_s": s2.n / (t_msm / 1e3) * world,
                "coset_ntt_ms": t_ntt, "ntt_elements_per_s": (1 << s2.ext_k) / (t_ntt / 1e3),
                "assign_ms": t_asg, "assign_cells_per_s": (w2.n_cells + w2.n_lookup) / (t_asg / 1e3),
                "roofline": {"msm_hbm_frac": 96.0 * w2.n_loc / (t_msm / 1e3) / 1e9 / measured_hbm_peak()[0],
                             "ntt_hbm_frac": 64.0 * (1 << s2.ext_k) / (t_ntt / 1e3) / 1e9 / measured_hbm_peak()[0],
                             "assign_hbm_frac": 64.0 * (w2.n_cells + w2.n_lookup) / (t_asg / 1e3) / 1e9 / measured_hbm_peak()[0]},
                "steps": st, "gpu_launches": r2["gpu_launches"], "e2e_resident_proof": e2e2,
                "verified": {"msm": r2["verified_resident"], "of": len(s2.msm), "ntt": ntt2, "ok": rig.all_true(ok)},
            }
            w2.close()
            del w2
            torch.cuda.empty_cache()
        except Exception as e:  # a sweep extra must not take the headline down; it is reported as failed
            sweep[f"config{cid}"] = {"error": f"{type(e).__name__}: {e}"}
            import traceback
            print(f"sweep config {cid} failed:\n" + traceback.format_exc(), file=sys.stderr)
            if not rig.all_true(False):
                pass

    ok_all = (res["verified_resident"] == len(sched.msm) and verified_e2e == len(sched.msm)
              and prover_check["commitments"] == prover_check["of"] and prover_check["quotient_identity"]
              and all(v for kk, v in ntt_check.items() if kk != "points_checked")
              and all(v.get("verified", {}).get("ok", False) for v in sweep.values()))
    ok_all = rig.all_true(ok_all)
    verified = {"msm": res["verified_resident"], "msm_e2e": prover_check["commitments"], "msm_e2e_host_buffers": verified_e2e, "of": len(sched.msm),
                "e2e_quotient_identity": prover_check["quotient_identity"], "ntt": ntt_check,
                "sweep_ok": {kk: v.get("verified", {}).get("ok", False) for kk, v in sweep.items()},
                "method": "closed form sum_i s_i*(a0+d*i)*G with Python integers (bases are that progression), after the all-reduce at N>1; Horner evaluations for the transforms",
                "all_ranks_ok": ok_all}
    if rank != 0:
        if rig.dist:
            rig.dist.destroy_process_group()
        sys.exit(0 if ok_all else 3)

    n_loc = n // world
    value = sched.pairs / (ms_step / 1e3)
    peak, peak_src = measured_hbm_peak()
    # the dominant kernel: bucket accumulation = the batch-affine reduction passes + the XYZZ accumulation of what is left
    # a launch of the grouped pipeline accumulates the columns of a whole group (1-2 at k = 19): per launch the
    # algorithmic bytes are 96 B x pairs of ALL its columns, so the average is formed over the step's totals
    msm_per_launch = len(sched.msm) * args.steps / max(acc_cnt, 1)
    acc_avg_ms = (acc_ms + res["bred"][0]) / max(acc_cnt, 1)
    iso_avg_ms = (iso_ms + iso_aff_ms) / max(iso_cnt, 1)
    achieved = 96.0 * n_loc * msm_per_launch / (acc_avg_ms / 1e3) / 1e9  # algorithmic 96 B per pair (32 B scalar + 64 B base), SURVEY.md §8d
    achieved_iso = 96.0 * n_loc / (iso_avg_ms / 1e3) / 1e9
    traffic = None
    tpath = os.path.join(ROOT, "profiles", "traffic.json")  # dram bytes per launch from the committed ncu --set full capture
    if os.path.exists(tpath):
        try:
            traffic = json.load(open(tpath)).get(f"k{k}_n{world}")  # per MSM column
            traffic = traffic * msm_per_launch if traffic else None
        except Exception:
            traffic = None
    roofline = {"bound": "hbm", "kernel": "bucket accumulation (k_batch_affine passes + k_accumulate)", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                "traffic": traffic, "peak_source": peak_src,
                "avg_launch_ms": acc_avg_ms, "launches_timed": acc_cnt, "msm_columns_per_launch": msm_per_launch,
                "algorithmic_bytes_per_launch": 96 * n_loc * msm_per_launch,
                "timed_region_note": "launches of the timed region overlap with the kernels of the other two MSM lanes, which stretches each launch",
                "isolated": {"avg_launch_ms": iso_avg_ms, "launches": iso_cnt, "achieved": achieved_iso, "frac": achieved_iso / peak,
                             "k_accumulate_ms": iso_ms / max(iso_cnt, 1), "k_batch_affine_ms": iso_aff_ms / max(iso_cnt, 1)},
                "note": "bucket accumulation is bound by the integer multiplier (IMAD.WIDE), not by HBM; see DESIGN.md 4.1/4.2 and profiles/"}
    npoly = sched.n_poly
    adv_bytes = (sched.A + sched.L) * n * 32
    # per step and rank 0: virtual column + looked-up cells, every MSM's scalar shard, the polynomials of the transforms
    # this rank owns (coefficients go up once for both transforms), the extended polynomial of extended_to_coeff
    h2d = (n_cells_total * 32 + len(sched.msm) * n_loc * 32 + (npoly * n * 32 + (1 << ext_k) * 32) // world)
    d2h = (adv_bytes + len(sched.msm) * 96 + (npoly * n * 32 + npoly * (1 << ext_k) * 32 + (1 << ext_k) * 32) // world)
    cpu = cpu_sample(sched) if world == 1 and not args.no_cpu else None
    line = {
        "metric": metric_name(sched), "value": value, "unit": "G1 pairs/s",
        "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "u32x8 (254-bit Montgomery integers)", "data": "synthetic",
        "config": res["config"],
        "create_proof_schedule_ms": ms_step,
        "create_proof_schedule_ms_no_ntt_overlap": ms_step_seq,
        "create_proof_schedule_ms_ntt_overlap": res["ms_per_step_ovl"],
        "transform_placement": res["transform_placement"],
        "ntt_fr_elements_per_s": (1 << ext_k) / (op_ms["coset_ntt"] / 1e3),
        "msm_only_pairs_per_s": n / (op_ms["msm_uniform"] / 1e3),
        "msm_window_bits": window_bits, "msm_windows": windows,
        "op_ms": op_ms,
        "e2e": {"value": sched.pairs / (ms_e2e / 1e3), "unit": "G1 pairs/s", "ms_per_step": ms_e2e,
                "h2d_bytes_per_step": prover_check["h2d_bytes"], "d2h_bytes_per_step": prover_check["d2h_bytes"], "gpu_launches": e2e_launches,
                "path": "halo2_lib_b200.ProverSession.prove (h2b_poly handles): pinned witness cells + random polynomial up, 12 commitments + 26 evaluations down; assignment, q_lookup*a, permute_expression_pair, permutation / lookup product columns, 5 x (lagrange_to_coeff + coeff_to_extended), gate + permutation + lookup terms folded on the extended coset, divide_by_vanishing_poly, extended_to_coeff, h pieces, evaluations, SHPLONK-shaped linear combinations and kate divisions all on the device; host: Blake2b transcript + blinding scalars; one synchronisation per commitment phase"},
        "e2e_host_buffers": {"value": sched.pairs / (ms_e2e_host / 1e3), "unit": "G1 pairs/s", "ms_per_step": ms_e2e_host,
                "ms_per_step_overlapped": ms_e2e_ovl, "ms_per_step_sequential_calls": ms_e2e_seq,
                "reported": "overlapped" if ms_e2e_ovl <= ms_e2e_seq else "sequential_calls",
                "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                "path": "round-1 path kept for continuity: h2b_assign_columns / h2b_msm_g1_batch_reduced / h2b_lagrange_to_coeff_and_extended_batch / h2b_extended_to_coeff, every call with pinned HOST buffers in and out (no quotient work); transforms driven by a second host thread + context; the faster of the overlapped and the strictly sequential call order is reported"},
        "gpu_launches": launches,
        "verified": verified,
        "clocks": clocks,
        "roofline": roofline,
        "cpu_baseline": cpu,
        "extra": {"configs": sweep},
    }
    if not ok_all:
        print("VERIFICATION FAILED: " + json.dumps(verified), file=sys.stderr)
        if rig.dist:
            rig.dist.destroy_process_group()
        sys.exit(3)
    print(json.dumps(line))
    if rig.dist:
        rig.dist.destroy_process_group()


def run_single_process(args):
    """ONE process drives --gpus N devices through a device-group context (h2b_ctx_create_multi): the host-buffer schedule
    (assignment, per-phase h2b_msm_g1_batch over the internally sharded SRS, batched transforms dealt over the devices).
    Every call is synchronous, so the CUDA events on the lead device's stream bracket all devices' work."""
    import ctypes as C
    import torch
    import halo2_lib_b200 as h
    from halo2_lib_b200._capi import lib
    N = args.gpus
    sched = Schedule(args.config, args.k)
    assert sched.A == 1 and sched.L == 0, "--single-process covers the single-advice-column shapes (configs 1, 3, 5)"
    k, n, ext_k = sched.k, sched.n, sched.ext_k
    torch.cuda.set_device(0)
    grp = h.Context(list(range(N)))
    stream = torch.cuda.Stream(device=0)
    torch.cuda.set_stream(stream)
    grp.set_stream(stream.cuda_stream)
    vp = C.c_void_p
    rng = np.random.default_rng(0xB2000000 + 97 * sched.cfg_id + k)
    gbase = np.array([0xd35d438dc58f0d9d, 0x0a78eb28f5c70b3d, 0x666ea36f7879462c, 0x0e0a77c19a07df2f,
                      0xa6ba871b8b1e1b3a, 0x14f1d651eb8e167b, 0xccdd46def0f28c58, 0x1c14ef83340fbe5e], dtype=np.uint64)
    host_bases = {}
    for name, (a0, d) in BASES.items():
        sc = np.zeros((n, 4), dtype=np.uint64)
        sc[:, 0] = (a0 + d * np.arange(n, dtype=np.uint64)).astype(np.uint64)
        host_bases[name] = grp.g1_fixed_base_mul(gbase, grp.field_op(1, 5, sc))
    params = h.ParamsKZG(grp, k, g=host_bases["monomial"], g_lagrange=host_bases["lagrange"])
    del host_bases
    pin = lambda arr: torch.from_numpy(np.ascontiguousarray(arr).view(np.int64)).pin_memory()
    usable = n - UNUSABLE_ROWS
    n_cells = usable - 5
    v_host = grp.field_op(1, 5, witness_like(rng, n_cells))
    vcol = pin(v_host)
    acol = torch.empty((n, 4), dtype=torch.int64).pin_memory()
    cols, expect = [], []
    basis_id = [0 if b == "monomial" else 1 for b, _, _ in sched.msm]
    for j, (basis, cls, tag) in enumerate(sched.msm):
        a0, d = BASES[basis]
        if tag == "advice":
            full = np.zeros((n, 4), dtype=np.uint64)
            full[:n_cells] = v_host
            cols.append(acol)
        else:
            full = uniform_residues(rng, n) if cls == "uniform" else grp.field_op(1, 5, witness_like(rng, n))
            cols.append(pin(full))
        expect.append(ec_mul_g(progression_dot(full, a0, d, 0) * MONT_RINV_R % R_MOD))
    polys = [pin(uniform_residues(rng, n)) for _ in range(sched.n_poly)]
    exts = [torch.empty((1 << ext_k, 4), dtype=torch.int64).pin_memory() for _ in range(sched.n_poly)]
    outs = np.zeros((len(sched.msm), 12), dtype=np.uint64)

    def step():
        grp.check(lib.h2b_assign_columns(grp.h, vp(vcol.data_ptr()), n_cells, None, 0, k, 1, vp(acol.data_ptr())))
        for pi, phase in enumerate(sched.phases):
            if pi == sched.h_phase:
                pa = (C.c_void_p * sched.n_poly)(*[p.data_ptr() for p in polys])
                pe = (C.c_void_p * sched.n_poly)(*[e.data_ptr() for e in exts])
                grp.check(lib.h2b_lagrange_to_coeff_and_extended_batch(grp.h, pa, sched.n_poly, k, ext_k, pe))
                grp.check(lib.h2b_extended_to_coeff(grp.h, vp(exts[0].data_ptr()), ext_k))
            m = len(phase)
            ptrs = (C.c_void_p * m)(*[cols[j].data_ptr() for j in phase])
            bs = (C.c_int * m)(*[basis_id[j] for j in phase])
            out = np.empty((m, 12), dtype=np.uint64)
            grp.check(lib.h2b_msm_g1_batch(grp.h, params.h, bs, ptrs, m, n, vp(out.ctypes.data)))
            outs[phase] = out

    for _ in range(args.warmup):
        step()
    torch.cuda.synchronize()
    l0 = grp.kernel_launches
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    sampler = ClockSampler(0)
    sampler.start()
    e0.record(stream)
    for _ in range(args.steps):
        step()
    e1.record(stream)
    torch.cuda.synchronize()
    clocks = sampler.stop()
    ms = e0.elapsed_time(e1) / args.steps
    launches = grp.kernel_launches - l0
    ok = sum(1 for j in range(len(sched.msm)) if point_matches(outs[j], expect[j]))
    h2d = n_cells * 32 + len(sched.msm) * n * 32 + sched.n_poly * n * 32 + (1 << ext_k) * 32
    d2h = n * 32 + len(sched.msm) * 96 + sched.n_poly * (n + (1 << ext_k)) * 32 + (1 << ext_k) * 32
    cfg = sched.describe(N)
    cfg["parallelism"] = f"ONE process, {N} devices through a device-group context (h2b_ctx_create_multi): SRS sharded inside h2b_srs_upload, partial sums combined by the fused all-reduce kernel over in-process peer mappings, transforms dealt round-robin"
    cfg["overlap"] = "strictly sequential host calls (no side thread); uploads pipelined against the kernels inside each call"
    value = sched.pairs / (ms / 1e3)
    line = {"metric": metric_name(sched), "value": value, "unit": "G1 pairs/s", "n_gpus": N, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "u32x8 (254-bit Montgomery integers)",
            "data": "synthetic", "config": cfg, "single_process": True,
            "e2e": {"value": value, "unit": "G1 pairs/s", "ms_per_step": ms, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "path": "h2b_assign_columns / h2b_msm_g1_batch / h2b_lagrange_to_coeff_and_extended_batch / h2b_extended_to_coeff on a device-group context, pinned HOST buffers in and out"},
            "gpu_launches": launches, "verified": {"msm_e2e": ok, "of": len(sched.msm)}, "clocks": clocks,
            "roofline": None, "cpu_baseline": None}
    params.close()
    grp.close()
    if ok != len(sched.msm):
        print("VERIFICATION FAILED: " + json.dumps(line["verified"]), file=sys.stderr)
        sys.exit(3)
    print(json.dumps(line))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10, help="timed steps of each step timing of the headline config")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", type=int, default=3, choices=[1, 2, 3, 4, 5], help="BASELINE.json config (1-based); 3 = ECDSA k=19 is the headline")
    ap.add_argument("--k", type=int, default=None, help="override the config's k")
    ap.add_argument("--sweep", default="1,2,4,5", help="other BASELINE configs run as extras (comma list, or 'none')")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg (profiling runs)")
    ap.add_argument("--inject-fault", default=None, choices=["skip_allreduce"], help="testing: break the multi-GPU exchange; the run must exit 3")
    ap.add_argument("--single-process", action="store_true", help="one process drives --gpus N devices through a device-group context (no torchrun)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed resident step computed to DIR/<name>.npy (float64, at most 64 MB; seeded inputs, the same on every run)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    if args.dump_outputs and (args.impl != "b200" or args.single_process):
        ap.error("--dump-outputs writes the outputs of the default GPU path (--impl b200 without --single-process)")
    args.sweep_ids = [] if args.sweep in ("none", "") else [int(x) for x in args.sweep.split(",")]
    if args.impl == "reference":
        run_reference(args)
    elif args.single_process:
        run_single_process(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
