#!/usr/bin/env python3
"""bench.py -- one JSON line per run (contract in the task statement).

A "step" is one pass of the hot path over one batch of synthetic input.  The headline workload (--workload, default
dense4m) fills the contract's top-level keys; the other BASELINE.json workloads are measured in the same run and reported
under "workloads" so ONE driver invocation carries all of them:
  dense4m     BASELINE.json configs[1]: full zkml proof (Prover::prove: witness commits, LogUp-GKR lookups, per-layer
              sumchecks, table proofs, Basefold batch opening; host Poseidon2 Fiat-Shamir) of the Dense-4M MLP of SURVEY.md
              8(d) Cfg 2 -- 4 x [Dense 1024x1024 + bias -> Requant -> ReLU], BIT_LEN 8.  Context::generate (weight commits)
              is setup and is not timed, exactly as zkml/src/bin/bench.rs:390-408 times it.  A step = 16 independent proofs.
  cnn264k     configs[2]: the same for the CNN-264k model (deep-prove_b200/models.py).
  sumcheck20  configs[0] shape: IOPProverState::prove_parallel, nu=20, degree 3, three Base MLEs -> proofs/s, field-ops/s
              and achieved GB/s against the measured HBM peak.
  basefold24  configs[3] on one GPU: Basefold commit+open of 2^24 Base evaluations -> openings/s and Poseidon2
              permutations/s against the INT32-issue ceiling.
`value`  : units/s with everything the step reads already resident in HBM; `e2e`: through the host-facing call with HOST
           buffers (inference + witness upload + prove + proof back for the models; upload + prove otherwise).
`roofline`: per-kernel table taken from a profiled pass of the SAME concurrent batch (per-launch CUDA events on every proving
           thread's stream), each kernel against the bound that actually limits it (HBM bytes or INT32 issue slots).
`cpu_baseline` / `--impl reference`: the CPU path (the C++ oracle port -- the reference itself is Rust with un-vendored
           dependencies and cannot be built here, DESIGN.md section 3) in latency mode (1 proof x all host threads) AND in
           throughput mode (k concurrent proofs x T/k threads); the better of the two is the value.
`parity_checked`: the GPU proof and the CPU-arm proof of the same input compared word for word outside the timed region.
"""
import os
os.environ.setdefault("CUDA_DEVICE_MAX_CONNECTIONS", "32")   # before torch/CUDA initialise: 16 proof streams + commit pools need more than 8 hardware queues
import argparse
import json
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(ROOT, "deep-prove_b200"))

P = np.uint64(0xFFFFFFFF00000001)
MASK = (1 << 64) - 1
DTYPE = "u64 (Goldilocks / GoldilocksExt2 modular integers)"


def splitmix_raw(seed, n, start=0):
    with np.errstate(over="ignore"):
        i = np.arange(start + 1, start + n + 1, dtype=np.uint64)
        z = np.uint64(seed & MASK) + i * np.uint64(0x9E3779B97F4A7C15)
        z = (z ^ (z >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
        z = (z ^ (z >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
        return z ^ (z >> np.uint64(31))


def splitmix_f(seed, n):
    """n splitmix64 draws mod p (vectorised; identical stream to oracle/field.hpp SplitMix64)."""
    return splitmix_raw(seed, n) % P


class ClockSampler:
    QUERY = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.idx = gpu_index
        self.samples = []
        self.proc = None

    def __enter__(self):
        # ONE long-running nvidia-smi (-lms 200) for the whole timed region, as in the profiling recipe; rank 0 only (its
        # line is the one printed, and N pollers taking driver locks perturb a launch-heavy workload)
        if int(os.environ.get("RANK", "0")) != 0:
            return self
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.idx), "--query-gpu=" + self.QUERY,
                                          "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.proc = None
        return self

    def __exit__(self, *a):
        if self.proc is None:
            return
        time.sleep(0.25)
        self.proc.terminate()
        try:
            out, _ = self.proc.communicate(timeout=5)
        except Exception:
            self.proc.kill()
            out = ""
        for line in out.strip().splitlines():
            self.samples.append([x.strip() for x in line.split(",")])

    def summary(self):
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for s in self.samples:
            try:
                sm.append(float(s[1])); mx.append(float(s[2]))
                for nm, v in zip(names, s[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(nm)
            except Exception:
                pass
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": max(mx), "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------------------------------------
# Workloads.  Common interface:
#   setup_device(dp); step_resident(i) / step_e2e(i) [single-stream workloads] or run_resident(k, dev) / run_e2e(k, dev)
#   [batches of concurrent proofs]; gpu_proof() / cpu_proof(O): the proof of the SAME input on both arms (parity check);
#   cpu_step(O, i): one CPU unit; returns seconds when the unit is a scaled sample (cpu_returns_seconds).
class SumcheckWorkload:
    key = "sumcheck20"
    metric, unit = "proofs/sec", "proofs/s"
    name = "sumcheck prove_parallel nu=20 deg=3 3xBase (BASELINE configs[0] shape), host Poseidon2 FS"
    NV = 20
    NSETS = 8   # 8 x 24 MiB = 192 MiB of inputs > 126 MB L2: a set is evicted before it is reused
    units_per_step = 1
    cpu_frac = 1.0

    def __init__(self):
        self.products = [((1, 0), [0, 1, 2])]
        n = 1 << self.NV
        self.host_sets = [[splitmix_f(3 * k + j + 1, n) for j in range(3)] for k in range(self.NSETS)]
        self.h2d = 3 * n * 8
        self.d2h = self.NV * 4 * 16 + 3 * 16 + self.NV * 16
        # algorithmic bytes of one proof (SURVEY.md 8d: 48 n per Base MLE)
        self.alg_bytes = 3 * 48 * n
        # field operations of one proof, in the operand field, SURVEY.md 8(d) "Field-op counts, K1 per pair": (d-1)(d+1) mul +
        # (5d+4) add per pair; the fused fold of round r >= 2 costs (1 mul + 2 add) for each of the 2 new elements of each
        # of the d operands of a pair
        d = 3
        self.field_ops = sum((1 << (self.NV - 1 - r)) * ((d - 1) * (d + 1) + 5 * d + 4 + (6 * d if r > 0 else 0)) for r in range(self.NV))

    def setup_device(self, dp):
        self.dp = dp
        self.dev_sets = [[dp.Mle.upload(a, False) for a in s] for s in self.host_sets]
        dp.lib().dp_synchronize()

    def step_resident(self, i):
        self.last = self.dp.sumcheck_prove_parallel(self.dev_sets[i % self.NSETS], self.products, self.NV)
        return self.last

    def outputs(self):
        point, msgs, fin = self.last
        return {"point": point, "msgs": msgs, "final_evals": fin}

    def step_e2e(self, i):
        ms = [self.dp.Mle.upload(a, False) for a in self.host_sets[i % self.NSETS]]
        out = self.dp.sumcheck_prove_parallel(ms, self.products, self.NV)
        for m in ms:
            m.free()
        return out

    def cpu_step(self, O, i):
        mles = [(a, False) for a in self.host_sets[i % self.NSETS]]
        return O.sumcheck_prove(mles, self.products, self.NV)

    def gpu_proof(self):
        return np.concatenate([np.asarray(a).reshape(-1) for a in self.step_resident(0)])

    def cpu_proof(self, O):
        return np.concatenate([np.asarray(a).reshape(-1) for a in self.cpu_step(O, 0)])

    cpu_sample = "1 full proof (same workload) per step"
    cpu_returns_seconds = False
    l2_note = "rotating input sets (8 x 24 MiB > L2)"
    flush = False


class BasefoldWorkload:
    """BASELINE.json configs[3] on one GPU: Basefold commit + open of one Base polynomial with 2^24 evaluations
    (splitmix64 mod p), Poseidon2 Merkle, point of 24 E challenges from a fixed seed (SURVEY.md 8d Cfg 4)."""
    key = "basefold24"
    metric, unit = "commit+open/sec", "openings/s"
    NV = 24
    CPU_NV = 20      # bounded CPU sample: the first 2^20 evaluations (1/16 of the workload)
    units_per_step = 1
    cpu_frac = 1.0 / 16

    def __init__(self):
        self.name = "Basefold commit+open, 2^%d Base evaluations, RS rate 1/2, Poseidon2 Merkle, 200 queries" % self.NV
        n = 1 << self.NV
        self.evals = splitmix_f(1, n)
        self.point = splitmix_f(4, 2 * self.NV).reshape(self.NV, 2)
        self.h2d = 8 * n
        self.d2h = None
        # SURVEY.md 8(d): commit ~64 n, open ~240 n bytes; Poseidon2 permutations: commit 2(2n - 1) ~ 2^26 / 2 ... counted exactly below
        self.alg_bytes = (64 + 240) * n
        # compressions: commit tree over 2n leaves -> 2n/2 - 1... levels >= 1 of a 2n-leaf tree: n - 1; opening oracles: n + n/2 + ... ~ n
        self.permutations = 2 * ((n - 1) + (n - 1))

    def setup_device(self, dp):
        self.dp = dp
        self.mle = dp.Mle.upload(self.evals, False)
        _, flat = dp.pcs_open(self.mle, self.NV, self.point, cap=1 << 23)
        self.d2h = int(flat.size * 8)

    def step_resident(self, i):
        self.last = self.dp.pcs_open(self.mle, self.NV, self.point, cap=1 << 23)

    def outputs(self):
        root, flat = self.last
        return {"root": root, "proof": flat}

    def step_e2e(self, i):
        m = self.dp.Mle.upload(self.evals, False)
        out = self.dp.pcs_open(m, self.NV, self.point, cap=1 << 23)
        m.free()
        return out

    def cpu_step(self, O, i):
        nv = self.CPU_NV
        ev = self.evals[: 1 << nv]
        t0 = time.perf_counter()
        O.pcs_open(ev, False, nv, self.point[:nv], cap=1 << 23)
        return (time.perf_counter() - t0) * (1 << (self.NV - nv))

    def gpu_proof(self):   # parity on the CPU sample's input (the full 2^24 case is a -m gpu test: tests/test_gpu_baseline_size.py)
        nv = self.CPU_NV
        m = self.dp.Mle.upload(self.evals[: 1 << nv], False)
        root, flat = self.dp.pcs_open(m, nv, self.point[:nv], cap=1 << 23)
        m.free()
        return np.asarray(flat)

    def cpu_proof(self, O):
        nv = self.CPU_NV
        return np.asarray(O.pcs_open(self.evals[: 1 << nv], False, nv, self.point[:nv], cap=1 << 23))

    cpu_sample = "commit+open of the first 2^20 evaluations (1/16 of the workload), time scaled x16"
    cpu_returns_seconds = True
    l2_note = "256 MiB L2 flush between steps; the 128 MiB input + 256 MiB codeword + 512 MiB oracle exceed L2 anyway"
    flush = True


class DenseWorkload:
    """n_layers x [Dense(width x width) + bias -> Requant -> ReLU]; the tensors are the same splitmix64 streams the
    oracle's synthetic_mlp()/synthetic_input() draw, so both arms prove the identical model and input."""
    key = "dense4m"
    metric, unit = "proofs/sec", "proofs/s"
    NL, W = 4, 1024
    SEED_MODEL, SEED_INPUT = 1, 2
    cpu_frac = 1.0

    def __init__(self):
        nl, w = self.NL, self.W
        self.name = "Dense-4M: %d x [Dense %dx%d + bias -> Requant -> ReLU] (%.1fM weights), BIT_LEN 8, full zkml Prover::prove" % (nl, w, w, nl * w * w / 1e6)
        per = w * w + w
        draws = splitmix_raw(self.SEED_MODEL, nl * per).astype(np.int64)
        vals = (draws.view(np.uint64) % np.uint64(255)).astype(np.int64) - 127
        self.weights = np.concatenate([vals[l * per: l * per + w * w] for l in range(nl)])
        self.bias = np.concatenate([vals[l * per + w * w: (l + 1) * per] for l in range(nl)])
        lw = w.bit_length() - 1
        fp = ((lw + 24 + 7) // 8) * 8 - lw
        self.rq = np.array([[lw, fp, 3 << (fp - 2), 2 * 7 + lw + 1]] * nl, dtype=np.int64)
        self.x = (splitmix_raw(self.SEED_INPUT, w) % np.uint64(128)).astype(np.int64)
        # algorithmic bytes of the big streaming parts of one proof (DESIGN.md section 5): fix_high over the
        # 4 weight matrices (8 B/elt, one pass) + batch_open over 4 x 2^20 codewords/evals
        n = w * w
        self.alg_bytes = nl * 8 * n + (nl * (16 * n + 8 * n) + 240 * n // 4)
        self.h2d = None
        self.d2h = None

    def setup_device(self, dp):
        self.dp = dp
        self.ctx = dp.ZkmlContext(self.NL, self.W, self.weights, self.bias, self.rq)
        proof = self.ctx.prove(self.x)            # warm everything once; also sizes the proof
        self._gpu_proof = np.asarray(proof)
        self.d2h = int(proof.size * 8)
        nl, w = self.NL, self.W
        self.h2d = int(8 * w)     # the model input vector: inference and every witness column are produced on the device (csrc/witness.cu)
        self.ctx.run_inference(self.x)
        dp.lib().dp_synchronize()

    STREAMS = 48    # concurrent independent proofs per GPU (one host thread + CUDA stream + device arena each)
    units_per_step = STREAMS   # one bench step = one batch of STREAMS inference inputs, each proved independently

    def step_resident(self, i):
        self.ctx.prove_trace()

    def step_e2e(self, i):
        return self.ctx.prove(self.x)

    def run_resident(self, k, device):
        self.ctx.prove_concurrent(host_workers(self.STREAMS), k * self.units_per_step, device=device, e2e=False)

    def run_e2e(self, k, device):
        self.ctx.prove_concurrent(host_workers(self.STREAMS), k * self.units_per_step, device=device, e2e=True)

    def outputs(self):
        return {"proof": self.ctx.last_concurrent_proof()}

    def cpu_step(self, O, i):
        _, ms = O.zkml_prove(self.NL, self.W, self.SEED_MODEL, self.SEED_INPUT, want_proof=False)
        return ms[1] * 1e-3     # Prover::prove only; Context::generate (ms[0]) is setup

    def gpu_proof(self):
        return self._gpu_proof

    def cpu_proof(self, O):
        return np.asarray(O.zkml_prove(self.NL, self.W, self.SEED_MODEL, self.SEED_INPUT)[0])

    cpu_sample = "full proofs of the same model and input (Context::generate not counted)"
    cpu_returns_seconds = True
    l2_note = ("%d proofs in flight per GPU: aggregate working set (~130 MB of weights/codewords/oracles/trees per proof) "
               "is >> the 126 MB L2; single-stream latency is measured with a 256 MiB L2 flush between proofs" % STREAMS)
    flush = True


class CnnWorkload:
    """CNN-264k (SURVEY.md 8(d) Cfg 3) in its padded form: conv5x5 -> requant -> relu -> maxpool (x2) -> fc x3 on a
    3x32x32 input; the arrays come from deep-prove_b200/models.py and both arms prove the identical model and input."""
    key = "cnn264k"
    metric, unit = "proofs/sec", "proofs/s"
    STREAMS = 48
    units_per_step = STREAMS
    cpu_frac = 1.0

    def __init__(self):
        import models
        self.desc, self.data, self.x, self.n_params = models.cnn(seed=1)
        self.name = ("CNN-264k: conv5x5(12) -> requant -> relu -> maxpool -> conv5x5(33) -> requant -> relu -> maxpool -> fc 247 -> fc 173 -> fc 10 "
                     "on 3x32x32 (%d parameters, padded to powers of two), BIT_LEN 8, full zkml Prover::prove" % self.n_params)
        # big streaming parts of one proof: fix_high over the fc1 matrix (2^20 Base) + Basefold batch_open over the 2^20-sized commitments
        n = 1 << 20
        self.alg_bytes = 8 * n + (16 * n + 8 * n) + 240 * n
        self.h2d = None
        self.d2h = None

    def setup_device(self, dp):
        self.dp = dp
        self.ctx = dp.ModelContext(self.desc, self.data, self.x.size)
        proof = self.ctx.prove(self.x)
        self._gpu_proof = np.asarray(proof)
        self.d2h = int(proof.size * 8)
        # input + each convolution's input/output tensors (the FFT convolution op keeps a host-vector interface; everything else stays on the device)
        self.h2d = int(8 * self.x.size + 8 * (12 * 32 * 32 + 33 * 16 * 16 * 2))
        self.ctx.run_inference(self.x)
        dp.lib().dp_synchronize()

    def step_resident(self, i):
        self.ctx.prove_trace()

    def step_e2e(self, i):
        return self.ctx.prove(self.x)

    def run_resident(self, k, device):
        self.ctx.prove_concurrent(host_workers(self.STREAMS), k * self.units_per_step, device=device, e2e=False)

    def run_e2e(self, k, device):
        self.ctx.prove_concurrent(host_workers(self.STREAMS), k * self.units_per_step, device=device, e2e=True)

    def outputs(self):
        return {"proof": self.ctx.last_concurrent_proof()}

    def cpu_step(self, O, i):
        _, ms = O.model_prove(self.desc, self.data, self.x, want_proof=False)
        return ms[1] * 1e-3

    def gpu_proof(self):
        return self._gpu_proof

    def cpu_proof(self, O):
        return np.asarray(O.model_prove(self.desc, self.data, self.x)[0])

    cpu_sample = "full proofs of the same model and input (Context::generate not counted)"
    cpu_returns_seconds = True
    l2_note = ("%d proofs in flight per GPU (aggregate working set >> the 126 MB L2); single-stream latency is measured with a 256 MiB L2 flush between proofs" % STREAMS)
    flush = True


WORKLOADS = {"dense4m": DenseWorkload, "cnn264k": CnnWorkload, "sumcheck20": SumcheckWorkload, "basefold24": BasefoldWorkload}


_CPU_BUDGET = None


def cpu_budget():
    """(cached at first call, i.e. before this rank pins itself to its GPU's NUMA node) CPUs this rank may use: the process's affinity mask and the cgroup CPU quota (the 1-GPU measurement boxes report 128 logical
    CPUs but run the container under cpu.max = 16 CPUs: a spinning thread per proof in flight is throttled beyond that),
    divided among the ranks of this node"""
    try:
        cpus = float(len(os.sched_getaffinity(0)))
    except Exception:
        cpus = float(os.cpu_count() or 16)
    try:
        quota, period = open("/sys/fs/cgroup/cpu.max").read().split()
        if quota != "max":
            cpus = min(cpus, float(quota) / float(period))
    except Exception:
        pass
    global _CPU_BUDGET
    if _CPU_BUDGET is None:
        world = int(os.environ.get("LOCAL_WORLD_SIZE", os.environ.get("WORLD_SIZE", "1")))
        _CPU_BUDGET = max(2.0, cpus / max(world, 1))
    return _CPU_BUDGET


def host_workers(streams):
    """independent proofs in flight per GPU = proving threads.  They wait for the device through the library's blocking mode
    (dp_set_wait_mode(1): sleeping threads, one poller), so the count is set by what keeps the GPU busy (`streams`), capped at
    four threads per CPU of this rank's budget (a proof costs ~30 CPU-ms when its thread sleeps through the waits: 48 proofs in
    flight at ~290 proofs/s keep ~9 CPUs busy)."""
    return int(max(4, min(streams, 4 * cpu_budget())))


def pin_to_gpu_numa_node(torch, local_rank):
    """Every round trip of the prover crosses PCIe twice (mapped-memory message, challenge mailbox): keep this rank's
    host threads on the CPUs local to its GPU (sysfs local_cpulist of the GPU's PCI function).  Best effort."""
    try:
        pr = torch.cuda.get_device_properties(local_rank)
        path = "/sys/bus/pci/devices/%04x:%02x:%02x.0/local_cpulist" % (pr.pci_domain_id, pr.pci_bus_id, pr.pci_device_id)
        cpus = set()
        for part in open(path).read().strip().split(","):
            lo, _, hi = part.partition("-")
            cpus.update(range(int(lo), int(hi or lo) + 1))
        if cpus:
            os.sched_setaffinity(0, cpus)
            return len(cpus)
    except Exception:
        pass
    return None


def load_peaks():
    try:
        return json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json"))), "measured"
    except Exception:
        return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "sm_max_mhz": 1965.0}, "fallback"


def max_over_ranks(ms, dist, device="cuda"):
    """device-timed milliseconds -> the slowest rank's value (the job is only done when every rank is)"""
    if dist is None:
        return float(ms)
    import torch
    t = torch.tensor([ms], device=device, dtype=torch.float64)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


def whole_job_value(units_per_rank, world, ms):
    """replicas: every rank processes `units_per_rank` independent units; value = all units / slowest rank's time"""
    return units_per_rank * world / (ms * 1e-3)


DUMP_LIMIT = 64 << 20


def dump_outputs(outdir, outputs):
    """outputs: {workload: {name: uint64 array}} -> outdir/<workload>_<name>.npy.  Every 64-bit field word is stored exactly as
    two float64 values, its low and high 32 bits, along a new last axis of size 2."""
    arrays = {}
    for wk, outs in outputs.items():
        for name, a in outs.items():
            a = np.asarray(a, dtype=np.uint64)
            arrays["%s_%s" % (wk, name)] = np.stack([a & np.uint64(0xFFFFFFFF), a >> np.uint64(32)], axis=-1).astype(np.float64)
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_LIMIT:
        raise SystemExit("bench.py: outputs take %d bytes, more than the %d-byte limit of --dump-outputs" % (total, DUMP_LIMIT))
    os.makedirs(outdir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(outdir, name + ".npy"), a)


# ---- CPU arm -----------------------------------------------------------------------------------------
CPU_CONCURRENCY = 8     # throughput mode: this many proofs at once, each with (hardware threads / this many) worker threads


def cpu_arm(wl, O, steps, warm):
    """The CPU path in its two modes.  latency: one unit at a time on all host threads.  throughput: CPU_CONCURRENCY units at
    once, each on an equal share of the host threads (the like-for-like comparison with the GPU's concurrent batch).
    Returns a dict; `value` is the better mode's units/s."""
    lib = O.lib()
    hw_all = int(lib.dpo_num_threads())
    # the container may be allowed fewer CPUs than the machine has hardware threads (cgroup cpu.max: 16 CPUs on the 1-GPU measurement
    # boxes): more runnable threads than that only get throttled, so the CPU arm uses -- and reports -- what it can actually run on
    hw = max(1, min(hw_all, int(round(cpu_budget() * max(1, int(os.environ.get("LOCAL_WORLD_SIZE", os.environ.get("WORLD_SIZE", "1"))))))))
    lib.dpo_set_threads(hw)

    def unit_seconds(i):
        t0 = time.perf_counter()
        r = wl.cpu_step(O, i)
        dt = time.perf_counter() - t0
        return r if wl.cpu_returns_seconds else dt

    for i in range(warm):
        unit_seconds(i)
    tot = sum(unit_seconds(i) for i in range(steps))
    lat_v = steps / tot
    k = max(1, min(CPU_CONCURRENCY, hw // 4))
    thr_v, thr_wall = None, None
    if k > 1:
        lib.dpo_set_threads(max(1, hw // k))
        batches = max(1, min(steps, 3))

        def one_batch():
            th = [threading.Thread(target=wl.cpu_step, args=(O, j)) for j in range(k)]
            t0 = time.perf_counter()
            for t in th:
                t.start()
            for t in th:
                t.join()
            return time.perf_counter() - t0
        if warm:
            one_batch()
        wall = sum(one_batch() for _ in range(batches))
        lib.dpo_set_threads(hw)
        # a unit that is a scaled sample (basefold24: 1/16 of the polynomial) counts as cpu_frac of a unit
        thr_v = batches * k * wl.cpu_frac / wall
        thr_wall = wall / batches
    best = max(lat_v, thr_v or 0.0)
    return {"value": best, "unit": wl.unit, "cores": hw, "kind": "port",
            "mode": "throughput" if (thr_v or 0.0) > lat_v else "latency",
            "latency_mode": {"value": lat_v, "sec_per_unit": tot / steps, "threads": hw},
            "throughput_mode": ({"value": thr_v, "concurrent": k, "threads_each": max(1, hw // k), "sec_per_batch": thr_wall} if thr_v else None),
            "hardware_threads": hw_all,
            "sample": wl.cpu_sample + " (C++ restatement of the reference algorithm, not the Rust reference; `cores` = threads used = the CPUs this container may run on: min(hardware threads, cgroup cpu.max))"}


# ---- facts taken from the committed ncu captures (profiles/ncu_facts.json, written next to the capture summaries) ----
# The Poseidon2 kernels are bound by the FMA-heavy pipe that executes the 32 x 32 -> 64-bit multiplies (IMAD.WIDE) of the Goldilocks
# products: ncu (profiles/r02d_ncu_full_k_merkle_up.csv) shows sm__pipe_fmaheavy_cycles_active = 90.65 % at 1.69 Gperm/s, i.e. a
# ceiling of 1.865 Gperm/s per B200 at 1965 MHz for this formulation (12.85 k thread instructions per permutation).
P2_INSTR_PER_PERM = 12850.0
P2_CEILING_GPS, P2_CEILING_MHZ = 1.865, 1965.0
P2_CEILING_SOURCE = "profiles/r02d_ncu_full_k_merkle_up.csv"
NCU_TRAFFIC = {
    ("sumcheck20", "k_sc_round"): (7.69e6, "profiles/r01c_sumcheck20_rounds_ncu.csv: rounds 2-11 of one nu=20 proof, mean per launch (algorithmic 6.6 MB)"),
    ("dense4m", "k_sc_round"): (7.1e4, "profiles/r01_ncu_full_summary.csv: one small round (latency-bound)"),
}
try:
    _f = json.load(open(os.path.join(ROOT, "profiles", "ncu_facts.json")))
    P2_INSTR_PER_PERM = float(_f.get("p2_instr_per_perm", P2_INSTR_PER_PERM))
    P2_CEILING_GPS = float(_f.get("p2_perm_ceiling_gps_at_1965mhz", P2_CEILING_GPS))
    for k_, v_ in _f.get("traffic", {}).items():
        NCU_TRAFFIC[tuple(k_.split("/"))] = (v_[0], v_[1])
except Exception:
    pass

# BASELINE.md section 1: "Dense 4M proving time 2335 ms" (README.md:18; hardware and exact architecture NOT stated)
PUBLISHED = {"dense4m": 1.0 / 2.335, "cnn264k": 1.0 / 1.242}   # and "CNN 264k ... proving time 1242 ms" (README.md:17)


def kernel_table(prof, peaks, sm_mhz, sm_count=148):
    """per-kernel rows from dp_profile_read_ex: each kernel against the bound that limits it.
    Poseidon2 kernels: permutations/s against the FMA-heavy-pipe ceiling measured with ncu (scaled by the SM clock and count);
    sumcheck rounds: field-ops/s and GB/s against the measured HBM copy bandwidth; everything else: GB/s vs HBM.
    Kernels that process a handful of elements per launch are latency chains and are labelled so (no roofline applies)."""
    clock = (sm_mhz or peaks.get("sm_max_mhz") or 1965.0)
    perm_ceiling = P2_CEILING_GPS * 1e9 * (clock / P2_CEILING_MHZ) * (sm_count / 148.0)
    rows = {}
    for name, (cnt, ms, by, units) in prof.items():
        sec = ms * 1e-3
        row = {"launches": int(cnt), "ms": round(ms, 4), "avg_us": round(1e3 * ms / max(cnt, 1), 3),
               "GBps": round(by / sec / 1e9, 2) if sec > 0 else 0.0,
               "hbm_frac": round(by / sec / 1e9 / peaks["hbm_gbs"], 5) if sec > 0 else 0.0}
        if "poseidon2" in name:
            pps = units / sec if sec > 0 else 0.0
            row.update({"bound": "fma-heavy pipe (IMAD.WIDE of the 64-bit field products)" if cnt and units / cnt > 60000 else "latency (dependent hash chain)",
                        "perm_per_s": pps, "ceiling_perm_per_s": perm_ceiling, "pipe_frac": round(pps / perm_ceiling, 5)})
        elif name.startswith("k_sc_"):
            row.update({"bound": "hbm" if cnt and by / cnt > 4e6 else "latency (one round trip per Fiat-Shamir challenge)",
                        "field_ops_per_s": units / sec if sec > 0 else 0.0})
        else:
            row["bound"] = "hbm" if cnt and by / cnt > 4e6 else "latency"
        rows[name] = row
    return rows, perm_ceiling


def roofline_block(wl_key, rows, ceiling, peaks, peak_kind, source):
    """the dominant THROUGHPUT-bound kernel of a per-kernel table against its own bound (latency chains are listed, not rated)"""
    cand = {k: r for k, r in rows.items() if not k.startswith("k_sc_res") and not r["bound"].startswith("latency")}
    if not cand:
        cand = {k: r for k, r in rows.items() if not k.startswith("k_sc_res")} or rows
    name = max(cand, key=lambda k: cand[k]["ms"])
    r = rows[name]
    all_ms = sum(x["ms"] for k, x in rows.items() if not k.startswith("k_sc_res"))
    traffic = NCU_TRAFFIC.get((wl_key, name.split("(")[0]))
    if "perm_per_s" in r and not r["bound"].startswith("latency"):
        roof = {"kernel": name, "bound": r["bound"], "achieved": r["perm_per_s"] / 1e9, "peak": ceiling / 1e9, "unit": "Gperm/s", "frac": r["pipe_frac"],
                "peak_kind": "measured with ncu: the thread-per-hash level kernel reaches 1.69 Gperm/s at sm__pipe_fmaheavy_cycles_active = 90.65 %% (%s); scaled by SM clock" % P2_CEILING_SOURCE}
    else:
        roof = {"kernel": name, "bound": r["bound"], "achieved": r["GBps"], "peak": peaks["hbm_gbs"], "unit": "GB/s", "frac": r["hbm_frac"],
                "peak_kind": peak_kind + " (MEASURED_PEAKS.json hbm_gbs)"}
    roof.update({"hbm": {"achieved": r["GBps"], "peak": peaks["hbm_gbs"], "unit": "GB/s", "frac": r["hbm_frac"]},
                 "traffic": traffic[0] if traffic else None, "traffic_source": traffic[1] if traffic else None,
                 "launches": r["launches"], "avg_us": r["avg_us"], "share_of_kernel_time": round(r["ms"] / all_ms, 4) if all_ms > 0 else None,
                 "source": source})
    return roof


def run_gpu_workload(env, wl, K, W, full):
    """time one workload on this rank's GPU; returns the result dict (rank 0 fills the CPU / parity parts when world == 1)"""
    torch, dp, dist = env["torch"], env["dp"], env["dist"]
    rank, world, local_rank = env["rank"], env["world"], env["local_rank"]
    wl.setup_device(dp)
    flush_buf = env["flush_buf"] if wl.flush else None

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps, warm):
        """K steps, each bracketed by CUDA events on the launch stream; the L2 flush sits between steps outside the
        events; barrier + synchronize on both sides; max over ranks."""
        for i in range(warm):
            fn(i)
        barrier()
        l0 = dp.lib().dp_kernel_launches()
        evs = []
        for i in range(steps):
            if flush_buf is not None:
                flush_buf.zero_()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            fn(warm + i)
            e1.record()
            evs.append((e0, e1))
        barrier()
        ms = sum(a.elapsed_time(b) for a, b in evs)
        launches = dp.lib().dp_kernel_launches() - l0
        return max_over_ranks(ms, dist), launches

    def timed_many(run, steps, warm):
        """K steps issued as one batch (concurrent proof streams): bracketed by CUDA events recorded on the main stream
        with barrier + synchronize on both sides (the worker streams are drained before the call returns)"""
        if warm:
            run(warm, local_rank)
        barrier()
        l0 = dp.lib().dp_kernel_launches()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        run(steps, local_rank)
        e1.record()
        barrier()
        return max_over_ranks(e0.elapsed_time(e1), dist), dp.lib().dp_kernel_launches() - l0

    batched = hasattr(wl, "run_resident")
    latency_ms = None
    clk = ClockSampler(local_rank)
    if batched:
        dp.set_wait_mode(1)      # many proofs in flight: proving threads sleep on the library's poller instead of spinning (DESIGN.md section 5)
        with clk:
            ms, launches = timed_many(wl.run_resident, K, W)
        outputs = wl.outputs()   # the last timed step's result, before the legs below overwrite it
        ms_e2e, _ = timed_many(wl.run_e2e, K, 1)
        if full:
            dp.set_wait_mode(0)  # one proof at a time: the single proving thread spins (lowest latency)
            lat, _ = timed(wl.step_resident, min(K, 10), 2)     # one proof at a time, L2 flushed between proofs
            latency_ms = lat / min(K, 10)
            dp.set_wait_mode(1)
    else:
        with clk:
            ms, launches = timed(wl.step_resident, K, W)
        outputs = wl.outputs()
        ms_e2e, _ = timed(wl.step_e2e, K, 2)
    clocks = clk.summary()

    # per-kernel legs.  (1) the SAME concurrent batch once more with per-launch CUDA events on every proving thread's stream: what runs
    # in the timed region (its per-kernel times overlap and stretch each other, so they give shares, not rates).  (2) for the
    # batched workloads, one proof at a time: every kernel alone on the GPU -- the rates the roofline fraction is computed from.
    peaks, peak_kind = env["peaks"]
    dp.profile_reset(); dp.profile_enable(True)
    if batched:
        wl.run_resident(min(K, 2), local_rank)
    else:
        for i in range(min(K, 5)):
            if flush_buf is not None:
                flush_buf.zero_()
            wl.step_resident(i)
    torch.cuda.synchronize()
    prof = dp.profile_read(with_units=True)
    dp.profile_enable(False)
    dp.set_wait_mode(0)
    rows, ceiling = kernel_table(prof, peaks, clocks.get("sm_mhz"), env["sm_count"])
    rows_alone = None
    if batched:
        dp.profile_reset(); dp.profile_enable(True)
        for i in range(3):
            if flush_buf is not None:
                flush_buf.zero_()
            wl.step_resident(i)
        torch.cuda.synchronize()
        rows_alone, _ = kernel_table(dp.profile_read(with_units=True), peaks, clocks.get("sm_mhz"), env["sm_count"])
        dp.profile_enable(False)

    ups = getattr(wl, "units_per_step", 1)
    v = whole_job_value(K * ups, world, ms)
    res = {"metric": wl.metric, "value": v, "unit": wl.unit, "steps": K, "warmup": W, "ms_per_step": ms / K,
           "e2e": {"value": whole_job_value(K * ups, world, ms_e2e), "unit": wl.unit, "h2d_bytes_per_step": wl.h2d * ups, "d2h_bytes_per_step": wl.d2h * ups},
           "gpu_launches": int(launches), "units_per_step": ups, "single_stream_latency_ms": latency_ms,
           "alg_GBps_whole_step": wl.alg_bytes * v / world / 1e9, "workload": wl.name, "l2": wl.l2_note, "clocks": clocks,
           "outputs": outputs}
    if hasattr(wl, "field_ops"):
        res["field_ops_per_s"] = wl.field_ops * v / world
        res["hbm_frac_whole_proof"] = wl.alg_bytes * v / world / 1e9 / peaks["hbm_gbs"]
    if hasattr(wl, "permutations"):
        res["poseidon2_perm_per_s"] = wl.permutations * v / world
        res["pipe_frac_whole_step"] = wl.permutations * v / world / ceiling

    roof = None
    if rows:
        if batched and rows_alone:
            roof = roofline_block(wl.key, rows_alone, ceiling, peaks, peak_kind, "profiled pass of single proofs (each kernel alone on the GPU, per-launch CUDA events on the launch stream)")
            # the whole timed region against the same ceiling: Poseidon2 permutations of all Merkle kernels per second of the batch
            perms = sum(u for n_, (c_, m_, b_, u) in prof.items() if "poseidon2" in n_)
            proofs_profiled = min(K, 2) * ups
            if proofs_profiled:
                pps = perms / proofs_profiled * v / world
                roof["whole_step"] = {"poseidon2_perm_per_proof": perms / proofs_profiled, "poseidon2_perm_per_s": pps, "frac_of_pipe_ceiling": round(pps / ceiling, 4),
                                      "note": "all Merkle kernels of the concurrent timed region: permutations per proof x proofs/s, against the same fma-heavy-pipe ceiling"}
            roof["kernels_concurrent_batch"] = dict(sorted(rows.items(), key=lambda kv: -kv[1]["ms"]))
            roof["kernels"] = dict(sorted(rows_alone.items(), key=lambda kv: -kv[1]["ms"]))
        else:
            roof = roofline_block(wl.key, rows, ceiling, peaks, peak_kind, "profiled pass of the same steps (per-launch CUDA events on the launch stream)")
            roof["kernels"] = dict(sorted(rows.items(), key=lambda kv: -kv[1]["ms"]))
    res["roofline"] = roof

    res["cpu_baseline"], res["parity_checked"] = None, None
    if rank == 0 and world == 1 and not env["no_cpu"]:
        sys.path.insert(0, os.path.join(ROOT, "tests"))
        import oracle_py as O   # cpu_baseline leg: the oracle is the checker/baseline, never the measured product
        try:
            g, c = wl.gpu_proof(), wl.cpu_proof(O)
            res["parity_checked"] = bool(g.shape == c.shape and (g == c).all())
        except Exception as e:   # a failed check must be visible, never silently true
            res["parity_checked"] = False
            res["parity_error"] = repr(e)[:200]
        res["cpu_baseline"] = cpu_arm(wl, O, 5 if wl.key == "sumcheck20" else 1, 0)
    return res


def sharded_sumcheck(env, nv=26, reps=3):
    """BASELINE configs[4] (B), N > 1 only: ONE sumcheck proof (nu = 26, degree 3, three Base MLEs, splitmix64 seeds 1, 2, 3) sharded over
    the ranks -- rank g owns elements [g n/N, (g+1) n/N) of every MLE on its own GPU; per round one local launch + one
    exchange of the (deg+1)-element partial message through a same-node shared-memory mailbox (the message has to reach the
    hosts for Fiat-Shamir anyway); the last log N rounds run replicated (IOPProverState::prove_sharded = prove_batch_polys with
    a rank per thread, sumcheck/src/prover.rs:37-321).  Timed with CUDA events, max over ranks; rank 0 then proves the unsplit
    polynomial alone and the two proofs are compared word for word."""
    import multigpu as mg
    torch, dp, dist, rank, world = env["torch"], env["dp"], env["dist"], env["rank"], env["world"]
    n = 1 << nv
    lo, hi = mg.shard_range(n, rank, world)
    products = [((1, 0), [0, 1, 2])]
    slices = [splitmix_raw(s, hi - lo, start=lo) % P for s in (1, 2, 3)]
    mb = mg.ShmMailbox("dpb200_bench_%d" % os.getppid(), rank, world, dist.barrier)

    def one():
        mles = [dp.Mle.upload(a, False) for a in slices]
        torch.cuda.synchronize(); dist.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        out = mg.prove_sharded_native(mles, products, nv, rank, world, mailbox=mb)
        e1.record(); torch.cuda.synchronize()
        return out, max_over_ranks(e0.elapsed_time(e1), dist)
    one()
    runs = [one() for _ in range(reps)]
    ms = min(r[1] for r in runs)
    point, msgs, fin = runs[-1][0]
    single_ms, same = None, None
    if rank == 0:
        full = [splitmix_raw(s, n) % P for s in (1, 2, 3)]
        ts = []
        for _ in range(3):                       # the first run grows the device arena: take the best
            mles = [dp.Mle.upload(a, False) for a in full]
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(); ref = dp.sumcheck_prove_parallel(mles, products, nv); e1.record(); torch.cuda.synchronize()
            ts.append(e0.elapsed_time(e1))
            del mles
        single_ms = min(ts)
        same = bool((ref[0] == point).all() and (ref[1] == msgs).all() and (ref[2] == fin).all())
    dist.barrier()
    mb.close(dist.barrier)
    return {"workload": "sumcheck nu=%d deg=3 3xBase: ONE proof sharded over %d GPUs (devirgo split across ranks)" % (nv, world),
            "sharded_ms": ms, "single_gpu_ms": single_ms, "speedup": (single_ms / ms) if single_ms else None,
            "bit_identical_to_single_gpu_proof": same, "exchange": "same-node shared-memory mailbox, %d B per rank per round" % (16 * 4),
            "alg_GBps_aggregate": 3 * 48 * n / (ms * 1e-3) / 1e9}


def sharded_basefold(env, nv=24, reps=3):
    """BASELINE configs[3], N > 1 only: Basefold commit + open of ONE 2^24-evaluation polynomial sharded over the ranks (every rank
    holds the polynomial; rank g keeps the slice [g/N, (g+1)/N) of the bit-reversed evaluations, codeword, folded oracles and
    Merkle subtrees; per round one all-gather of a partial message + a 32-byte subtree root through the same-node mailbox;
    csrc/basefold.cu dp_pcs_commit_shard, host/mpcs.hpp commit_sharded / open_sharded).  Timed with CUDA events, max over ranks;
    rank 0 then runs the unsharded commit + open alone and the two proofs are compared word for word."""
    import multigpu as mg
    torch, dp, dist, rank, world = env["torch"], env["dp"], env["dist"], env["rank"], env["world"]
    ev = splitmix_raw(7, 1 << nv) % P
    rng = splitmix_raw(8, 2 * nv) % P
    pt = rng.reshape(nv, 2)
    mb = mg.ShmMailbox("dpb200_bf_%d" % os.getppid(), rank, world, dist.barrier)
    poly = dp.Mle.upload(ev, False)

    def one():
        torch.cuda.synchronize(); dist.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        out = mg.basefold_commit_open_sharded(poly, nv, pt, rank, world, mailbox=mb)
        e1.record(); torch.cuda.synchronize()
        return out, max_over_ranks(e0.elapsed_time(e1), dist)
    one()
    runs = [one() for _ in range(reps)]
    ms = min(r[1] for r in runs)
    root, flat, times = runs[-1][0]
    single_ms, same = None, None
    if rank == 0:
        ts = []
        for _ in range(3):
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(); ref_root, ref_flat = dp.pcs_open(poly, nv, pt); e1.record(); torch.cuda.synchronize()
            ts.append(e0.elapsed_time(e1))
        single_ms = min(ts)
        same = bool((ref_root == root).all() and ref_flat.shape == flat.shape and (ref_flat == flat).all())
    dist.barrier()
    mb.close(dist.barrier)
    return {"workload": "Basefold commit+open, 2^%d Base evaluations: ONE polynomial sharded over %d GPUs" % (nv, world),
            "sharded_ms": ms, "commit_ms": times[0], "open_ms": times[1], "single_gpu_ms": single_ms, "speedup": (single_ms / ms) if single_ms else None,
            "bit_identical_to_single_gpu_proof": same,
            "exchange": "same-node shared-memory mailbox: 32 B per rank (commit), 80 B per rank per round, final message, query rows",
            "poseidon2_perm_per_s_aggregate": 4.0 * (1 << nv) / (ms * 1e-3)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="dense4m", choices=list(WORKLOADS))
    ap.add_argument("--only", action="store_true", help="measure only --workload (skip the other BASELINE workloads)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step of each measured workload computed to DIR/<workload>_<name>.npy")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes what the GPU path computed: it needs --impl ours")
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    W = max(args.warmup, 0)
    others = [] if args.only else [k for k in ("cnn264k", "sumcheck20", "basefold24", "dense4m") if k != args.workload]

    if args.impl == "reference":
        if rank != 0:
            return
        K = args.steps if args.steps is not None else 2
        sys.path.insert(0, os.path.join(ROOT, "tests"))
        import oracle_py as O   # the reference arm is one of the two places allowed to execute oracle/
        wl = WORKLOADS[args.workload]()
        cb = cpu_arm(wl, O, K, W)
        extra = {}
        for k in others:
            w2 = WORKLOADS[k]()
            c2 = cpu_arm(w2, O, min(K, 2), 1)
            extra[k] = {"metric": w2.metric, "value": c2["value"], "unit": w2.unit, "cpu_baseline": c2, "workload": w2.name}
        print(json.dumps({
            "impl": "reference", "metric": wl.metric, "value": cb["value"], "unit": wl.unit, "n_gpus": args.gpus, "steps": K,
            "warmup": W, "ms_per_step": 1e3 / cb["value"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": DTYPE, "data": "synthetic", "config": {"workload": wl.name},
            "cpu_baseline": cb,
            "e2e": {"value": cb["value"], "unit": wl.unit, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "workloads": extra,
        }))
        return

    import torch
    import dpb200 as dp
    if not torch.cuda.is_available() or dp.device_count() <= 0:
        raise SystemExit("bench.py: no CUDA device -- the product has no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local_rank)
    cpu_budget()                                 # from the unpinned affinity mask and the container's quota
    pin_to_gpu_numa_node(torch, local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    dp.init(local_rank)
    dp.use_torch_stream()
    env = {"torch": torch, "dp": dp, "dist": dist, "rank": rank, "world": world, "local_rank": local_rank, "peaks": load_peaks(),
           "flush_buf": torch.empty(256 << 20, dtype=torch.uint8, device="cuda"), "no_cpu": args.no_cpu_baseline,
           "sm_count": torch.cuda.get_device_properties(local_rank).multi_processor_count}

    wl = WORKLOADS[args.workload]()
    K = args.steps if args.steps is not None else {"dense4m": 6, "cnn264k": 6, "sumcheck20": 20, "basefold24": 5}[args.workload]
    head = run_gpu_workload(env, wl, K, max(W, 3), True)
    outputs = {args.workload: head.pop("outputs")}
    extra = {}
    for k in others:
        if world > 1 and k in ("sumcheck20", "basefold24"):
            continue      # single-GPU workloads: measured at N = 1 (their N > 1 form is the sharded mode)
        w2 = WORKLOADS[k]()
        k2 = min(K, {"dense4m": 6, "cnn264k": 6, "sumcheck20": 20, "basefold24": 5}[k])
        r2 = run_gpu_workload(env, w2, k2, 3, False)
        outputs[k] = r2.pop("outputs")
        r2.pop("clocks", None)
        if r2.get("roofline"):
            r2["roofline"].pop("kernels", None)     # the per-kernel tables are printed for the headline workload only
            r2["roofline"].pop("kernels_concurrent_batch", None)
        extra[k] = r2
        del w2

    sharded = None
    if world > 1 and not args.only:
        try:
            sharded = {"sumcheck26": sharded_sumcheck(env)}
        except Exception as e:      # the replica numbers above stand on their own
            sharded = {"error": repr(e)[:300]}
        try:
            sharded["basefold24"] = sharded_basefold(env)
        except Exception as e:
            sharded["basefold24"] = {"error": repr(e)[:300]}
    if rank == 0:
        pub = PUBLISHED.get(args.workload)
        out = {
            "metric": head["metric"], "value": head["value"], "unit": head["unit"],
            "n_gpus": world, "steps": K, "warmup": max(W, 3),
            "ms_per_step": head["ms_per_step"], "higher_is_better": True, "scaling": "weak",
            "vs_baseline": (head["value"] / pub) if (pub and world == 1) else None,
            "dtype": DTYPE, "data": "synthetic",
            "config": {"workload": wl.name},
            "run": {"l2": head["l2"],
                    "parallelism": "replicas x%d GPUs (no data-path collective)%s" % (world, (", %d concurrent independent proofs per GPU" % host_workers(wl.STREAMS)) if hasattr(wl, "STREAMS") else ""),
                    "proofs_per_step": head["units_per_step"], "single_stream_latency_ms": head["single_stream_latency_ms"],
                    "host_waits": "throughput legs: dp_set_wait_mode(1) -- proving threads sleep on the library's poller thread; latency leg: spin",
                    "cpu_budget_per_rank": cpu_budget(),
                    "baseline_note": "vs_baseline divides by the reference README's proving time (Dense 4M 2335 ms / CNN 264k 1242 ms; hardware and exact architecture not stated)"},
            "e2e": head["e2e"], "gpu_launches": head["gpu_launches"], "clocks": head["clocks"],
            "roofline": head["roofline"], "cpu_baseline": head["cpu_baseline"], "parity_checked": head["parity_checked"],
            "alg_GBps_whole_step": head["alg_GBps_whole_step"],
            "workloads": extra, "sharded": sharded,
        }
        for k in ("field_ops_per_s", "hbm_frac_whole_proof", "poseidon2_perm_per_s", "pipe_frac_whole_step", "parity_error"):
            if k in head:
                out[k] = head[k]
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, outputs)
        print(json.dumps(out))
    if dist is not None:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
