#!/usr/bin/env python
"""bench.py -- Mcell-iters/s of the PCG pressure solve on the synthetic 256^3 hex cavity
(BASELINE.json metric / configs[1]) + Amul SpMV achieved HBM GB/s against the roofline.

  python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path
  python bench.py --impl reference --gpus N --steps K ...  # the reference's CPU solver, all host cores
  python bench.py ... --dump-outputs DIR                   # also write the last timed step's results to DIR/*.npy

A "step" is what icoFoam does per pressure solve: the assembled coefficients go into the
solver's layout (b200ldu_matrix_set = the reference's calcSortCoeffs, lduMatrix.C:380-471) and
PCG + DIC (=AINV in the reference) runs a fixed number of inner iterations (tolerance 0, so
every implementation does identical work).
value  = nCells(global) * iterations * steps / time, inputs resident in HBM (caller order);
e2e    = the same from HOST buffers: diag/upper/psi/source copied host->device from pinned
         memory, matrix_set, b200ldu_solve, psi copied back -- all inside the timed region.
N > 1: brick decomposition of the same global mesh, one rank per GPU (torchrun) => "strong".
Before anything is timed a parity gate compares the CUDA path with the (N-rank) oracle at the
benchmark size: Amul bit for bit, the first 30 normalised residuals to rel 1e-9.
"""
import argparse
import ctypes as C
import importlib
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


def ncu_traffic():
    """dram__bytes_read.sum + dram__bytes_write.sum per launch from the newest committed `ncu --set full`
    capture of the engine kernels (profiles/r0*_ncu_full_engine_raw.csv): the Amul kernel and one
    steady-state PCG iteration.  None where absent."""
    import csv
    import glob
    out = {"amul": None, "pcg_iteration": None, "source": None}
    files = sorted(glob.glob(os.path.join(ROOT, "profiles", "r0*_ncu_full_engine_raw.csv")))
    if not files:
        return out
    mult = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}
    last, src = {}, {}
    try:
        for p in files:                      # oldest first: the newest capture that holds a kernel wins
            rows = list(csv.reader(open(p)))
            hdr, units = rows[0], rows[1]
            kn, rd, wr = hdr.index("Kernel Name"), hdr.index("dram__bytes_read.sum"), hdr.index("dram__bytes_write.sum")
            for r in rows[2:]:
                byts = float(r[rd]) * mult[units[rd]] + float(r[wr]) * mult[units[wr]]
                for key in ("AmulOp<0>", "PcgAinvOp", "PcgAmulOp"):
                    if key in r[kn]:
                        last[key], src[key] = byts, os.path.relpath(p, ROOT)
        out["source"] = sorted(set(src.values()))
        out["amul"] = last.get("AmulOp<0>")
        if "PcgAinvOp" in last and "PcgAmulOp" in last:
            out["pcg_iteration"] = last["PcgAinvOp"] + last["PcgAmulOp"]
    except Exception:  # noqa: BLE001
        pass
    return out


class ClockSampler:
    """SM clock and clock-event (throttle) reasons sampled DURING the timed region: NVML polled from a thread every ~2 ms (the
    timed region is 35 ms at 8 GPUs -- nvidia-smi's loop mode, used in round 1, returned no sample in that time); nvidia-smi as
    the fallback where the NVML binding is missing."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.rows = []          # nvidia-smi fallback rows
        self.sm, self.mask = [], 0
        self.proc = self.th = self.h = None
        self.idx = gpu_index
        self.stop_flag = threading.Event()
        self.nvml = None
        try:
            import pynvml
            pynvml.nvmlInit()
            idx = gpu_index
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            if vis:
                try:
                    idx = int(vis.split(",")[gpu_index])
                except (ValueError, IndexError):
                    pass
            self.h = pynvml.nvmlDeviceGetHandleByIndex(idx)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
            self.nvml = pynvml
        except Exception:  # noqa: BLE001
            self.nvml = None

    def _poll(self):
        n = self.nvml
        while not self.stop_flag.is_set():
            try:
                self.sm.append(float(n.nvmlDeviceGetClockInfo(self.h, n.NVML_CLOCK_SM)))
                self.mask |= int(n.nvmlDeviceGetCurrentClocksEventReasons(self.h))
            except Exception:  # noqa: BLE001
                break
            time.sleep(0.002)

    def start(self):
        if self.nvml:
            self.th = threading.Thread(target=self._poll, daemon=True)
            self.th.start()
            return
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "20", "-i", str(self.idx)], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if self.nvml:
            self.stop_flag.set()
            self.th.join(timeout=2)
            n = self.nvml
            names = (("hw_slowdown", n.nvmlClocksEventReasonHwSlowdown), ("hw_thermal_slowdown", n.nvmlClocksEventReasonHwThermalSlowdown),
                     ("sw_thermal_slowdown", n.nvmlClocksEventReasonSwThermalSlowdown), ("sw_power_cap", n.nvmlClocksEventReasonSwPowerCap),
                     ("hw_power_brake", n.nvmlClocksEventReasonHwPowerBrakeSlowdown))
            return {"sm_mhz": float(np.median(self.sm)) if self.sm else None, "sm_max_mhz": self.max_mhz,
                    "reasons": sorted(nm for nm, bit in names if self.mask & bit), "samples": len(self.sm), "source": "nvml, 2 ms"}
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm = [float(r[1]) for r in self.rows if len(r) >= 9 and r[1].replace(".", "").isdigit()]
        mx = [float(r[2]) for r in self.rows if len(r) >= 9 and r[2].replace(".", "").isdigit()]
        reasons = set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            if len(r) >= 9:
                for nm, v in zip(names, r[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(nm)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm), "source": "nvidia-smi -lms 20"}


def build_case(meshmod, n, nRanks, rank):
    mesh = meshmod.hex_mesh(n) if nRanks == 1 else meshmod.decompose(n, nRanks, rank)
    coef = meshmod.pressure_laplacian(mesh)
    b = meshmod.cell_field_global(mesh, 9)  # zero-mean-ish random RHS (timing run)
    return mesh, coef, b


def workload_config(n, iters):
    """identical for both arms (the driver compares them)"""
    return {"workload": f"icoFoam cavity {n}^3 hex, PCG+DIC(AINV) pressure solve", "n": n,
            "iterations_per_step": iters, "preconditioner": "DIC->AINV"}


# ---------------------------------------------------------------------------
# CPU arm
# ---------------------------------------------------------------------------
def host_cores():
    """One thread per physical core this process may run on -- NOT what OMP_NUM_THREADS says: torchrun
    exports OMP_NUM_THREADS=1 to its workers, which made the round-1 reference arm single-threaded at
    N > 1.  SMT siblings stay idle (memory-bound row sweeps: 128 threads measured 3x slower than 64)."""
    try:
        aff = sorted(os.sched_getaffinity(0))
    except AttributeError:
        aff = list(range(os.cpu_count() or 1))
    cores = set()
    for c in aff:
        try:
            sib = open(f"/sys/devices/system/cpu/cpu{c}/topology/thread_siblings_list").read().strip()
            cores.add(sib)
        except OSError:
            cores.add(str(c))
    return max(1, len(cores))


def prepare_cpu_arm():
    """Process-wide settings of the CPU arm, before libgomp is loaded: an explicit OpenMP team (one thread
    per physical core, spread and pinned) and page interleaving over the NUMA nodes, so that the arrays the
    harness allocates and first-touches from one thread do not all sit on one memory controller (the
    round-1 numbers swung 110 <-> 388 Mcell-iters/s between boxes)."""
    nT = host_cores()
    os.environ["OMP_NUM_THREADS"] = str(nT)
    os.environ["OMP_PROC_BIND"] = "spread"
    os.environ["OMP_PLACES"] = "cores"
    os.environ.setdefault("OMP_WAIT_POLICY", "active")
    numa = "unavailable"
    try:
        nodes = open("/sys/devices/system/node/online").read().strip()
        ids = []
        for part in nodes.split(","):
            a, _, b = part.partition("-")
            ids += list(range(int(a), int(b or a) + 1))
        if len(ids) > 1:
            mask = 0
            for i in ids:
                mask |= 1 << i
            m = (C.c_ulong * 16)(*([mask & (2 ** 64 - 1)] + [0] * 15))
            libc = C.CDLL(None, use_errno=True)
            MPOL_INTERLEAVE, SYS_set_mempolicy = 3, 238  # x86_64
            rc = libc.syscall(SYS_set_mempolicy, MPOL_INTERLEAVE, m, C.c_ulong(max(ids) + 2))
            numa = f"interleave over {len(ids)} nodes" if rc == 0 else f"set_mempolicy failed (errno {C.get_errno()})"
        else:
            numa = "1 node"
    except Exception as e:  # noqa: BLE001
        numa = f"unavailable ({type(e).__name__})"
    return nT, numa


def set_omp_threads(n):
    """libgomp is shared by the oracle port and the OpenMP build of the reference code: set its team size."""
    try:
        C.CDLL("libgomp.so.1").omp_set_num_threads(int(n))
    except OSError:
        pass


def cpu_pcg(meshmod, orc, mesh, coef, nT):
    """The CPU PCG used by the reference arm and the cpu_baseline leg.  Where the reference's own solver
    sources were compiled here (oracle/_ref/libref_solvers_omp.so: PCG.C, AINVPreconditioner.C,
    lduMatrixATmul.C ... on thrust's OpenMP host back end, oracle/ref_harness/) that code runs, with the
    reference's default favourSpeedOverMemory 2 (etc/controlDict:66) -- kind "reference"; otherwise the
    oracle's OpenMP port -- kind "port".  Returns (run(iters, b) -> nIterations, kind, description)."""
    try:
        from oracle import ref_ldu
        if ref_ldu.omp_available():
            os_, ls, lo = ref_ldu.ldu_arrays(mesh.nCells, mesh.lower, mesh.upper)
            fixed = (mesh.nCells, np.ascontiguousarray(mesh.lower, np.int32), np.ascontiguousarray(mesh.upper, np.int32),
                     os_, ls, lo, np.ascontiguousarray(coef["diag"]), np.ascontiguousarray(coef["upper"]), None)
            set_omp_threads(nT)
            z = np.zeros(mesh.nCells)

            def run_ref(iters, b):
                _, p = ref_ldu.solve("PCG", "DIC", *fixed, z, b, tolerance=0.0, maxIter=iters - 1, favourSpeed=2,
                                     omp=True)
                return p["nIterations"]
            run_ref(1, np.ones(mesh.nCells))   # loads the library, starts the OpenMP team
            return run_ref, "reference", ("reference PCG.C + AINVPreconditioner.C + lduMatrixATmul.C compiled for the "
                                           "host, thrust OpenMP back end")
    except Exception as e:  # noqa: BLE001 -- any problem with the optional library: use the port
        sys.stderr.write(f"reference-code CPU arm unavailable ({e}); using the oracle port\n")
    oa = orc.Addr(mesh.nCells, mesh.lower, mesh.upper)
    om = orc.Matrix(oa, coef["diag"], coef["upper"], None)
    set_omp_threads(nT)

    def run_port(iters, b):
        _, perf = om.pcg_omp("DIC", np.zeros(mesh.nCells), b, nThreads=nT, tolerance=0.0, maxIter=iters - 1)
        return perf.nIterations
    run_port._keep = (oa, om)
    return run_port, "port", "oracle OpenMP rows (oracle/ldu_oracle_omp.c)"


def cpu_baseline_subprocess(n, ci):
    """cpu_baseline of the GPU arm's line: the CPU arm in a FRESH process (so that its OpenMP / NUMA settings
    apply before libgomp is loaded -- this process has torch's libgomp already)."""
    cmd = [sys.executable, os.path.abspath(__file__), "--impl", "reference", "--n", str(n), "--ref-iters", str(ci),
           "--steps", "1", "--warmup", "1", "--with-context"]
    env = {k: v for k, v in os.environ.items() if k not in ("RANK", "WORLD_SIZE", "LOCAL_RANK", "OMP_NUM_THREADS")}
    try:
        p = subprocess.run(cmd, capture_output=True, text=True, timeout=900, env=env, cwd=ROOT)
        line = [ln for ln in p.stdout.splitlines() if ln.startswith("{")][-1]
        d = json.loads(line)
        return d["cpu_baseline"]
    except Exception as e:  # noqa: BLE001
        return {"value": None, "unit": "Mcell-iters/s", "cores": 0, "kind": "port", "sample": f"failed: {e}"}


def run_reference(args, rank, world):
    """CPU arm on all physical host cores: the reference's own PCG loop where it compiled (oracle/_ref), else
    the oracle's OpenMP port -- RapidCFD numerics either way (AINV for DIC).  Rank 0 only under torchrun."""
    if rank != 0:
        return
    nT, numa = prepare_cpu_arm()
    meshmod = importlib.import_module("rapidcfd-dev_b200.mesh")
    from oracle import ldu_oracle as orc
    n = args.n
    mesh, coef, b = build_case(meshmod, n, 1, 0)
    run, kind, what = cpu_pcg(meshmod, orc, mesh, coef, nT)
    iters = args.ref_iters
    for _ in range(args.warmup):
        run(iters, b)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        nit = run(iters, b)
    dt = time.perf_counter() - t0
    assert nit == iters
    val = mesh.nCells * iters * args.steps / dt / 1e6
    cpu = {"value": val, "unit": "Mcell-iters/s", "cores": nT, "kind": kind, "numa": numa,
           "sample": f"{n}^3 cells x {iters} PCG iterations per step, {args.steps} step(s), {dt:.1f} s; {what}"}
    if args.with_context:
        # the oracle's own OpenMP port and stock OpenFOAM's serial DIC-PCG beside it (context, bounded)
        oa = orc.Addr(mesh.nCells, mesh.lower, mesh.upper)
        om = orc.Matrix(oa, coef["diag"], coef["upper"], None)
        if kind == "reference":
            t0 = time.perf_counter()
            om.pcg_omp("DIC", np.zeros(mesh.nCells), b, nThreads=nT, tolerance=0.0, maxIter=iters - 1)
            pdt = time.perf_counter() - t0
            cpu["port"] = {"value": mesh.nCells * iters / pdt / 1e6, "unit": "Mcell-iters/s", "cores": nT,
                           "sample": f"oracle OpenMP rows, {pdt:.1f} s"}
        si = max(2, min(8, iters // 2))
        t0 = time.perf_counter()
        om.pcg_stock_dic(np.zeros(mesh.nCells), b, tolerance=0.0, maxIter=si - 1)
        sdt = time.perf_counter() - t0
        cpu["stock_dic_serial"] = {"value": mesh.nCells * si / sdt / 1e6, "unit": "Mcell-iters/s", "cores": 1,
                                   "sample": f"{n}^3 cells x {si} PCG(true DIC) iterations, serial, {sdt:.1f} s"}
    line = {"impl": "reference", "metric": "Mcell-iters/sec (PCG pressure solve, 256^3 hex cavity)",
            "value": val, "unit": "Mcell-iters/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": workload_config(n, iters), "cpu_baseline": cpu,
            "e2e": {"value": val, "unit": "Mcell-iters/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


# ---------------------------------------------------------------------------
# parity gate (the oracle is the checker here, never the thing measured)
# ---------------------------------------------------------------------------
def gloo_comm(orc, dist, group, mesh, nCellsGlobal, rank, world):
    """exchange layer of the N-rank oracle over a gloo group (host tensors)"""
    import torch
    nbrs = [p.neighbRank for p in mesh.coupled_patches()]

    def halo(send, starts):
        recv = np.empty_like(send)
        ops, bufs = [], []
        for i, nb in enumerate(nbrs):
            s = torch.from_numpy(send[starts[i]:starts[i + 1]].copy())
            r = torch.empty(int(starts[i + 1] - starts[i]), dtype=torch.float64)
            ops.append(dist.P2POp(dist.isend, s, nb, group))
            ops.append(dist.P2POp(dist.irecv, r, nb, group))
            bufs.append((i, r, s))
        for q in dist.batch_isend_irecv(ops):
            q.wait()
        for i, r, _ in bufs:
            recv[starts[i]:starts[i + 1]] = r.numpy()
        return recv

    def _allgather(v):
        t = torch.from_numpy(np.ascontiguousarray(v).copy())
        parts = [torch.empty_like(t) for _ in range(world)]
        dist.all_gather(parts, t, group=group)
        return [p.numpy() for p in parts]

    def allsum(v):
        tot = np.zeros_like(v)
        for p in _allgather(v):  # rank-ordered sum
            tot = tot + p
        return tot

    def gather(mine):
        return np.stack(_allgather(mine))
    return orc.PyComm(halo, allsum, nCellsGlobal, gather, rank, world)


def parity_gate(capi, torch, dist, mesh, coef, b, mat, dev, rank, world, nGlobal, nHist=30):
    """Amul at the benchmark size bit for bit against the (N-rank) oracle; first nHist normalised PCG
    residuals within rel 1e-9 of the oracle's.  Every rank checks its part; the verdict is all-reduced."""
    from oracle import ldu_oracle as orc
    t0 = time.perf_counter()
    comm = None
    if world > 1:
        g = dist.new_group(backend="gloo")
        comm = gloo_comm(orc, dist, g, mesh, nGlobal, rank, world)
    ps, fc = mesh.patch_start_facecells()
    nr = [p.neighbRank for p in mesh.coupled_patches()]
    oa = orc.Addr(mesh.nCells, mesh.lower, mesh.upper, ps, fc, neighbRank=nr if nr else None)
    om = orc.Matrix(oa, coef["diag"], coef["upper"], coef.get("lower"), coef["bou"] if len(coef["bou"]) else None,
                    coef["int"] if len(coef["int"]) else None)
    tt = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)
    A_ref = om.amul(b, comm) if comm else om.amul(b)
    A_gpu = mat.Amul(tt(b)).cpu().numpy()
    amul_ok = bool(np.array_equal(A_gpu, A_ref))
    kw = dict(tolerance=0.0, maxIter=nHist - 1)
    _, perf_ref, hist_ref = om.solve("PCG", "DIC", np.zeros(mesh.nCells), b, comm=comm, histCap=nHist + 4, **kw)
    psi = torch.zeros(mesh.nCells, dtype=torch.float64, device=dev)
    perf, hist = mat.solve("PCG", "DIC", psi, tt(b), histCap=nHist + 4, **kw)
    k = min(nHist, len(hist), len(hist_ref))
    h, hr = np.asarray(hist[:k]), np.asarray(hist_ref[:k])
    rel = float(np.max(np.abs(h - hr) / np.abs(hr))) if k else float("inf")
    its_ok = perf.nIterations == perf_ref.nIterations
    ok = amul_ok and its_ok and rel <= 1e-9
    if world > 1:
        t = torch.tensor([0.0 if ok else 1.0, rel, 0.0 if amul_ok else 1.0], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ok, rel, amul_ok = bool(t[0].item() == 0.0), float(t[1].item()), bool(t[2].item() == 0.0)
    return {"ok": ok, "amul_bit_exact": amul_ok, "hist_max_rel": rel, "hist_entries": int(k),
            "hist_tol": 1e-9, "iterations_equal": bool(its_ok), "oracle": f"{world}-rank oracle (oracle/ldu_oracle.c)",
            "seconds": round(time.perf_counter() - t0, 1)}


# ---------------------------------------------------------------------------
# GPU arm
# ---------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200")
    ap.add_argument("--n", type=int, default=256)
    ap.add_argument("--iters", type=int, default=50, help="PCG iterations per step")
    ap.add_argument("--ref-iters", type=int, default=50,
                    help="PCG iterations per step of the CPU arm (same as --iters: per-solve set-up amortised alike)")
    ap.add_argument("--cpu-baseline-iters", type=int, default=50)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-parity", action="store_true", help="skip the parity gate (profiling runs only)")
    ap.add_argument("--no-secondary", action="store_true", help="skip the PBiCG / GAMG / channel-like legs")
    ap.add_argument("--with-context", action="store_true", help="reference arm: also time the port and stock DIC")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step returned as DIR/<name>.npy")
    args = ap.parse_args()
    args.warmup = max(args.warmup, 3) if args.impl != "reference" else args.warmup

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        return run_reference(args, rank, world)

    import torch
    import torch.distributed as dist
    capi = importlib.import_module("rapidcfd-dev_b200.capi")
    meshmod = importlib.import_module("rapidcfd-dev_b200.mesh")
    assert torch.cuda.is_available(), "bench.py needs a GPU (no CPU fallback)"
    torch.cuda.set_device(local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    assert world == args.gpus, f"--gpus {args.gpus} but WORLD_SIZE={world}"
    n, iters = args.n, args.iters
    mesh, coef, b = build_case(meshmod, n, world, rank)
    nGlobal = n ** 3

    ctx = capi.Context(local)
    if world > 1:
        ctx.comm_init_from_torch()
    dev = ctx.device
    t0 = time.perf_counter()
    addr = capi.mesh_to_device(ctx, mesh)
    t_layout = time.perf_counter() - t0
    mat = capi.LduMatrix(addr)
    tt = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)
    diag, upper = tt(coef["diag"]), tt(coef["upper"])
    bou = tt(coef["bou"]) if len(coef["bou"]) else None
    mat.set(diag, upper, None, bou, bou)
    src = tt(b)
    psi = torch.zeros(mesh.nCells, dtype=torch.float64, device=dev)
    kw = dict(tolerance=0.0, maxIter=iters - 1)
    info = addr.info()
    ar, hp = C.c_int(-1), C.c_int(-1)
    capi.check(capi.lib().b200ldu_comm_info(ctx.h, addr.h, C.byref(ar), C.byref(hp)))
    pathname = {1: "p2p (peer-memory kernels over NVLink)", 0: "nccl", -1: "n/a"}

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(ms):
        if world == 1:
            return ms
        t = torch.tensor([ms], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # ---------------- parity gate at the benchmark size ----------------
    parity = None
    if not args.no_parity:
        parity = parity_gate(capi, torch, dist, mesh, coef, b, mat, dev, rank, world, nGlobal)
        if not parity["ok"]:
            if rank == 0:
                print(json.dumps({"error": "parity gate failed", "parity": parity}), flush=True)
            sys.exit(3)

    # ---------------- device-resident arm: step = matrix_set + solve ----------------
    def step():
        mat.set(diag, upper, None, bou, bou)
        psi.zero_()
        return mat.solve("PCG", "DIC", psi, src, **kw)

    for _ in range(args.warmup):
        perf, _ = step()
    assert perf.nIterations == iters, perf.nIterations
    sampler = ClockSampler(local)
    barrier()
    if rank == 0:
        sampler.start()
    l0 = ctx.launches
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    for _ in range(args.steps):
        perf, _ = step()
    ev1.record()
    barrier()
    ms = max_over_ranks(ev0.elapsed_time(ev1))
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, psi.cpu().numpy(), perf, rank, world)
    launches = ctx.launches - l0
    value = nGlobal * iters * args.steps / (ms * 1e-3) / 1e6
    # the solve alone (round-1 definition of the step), for the roofline of the iteration kernels
    barrier()
    ev0.record()
    for _ in range(args.steps):
        psi.zero_()
        mat.solve("PCG", "DIC", psi, src, **kw)
    ev1.record()
    barrier()
    ms_solve = max_over_ranks(ev0.elapsed_time(ev1))
    value_solve = nGlobal * iters * args.steps / (ms_solve * 1e-3) / 1e6

    # ---------------- Amul kernel alone (roofline) ----------------
    vl = addr.vec_len
    xb = torch.zeros(vl, dtype=torch.float64, device=dev)
    yb = torch.zeros(vl, dtype=torch.float64, device=dev)
    capi.check(capi.lib().b200ldu_to_banded(addr.h, capi._dp(src), capi._dp(xb)))
    nA = 20
    for _ in range(3):
        capi.check(capi.lib().b200ldu_amul_banded(mat.h, capi._dp(xb), capi._dp(yb)))
    barrier()
    a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a0.record()
    for _ in range(nA):
        capi.check(capi.lib().b200ldu_amul_banded(mat.h, capi._dp(xb), capi._dp(yb)))
    a1.record()
    barrier()
    amul_ms = max_over_ranks(a0.elapsed_time(a1) / nA)
    N, F = mesh.nCells, mesh.nFaces
    amul_bytes = 24 * N + 16 * F  # SURVEY.md 8(d): psi, diag, Apsi + upper, owner, neighbour
    amul_gbs = amul_bytes / (amul_ms * 1e-3) / 1e9
    clocks = sampler.stop() if rank == 0 else None
    peak, peak_src = peaks()

    # ---------------- end-to-end arm: HOST coefficients and vectors ----------------
    pin = lambda a: torch.from_numpy(np.ascontiguousarray(a).copy()).pin_memory()
    diag_h, upper_h, src_h = pin(coef["diag"]), pin(coef["upper"]), pin(b)
    psi_h = torch.zeros(mesh.nCells, dtype=torch.float64).pin_memory()
    bou_h = pin(coef["bou"]) if bou is not None else None
    d_diag, d_upper, d_src, d_psi = (torch.empty_like(diag), torch.empty_like(upper), torch.empty_like(src),
                                     torch.empty_like(psi))
    d_bou = torch.empty_like(bou) if bou is not None else None

    def e2e_step(with_coeffs):
        if with_coeffs:
            d_diag.copy_(diag_h, non_blocking=True)
            d_upper.copy_(upper_h, non_blocking=True)
            if d_bou is not None:
                d_bou.copy_(bou_h, non_blocking=True)
            mat.set(d_diag, d_upper, None, d_bou, d_bou)
        d_psi.copy_(psi_h, non_blocking=True)
        d_src.copy_(src_h, non_blocking=True)
        mat.solve("PCG", "DIC", d_psi, d_src, **kw)
        psi_out.copy_(d_psi, non_blocking=True)

    psi_out = torch.empty(mesh.nCells, dtype=torch.float64).pin_memory()

    def e2e_run(with_coeffs):
        for _ in range(2):
            e2e_step(with_coeffs)
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(args.steps):
            e2e_step(with_coeffs)
        e1.record()
        barrier()
        return max_over_ranks(e0.elapsed_time(e1))

    e2e_ms = e2e_run(True)
    e2e_val = nGlobal * iters * args.steps / (e2e_ms * 1e-3) / 1e6
    e2e_vec_ms = e2e_run(False)
    e2e_vec_val = nGlobal * iters * args.steps / (e2e_vec_ms * 1e-3) / 1e6
    h2d = 8 * (nGlobal + sum_faces(meshmod, n, world)) + 16 * nGlobal

    # ---------------- secondary workloads (configs[2..3] building blocks) ----------------
    secondary = None
    if not args.no_secondary:
        secondary = secondary_legs(args, capi, torch, dist, meshmod, ctx, addr, mesh, dev, rank, world, n, nGlobal,
                                   barrier, max_over_ranks, peak)

    # ---------------- CPU baseline (rank 0, N=1 only, bounded sample, own process) ----------------
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cpu = cpu_baseline_subprocess(n, args.cpu_baseline_iters)

    if rank == 0:
        pcg_bytes = (160 * N + 32 * F)  # per iteration and rank, reference op list with AINV (SURVEY 8(d))
        it_ms = ms_solve / (iters * args.steps)
        pcg_gbs = pcg_bytes / (it_ms * 1e-3) / 1e9
        pcg_min_gbs = (104 * N + 32 * F) / (it_ms * 1e-3) / 1e9
        traffic = ncu_traffic()
        line = {
            "metric": "Mcell-iters/sec (PCG pressure solve, 256^3 hex cavity)", "value": value,
            "unit": "Mcell-iters/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic",
            "config": workload_config(n, iters),
            "step": "b200ldu_matrix_set (coefficients into the banded streams) + PCG solve, as icoFoam does per pressure solve",
            "value_solver_only": value_solve, "ms_per_step_solver_only": ms_solve / args.steps,
            "parity": parity,
            "layout": {"decomposition": "x".join(map(str, meshmod.brick_split(world))), "band_rows": info["bandRows"],
                       "bands": info["nBands"], "layout_build_s": round(t_layout, 2),
                       "l2": "inputs >> L2 (1.2 GB per SpMV at 256^3)"},
            "comm": {"halo_path": pathname[hp.value], "allreduce_path": pathname[ar.value]},
            # Dominant kernels of the timed region: the matrix sweeps of the PCG iteration.  One "launch" below =
            # one iteration, timed live as solver-only step time / iterations.  `achieved` uses SURVEY 8(d)'s
            # PCG-iteration figure 160N+32F (the reference's unfused op list) -- the fused sweeps need at least
            # 104N+32F, reported next to it, as is the ncu DRAM traffic.
            "roofline": {"bound": "hbm",
                         "kernel": "fused PCG iteration (AINV sweep + Amul sweep)",
                         "achieved": pcg_gbs, "peak": peak, "unit": "GB/s", "frac": pcg_gbs / peak,
                         "peak_source": peak_src, "algorithmic_bytes_per_launch": pcg_bytes,
                         "ms_per_launch": it_ms, "traffic": traffic["pcg_iteration"] if world == 1 else None,
                         "traffic_source": traffic["source"],
                         "fused": "achieved counts the reference op list's bytes (160N+32F); minimum for the fused pair 104N+32F",
                         "achieved_min_bytes": pcg_min_gbs, "frac_min_bytes": pcg_min_gbs / peak,
                         "dram_gbs": (traffic["pcg_iteration"] / (it_ms * 1e-3) / 1e9) if traffic["pcg_iteration"] and world == 1 else None,
                         "amul": {"kernel": "engine_kernel<AmulOp<0>> (Amul SpMV, banded)", "achieved": amul_gbs,
                                  "frac": amul_gbs / peak, "algorithmic_bytes_per_launch": amul_bytes,
                                  "ms_per_launch": amul_ms, "traffic": traffic["amul"] if world == 1 else None}},
            "cpu_baseline": cpu,
            "e2e": {"value": e2e_val, "unit": "Mcell-iters/s", "h2d_bytes_per_step": h2d,
                    "d2h_bytes_per_step": 8 * nGlobal, "ms_per_step": e2e_ms / args.steps,
                    "what": "pinned host diag/upper/psi/source -> device, matrix_set, solve, psi -> pinned host",
                    "vectors_only": {"value": e2e_vec_val, "ms_per_step": e2e_vec_ms / args.steps,
                                     "h2d_bytes_per_step": 16 * nGlobal,
                                     "what": "coefficients already on the device (the reference's gpuField matrix)"}},
            "secondary": secondary,
            "gpu_launches": int(launches), "clocks": clocks,
            "solver_line": perf.line("p"),
        }
        print(json.dumps(line), flush=True)
    mat.close()
    addr.close()
    ctx.close()
    if world > 1:
        dist.destroy_process_group()


def dump_outputs(path, psi, perf, rank, world):
    """What the last timed step hands its caller, as float64 .npy files: the solution psi and its solver performance.
    psi is a fixed, seeded sample of 2^21 cells over all ranks where it is larger (psi_cells.npy: which cells, in the
    rank's numbering), so that the files stay within 32 MB and two builds can be compared value for value."""
    os.makedirs(path, exist_ok=True)
    sfx = f".rank{rank}" if world > 1 else ""
    cap = (1 << 21) // world
    cells = np.arange(len(psi)) if len(psi) <= cap else np.sort(np.random.default_rng(0).choice(len(psi), cap, replace=False))
    np.save(os.path.join(path, f"psi{sfx}.npy"), psi[cells].astype(np.float64))
    np.save(os.path.join(path, f"psi_cells{sfx}.npy"), cells.astype(np.float64))
    np.save(os.path.join(path, f"solver_performance{sfx}.npy"),
            np.array([perf.initialResidual, perf.finalResidual, perf.normFactor, perf.nIterations, perf.converged,
                      perf.singular], np.float64))


def sum_faces(meshmod, n, world):
    """internal faces held by all ranks together (the coefficients every rank uploads in the e2e arm)"""
    nx, ny, nz = meshmod.brick_split(world)
    a, b_, c = n // nx, n // ny, n // nz
    return world * ((a - 1) * b_ * c + a * (b_ - 1) * c + a * b_ * (c - 1))


def secondary_legs(args, capi, torch, dist, meshmod, ctx, addr, mesh, dev, rank, world, n, nGlobal, barrier,
                   max_over_ranks, peak):
    """Building blocks of BASELINE configs[2..3] on the same mesh, each with its own time, algorithmic bytes
    and roofline fraction: PBiCG + DILU on the momentum matrix (asymmetric), GAMG on the pressure matrix;
    at 8 ranks also a 200^3 (8 M cells) PCG solve, the channel case's size."""
    out = {}
    tt = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)
    N, F = mesh.nCells, mesh.nFaces
    steps = args.steps

    def timed(fn):
        for _ in range(2):
            fn()
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            r = fn()
        e1.record()
        barrier()
        return max_over_ranks(e0.elapsed_time(e1)) / steps, r

    # ---- PBiCG(U) + DILU(->AINV), momentum matrix ----
    try:
        cu = meshmod.momentum_matrix(mesh)
        mu = capi.LduMatrix(addr)
        bouU = tt(cu["bou"]) if len(cu["bou"]) else None
        intU = tt(cu["int"]) if len(cu["int"]) else None
        mu.set(tt(cu["diag"]), tt(cu["upper"]), tt(cu["lower"]), bouU, intU)
        bU = tt(meshmod.cell_field_global(mesh, 11))
        x = torch.zeros(mesh.nCells, dtype=torch.float64, device=dev)
        itU = 20

        def run_u():
            x.zero_()
            return mu.solve("PBiCG", "DILU", x, bU, tolerance=0.0, maxIter=itU - 1)
        msU, (perfU, _) = timed(run_u)
        assert perfU.nIterations == itU
        # reference op list per iteration (PBiCG.C:131-243): 2 AINV (24N+24F each, asymmetric), 2 SpMV (24N+24F),
        # wArT dot 16N, two search-direction updates 24N each, wApT dot 16N, three AXPYs 24N each, sumMag 8N
        bytesU = 4 * (24 * N + 24 * F) + 16 * N + 48 * N + 16 * N + 72 * N + 8 * N
        gbs = bytesU / (msU / itU * 1e-3) / 1e9
        out["pbicg_momentum"] = {"workload": f"{n}^3 momentum matrix (asymmetric), PBiCG + DILU(->AINV), {itU} iterations",
                                 "value": nGlobal * itU / (msU * 1e-3) / 1e6, "unit": "Mcell-iters/s",
                                 "ms_per_solve": msU, "algorithmic_bytes_per_iteration": bytesU,
                                 "achieved_gbs": gbs, "frac": gbs / peak, "solver_line": perfU.line("Ux")}
        mu.close()
    except Exception as e:  # noqa: BLE001
        out["pbicg_momentum"] = {"error": f"{type(e).__name__}: {e}"}

    # ---- GAMG(p), GaussSeidel(->Jacobi) smoother, pressure matrix, to tolerance ----
    try:
        cp = meshmod.pressure_laplacian(mesh)
        mp = capi.LduMatrix(addr)
        bouP = tt(cp["bou"]) if len(cp["bou"]) else None
        mp.set(tt(cp["diag"]), tt(cp["upper"]), None, bouP, bouP)
        t0 = time.perf_counter()
        ag = capi.GamgAgglomeration(addr, meshmod.face_area_pair_weights(mesh), nCellsInCoarsestLevel=10, mergeLevels=1)
        t_agg = time.perf_counter() - t0
        xs_ = meshmod.cell_field_global(mesh, 42)
        bP = mp.Amul(tt(xs_))
        x = torch.zeros(mesh.nCells, dtype=torch.float64, device=dev)

        def run_p():
            x.zero_()
            return mp.solve("GAMG", "GaussSeidel", x, bP, gamg=ag, tolerance=1e-6, relTol=0.0, maxIter=100)
        msP, (perfP, _) = timed(run_p)
        cyc = max(perfP.nIterations, 1)
        # finest-level work of one V-cycle (GAMGSolverSolve.C:181-474 with the defaults: 2 finest sweeps, residual,
        # restrict, prolong + scale on the first coarse level): the coarser levels add ~1x the finest again
        bytesC = 2 * (40 * N + 16 * F) + (32 * N + 16 * F) + 20 * N + 28 * N
        gbs = bytesC / (msP / cyc * 1e-3) / 1e9
        out["gamg_pressure"] = {"workload": f"{n}^3 pressure matrix, GAMG (faceAreaPair, GaussSeidel->Jacobi) to 1e-6",
                                "value": nGlobal * cyc / (msP * 1e-3) / 1e6, "unit": "Mcell-cycles/s",
                                "ms_per_solve": msP, "cycles": perfP.nIterations, "ms_per_cycle": msP / cyc,
                                "levels": int(ag.nLevels),
                                "agglomeration_s": round(t_agg, 2),
                                "algorithmic_bytes_per_cycle_finest_level": bytesC, "achieved_gbs_finest_only": gbs,
                                "frac_finest_only": gbs / peak, "solver_line": perfP.line("p")}
        ag.close()
        mp.close()
    except Exception as e:  # noqa: BLE001
        out["gamg_pressure"] = {"error": f"{type(e).__name__}: {e}"}

    # ---- 8 M cells on 8 ranks (the channel case's size), PCG + DIC ----
    if world == 8 and n != 200:
        try:
            m2 = meshmod.decompose(200, world, rank)
            c2 = meshmod.pressure_laplacian(m2)
            a2 = capi.mesh_to_device(ctx, m2)
            mm = capi.LduMatrix(a2)
            bo = tt(c2["bou"]) if len(c2["bou"]) else None
            mm.set(tt(c2["diag"]), tt(c2["upper"]), None, bo, bo)
            b2 = tt(meshmod.cell_field_global(m2, 9))
            x = torch.zeros(m2.nCells, dtype=torch.float64, device=dev)
            it2 = 50

            def run_c():
                x.zero_()
                return mm.solve("PCG", "DIC", x, b2, tolerance=0.0, maxIter=it2 - 1)
            msC, (perfC, _) = timed(run_c)
            out["channel_size_pcg"] = {"workload": "200^3 hex (8 M cells, the channel case's size; wall-bounded, no cyclics), "
                                                   "8-way 2x2x2, PCG + DIC, 50 iterations",
                                       "value": 200 ** 3 * it2 / (msC * 1e-3) / 1e6, "unit": "Mcell-iters/s",
                                       "ms_per_solve": msC, "solver_line": perfC.line("p")}
            mm.close()
            a2.close()
        except Exception as e:  # noqa: BLE001
            out["channel_size_pcg"] = {"error": f"{type(e).__name__}: {e}"}
    return out


if __name__ == "__main__":
    main()
