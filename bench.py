#!/usr/bin/env python
"""bench.py — MPC solves/sec of the batched update -> solve -> output step (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--workload identical|random] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
        bench.py --gpus N --steps K --warmup W

A "step" is one pass of the hot path over one batch: new measurements in, u* out, for every instance,
in closed loop with the linear plant x+ = Ad x + Bd u (warm-started like the reference's update()).
N=1 workload = BASELINE configs[1]: 65 536 inverted-pendulum instances (nx=4, nu=1, Np=20) per GPU.
`value` : device-resident inputs (timed with CUDA events on the launching stream, max over ranks).
`e2e`   : the same metric through MPCController.update()/output() with pinned HOST buffers (H2D + D2H inside).
`configs`: (N=1) BASELINE configs[2] (random x0/xref, 1 000 warm steps) and configs[3] (MIMO nx=8 nu=4 Np=40, B=16 384),
           each with device / e2e throughput, solver statistics, an oracle spot check and its own roofline entry.
Multi-GPU: batch sharded over ranks (weak scaling, 65 536 instances per GPU); u* of every rank lands in every rank's
gathered buffer (peer stores fused into the solver epilogue + one arrival-flag kernel, or one NCCL all-gather with
--nccl-gather); the gathered buffer is verified against an NCCL all-gather after the timed loop.
The oracle (oracle/) is used ONLY for the cpu_baseline leg, the spot checks and --impl reference.
--dump-outputs DIR: after the run, DIR/u.npy holds u* [global batch, nu] (float64) of the last timed step of the device-resident loop
and DIR/u_e2e.npy that of the end-to-end loop (--impl reference: DIR/u.npy of the last timed CPU step).  The inputs are seeded, so
runs with the same arguments can be compared output for output.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True          # the benchmark writes nothing into the tree it runs from

B_PER_GPU = 65536
ALG_BYTES_PER_ITER = 24 * (188 + 2 * 209)     # SURVEY.md §8d: 24 (n + 2 m) on the reference QP dims = 14 544 B
METRIC = "mpc_solves_per_sec"
UNIT = "solves/s"
SYS_KEYS = ("Qx", "QxN", "Qu", "QDu", "xmin", "xmax", "umin", "umax", "Dumin", "Dumax", "eps_feas")


def pendulum_batch(B, workload, seed=0):
    from pympc_b200.workloads import pendulum, pendulum_random
    cfg = pendulum()
    if workload == "random":
        X0, Xref = pendulum_random(B, seed)
    else:
        X0 = np.tile(cfg["x0"], (B, 1)); Xref = np.tile(cfg["xref"], (B, 1))
    return cfg, np.ascontiguousarray(X0), np.ascontiguousarray(Xref)


def mimo_batch(B, seed=4):
    from pympc_b200.workloads import mimo
    cfg = mimo(); rng = np.random.default_rng(seed)
    return cfg, np.ascontiguousarray(0.3 * rng.standard_normal((B, 8))), np.ascontiguousarray(np.tile(cfg["xref"], (B, 1)))


def dump_outputs(out_dir, arrays):
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), np.ascontiguousarray(a, dtype=np.float64))


def load_json(*path):
    try:
        return json.load(open(os.path.join(ROOT, *path)))
    except Exception:
        return {}


# ---------------------------------------------------------------------------------------------- clocks
class ClockSampler:
    """Samples SM clock and throttle reasons DURING the timed region.  The timed region is only tens of milliseconds, far
    below nvidia-smi's start-up time, so NVML is polled in-process (every ~2 ms) from a background thread; nvidia-smi is
    the fallback."""
    REASONS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap"}

    def __init__(self, index):
        self.index, self.sm, self.bits, self.max_mhz = index, [], 0, None
        self._stop = threading.Event(); self._thr = None; self._h = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self._nv = pynvml
            self._h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self._h, pynvml.NVML_CLOCK_SM))
        except Exception:
            self._h = None

    def _poll(self):
        nv = self._nv
        while not self._stop.is_set():
            try:
                self.sm.append(float(nv.nvmlDeviceGetClockInfo(self._h, nv.NVML_CLOCK_SM)))
                try:
                    self.bits |= int(nv.nvmlDeviceGetCurrentClocksEventReasons(self._h))
                except Exception:
                    self.bits |= int(nv.nvmlDeviceGetCurrentClocksThrottleReasons(self._h))
            except Exception:
                pass
            time.sleep(0.002)

    def start(self):
        if self._h is not None:
            self._thr = threading.Thread(target=self._poll, daemon=True); self._thr.start()

    def stop(self):
        if self._thr is not None:
            self._stop.set(); self._thr.join(timeout=1)
        if not self.sm:
            try:     # fallback: one nvidia-smi query right after the timed region
                out = subprocess.run(["nvidia-smi", f"--id={self.index}", "--query-gpu=clocks.sm,clocks.max.sm",
                                      "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=10).stdout
                a, b = [float(v) for v in out.strip().split(",")[:2]]
                self.sm, self.max_mhz = [a], b
            except Exception:
                pass
        reasons = sorted(n for bit, n in self.REASONS.items() if self.bits & bit)
        return {"sm_mhz": float(np.median(self.sm)) if self.sm else None, "sm_max_mhz": self.max_mhz,
                "reasons": reasons, "samples": len(self.sm)}


# ---------------------------------------------------------------------------------------------- CPU arm
def cpu_arm(steps, warmup, sample_b, workload, threads=None, **settings):
    """Closed-loop steps of the oracle's C restatement of OSQP (one solver object per instance, OpenMP over
    instances, reference default eps=1e-3 like MPCController passes, mpc.py:266)."""
    from oracle.qp_assembly import QPData
    from oracle import osqp_port
    osqp_port.build()
    cfg, X0, Xref = pendulum_batch(sample_b, workload)
    Q = QPData(**cfg)
    bc = osqp_port.BatchCPU(Q, sample_b, **settings)         # OSQP defaults: eps 1e-3, adaptive rho, warm start
    X = X0.copy(); U = np.zeros((sample_b, 1))
    Ad, Bd = cfg["Ad"], cfg["Bd"]
    if threads is None:
        # give the CPU its best shot: the container may expose fewer cores than os.cpu_count() (cgroup quota), so
        # pick the fastest thread count among a few candidates on untimed steps
        try:
            navail = len(os.sched_getaffinity(0))
        except Exception:
            navail = os.cpu_count() or 1
        best = None
        for cand in sorted({navail, max(1, navail // 2), 64, 32, 16, 8}):
            if cand > navail:
                continue
            t0 = time.perf_counter(); Un, st, it = bc.step(X, U, Xref, nthreads=cand); dt = time.perf_counter() - t0
            U = Un; X = X @ Ad.T + U @ Bd.T
            if best is None or dt < best[0]:
                best = (dt, cand)
        threads = best[1]
    times, iters = [], []
    for t in range(warmup + steps):
        t0 = time.perf_counter()
        Un, st, it = bc.step(X, U, Xref, nthreads=threads)
        dt = time.perf_counter() - t0
        if t >= warmup:
            times.append(dt); iters.append(it.mean())
        U = Un; X = X @ Ad.T + U @ Bd.T
    bc.close()
    tot = float(np.sum(times))
    return {"u": Un, "value": sample_b * steps / tot, "unit": UNIT, "cores": int(threads), "kind": "port",
            "sample": f"{sample_b} pendulum instances x {steps} closed-loop steps ({workload}), OSQP-port eps={settings.get('eps_abs', 1e-3):g}, "
                      f"mean {np.mean(iters):.0f} ADMM its/solve, solver-only (no Python per-instance overhead)",
            "ms_per_step": 1e3 * tot / steps}


# ---------------------------------------------------------------------------------------------- roofline
def roofline_entries(shape_key, acc, steps, peaks):
    """One entry per kernel family of the timed steps.  fp64-pipe work = (thread-level fp64-pipe instructions counted in the
    SASS of the compiled kernel, profiles/fp64_ops.json, per active-set refinement / ADMM iteration) x (refinements /
    iterations the device counted) x 2 flop (every fp64-pipe instruction is charged like a DFMA), over the CUDA-event time of
    that kernel family, against the DFMA peak measured on this B200 pool (profiles/fp64_peak.json, tools/ubench_fp64.cu).
    DRAM: bytes per launch from the committed ncu capture of the same kernel over the same time, against MEASURED_PEAKS."""
    ops = load_json("profiles", "fp64_ops.json").get(shape_key, {})
    fpk = load_json("profiles", "fp64_peak.json")
    peak_tf = float(fpk.get("dfma_tflops", 34.19))
    hbm = float(peaks.get("hbm_gbs", 6650.0))
    out = []
    fams = (("polish", ops.get("polish_kernel", "k_polish"), acc["ms_polish"], acc["polish_steps"], ops.get("fp64_per_refinement"), ops.get("polish_dram_bytes_per_launch")),
            ("admm", ops.get("admm_kernel", "k_admm"), acc["ms_admm"], acc["admm_iters"], ops.get("fp64_per_admm_iteration"), ops.get("admm_dram_bytes_per_launch")))
    tot_ms = acc["ms_polish"] + acc["ms_admm"]
    for fam, name, ms, units, per_unit, dram in fams:
        if ms <= 0 or tot_ms <= 0 or ms / tot_ms < 0.10:
            continue
        e = {"kernel": name, "family": fam, "share_of_kernel_time": ms / tot_ms, "ms_per_step": ms / steps, "work_units": int(units)}
        if per_unit:
            tf = 2.0 * per_unit * units / (ms * 1e-3) / 1e12
            e.update({"bound": "fp64", "achieved": tf, "peak": peak_tf, "unit": "TFLOP/s (fp64-pipe instructions x 2)", "frac": tf / peak_tf,
                      "fp64_instr_per_unit": per_unit})
        if dram:
            gbs = dram * steps / (ms * 1e-3) / 1e9
            e.update({"traffic": dram, "dram_gbs": gbs, "dram_frac_of_hbm_peak": gbs / hbm})
        out.append(e)
    out.sort(key=lambda e: -e["share_of_kernel_time"])
    return out, peak_tf, hbm


# ---------------------------------------------------------------------------------------------- GPU loops
class Gather:
    """K6: every rank's u* in every rank's gathered buffer [2][Btot, nu] (double-buffered by step parity: step t+1's peer
    stores go to the other half, so they can never race a peer still reading step t).  Fused mode: the solver epilogue stores
    into all peers' buffers over NVLink (symmetric memory) and one small kernel publishes / awaits per-rank arrival flags;
    NCCL mode: one in-place all-gather."""

    def __init__(self, K, torch, dist, dev, B, nu, rank, world, use_nccl):
        self.K, self.torch, self.dist, self.rank, self.world, self.B, self.nu = K, torch, dist, rank, world, B, nu
        self.Btot = B * world; self.s = rank * B; self.e = self.s + B
        self.fused = False; self.epoch = 0
        L, h = K._L, K.handle
        if world > 1 and not use_nccl:
            try:
                import ctypes as ct
                import torch.distributed._symmetric_memory as symm_mem
                self.buf = symm_mem.empty((2, self.Btot, nu), dtype=torch.float64, device=dev); self.buf.zero_()
                self.hs = symm_mem.rendezvous(self.buf, dist.group.WORLD)
                self.flags = symm_mem.empty((world,), dtype=torch.int64, device=dev); self.flags.zero_()
                self.hf = symm_mem.rendezvous(self.flags, dist.group.WORLD)
                self.peer_bufs = [int(p) for p in self.hs.buffer_ptrs]
                self.peer_flags = [int(p) for r, p in enumerate(self.hf.buffer_ptrs) if r != rank]
                self.fused = True
                self.attach()
                dist.barrier(); torch.cuda.synchronize(dev)
            except Exception as exc:                               # pragma: no cover
                self.fused = False
                if rank == 0:
                    print("symmetric memory unavailable, using the NCCL all-gather:", exc, file=sys.stderr)
        if not self.fused:
            self.buf = torch.zeros(2, self.Btot, nu, dtype=torch.float64, device=dev)
        self.bind(0)

    def attach(self):
        """(re)bind the arrival flags to the controller's current handle (setup() creates a new one)"""
        if self.fused:
            import ctypes as ct
            arr = (ct.c_void_p * len(self.peer_flags))(*self.peer_flags)
            assert self.K._L.bmpc_bind_gather_flags(self.K.handle, self.flags.data_ptr(), arr, len(self.peer_flags), self.rank, self.world, self.epoch) == 0

    def bind(self, parity):
        """point the solver epilogue at this step's half of the gathered buffer (own slice + the same slice of every peer)"""
        import ctypes as ct
        L, h = self.K._L, self.K.handle
        self.parity = parity
        self.Uloc = self.buf[parity, self.s:self.e]
        self.K._external_output = True                             # the controller must not rebind its own pinned result arrays
        L.bmpc_bind_output(h, self.Uloc.data_ptr())
        if self.fused:
            off = (parity * self.Btot + self.s) * self.nu * 8
            peers = [p + off for r, p in enumerate(self.peer_bufs) if r != self.rank]
            arr = (ct.c_void_p * len(peers))(*peers)
            assert L.bmpc_bind_output_peers(h, arr, len(peers)) == 0

    def finish_step(self):
        """after output(): make the step's gathered buffer complete on this rank"""
        if self.world == 1:
            return
        if self.fused:
            self.epoch += 1
            assert self.K._L.bmpc_gather_arrive(self.K.handle, self.epoch) == 0
        else:
            from pympc_b200.dist import allgather_outputs
            allgather_outputs(self.buf[self.parity], self.s, self.e)

    def gathered(self):
        return self.buf[self.parity]

    def verify(self):
        """gathered buffer of the last step == NCCL all-gather of the ranks' own u* (every rank checks its whole buffer)"""
        if self.world == 1:
            return True
        torch, dist = self.torch, self.dist
        ref = torch.empty(self.Btot, self.nu, dtype=torch.float64, device=self.buf.device)
        dist.all_gather_into_tensor(ref, self.Uloc.contiguous())
        ok = torch.tensor([1.0 if torch.equal(ref, self.gathered()) else 0.0], device=self.buf.device)
        dist.all_reduce(ok, op=dist.ReduceOp.MIN)
        return bool(ok.item() == 1.0)


def device_loop(torch, dist, K, cfg, X0, steps, warmup, dev, world, gather, flush, sampler=None, t_off=0):
    """timed region of `value`: inputs resident in HBM, CUDA events on the launching stream around every step"""
    L, h = K._L, K.handle
    # ONE explicit stream for the solver, the L2 flush, the plant and the timing events.  (torch's default stream has handle 0,
    # which bmpc_set_stream reads as "use the handle's own stream": the flush would then overlap the solver kernels and the
    # events would not bracket them — round 1's bench had that flaw.)
    stream = torch.cuda.Stream(dev)
    torch.cuda.synchronize(dev)
    assert stream.cuda_stream != 0
    L.bmpc_set_stream(h, stream.cuda_stream)
    torch.cuda.set_stream(stream)
    Ad = torch.tensor(cfg["Ad"], device=dev); Bd = torch.tensor(cfg["Bd"], device=dev)
    Xd = torch.tensor(X0, device=dev); Xn = torch.empty_like(Xd)
    acc = dict(admm_iters=0, ms_admm=0.0, ms_polish=0.0, launches=0, polish_steps=0, unsolved=0); rounds = []; tot_ms = 0.0
    for t in range(warmup + steps):
        if t == warmup:
            torch.cuda.synchronize(dev)
            if world > 1:
                dist.barrier()
            torch.cuda.synchronize(dev)
            if sampler is not None:
                sampler.start()
        gather.bind((t + t_off) & 1)
        Uprev = gather.buf[((t + t_off) & 1) ^ 1, gather.s:gather.e]    # u* of the previous step = this step's u_-1
        flush.zero_()                                             # L2 flush between timed iterations (outside the events)
        e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        L.bmpc_update(h, Xd.data_ptr(), Uprev.data_ptr(), None, 1, 2)     # device-resident inputs, read in place (borrowed)
        rc = L.bmpc_solve(h)
        assert rc == 0, L.bmpc_last_error(h)
        L.bmpc_output(h, None, None, 1, 1)
        gather.finish_step()
        e1.record(stream)
        # the user's plant (not the hot path): x+ = Ad x + Bd u on the device, outside the timed window
        torch.matmul(Xd, Ad.T, out=Xn); Xn.addmm_(gather.Uloc, Bd.T)
        st = K.stats()
        torch.cuda.synchronize(dev)
        Xd, Xn = Xn, Xd
        if t >= warmup:
            tot_ms += e0.elapsed_time(e1)
            for k in acc:
                acc[k] += st[k]
            rounds.append(st["rounds"])
    torch.cuda.synchronize(dev)
    torch.cuda.set_stream(torch.cuda.default_stream(dev))
    if world > 1:
        dist.barrier()
    tmax = torch.tensor([tot_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
    return float(tmax.item()), acc, rounds, Xd


def e2e_loop(torch, dist, K, cfg, X0, steps, warmup, dev, world, gather, flush):
    """`e2e`: the public API with pinned HOST buffers — H2D of x0 and u_-1, solve, D2H of u* inside the timed region (and, at
    N > 1, the gather of u* into every rank's buffer)."""
    L, h = K._L, K.handle
    L.bmpc_set_stream(h, None)
    Xh = K.pinned_buffer("x0"); Uh = K.pinned_buffer("uminus1")
    Xh[...] = X0; Uh[...] = 0.0
    K.setup(solve=True); K.output()
    L, h = K._L, K.handle
    gather.attach()
    Adn, Bdn = cfg["Ad"], cfg["Bd"]
    e2e_t = 0.0
    for t in range(warmup + steps):
        if t == warmup and world > 1:
            dist.barrier()
        if world > 1:
            gather.bind(t & 1)                                 # N = 1: u* goes straight into the controller's pinned result array
        flush.zero_(); torch.cuda.synchronize(dev)
        t0 = time.perf_counter()
        K.update(Xh, Uh)                                       # H2D of x0, uminus1 + solve + D2H of u, status
        Uo = K.output()
        if world > 1:
            gather.finish_step(); L.bmpc_synchronize(h)
            if not gather.fused:
                torch.cuda.synchronize(dev)
        dt = time.perf_counter() - t0
        if t >= warmup:
            e2e_t += dt
        Uh[...] = Uo; Xh[...] = Xh @ Adn.T + Uo @ Bdn.T        # host plant, outside the timed region
    te = torch.tensor([e2e_t], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(te, op=dist.ReduceOp.MAX)
    return float(te.item()), Xh.copy(), Uh.copy()


def oracle_spot_check(K, cfg, X, Xref, Um1, n=8, seed=3):
    """max |u_gpu - u_oracle| over n sampled instances: one more solve through the public API at the state the loop reached,
    against the oracle's exact KKT solver on the reference-assembled QP of each sampled instance"""
    from oracle.qp_assembly import QPData
    from oracle.kkt import solve_exact
    K.update(X, Um1); U = K.output()
    rng = np.random.default_rng(seed); err = 0.0
    for b in rng.choice(X.shape[0], size=n, replace=False):
        c = dict(cfg); c["x0"] = X[b]; c["xref"] = Xref[b]; c["uminus1"] = Um1[b]
        Q = QPData(**c); z, y, r = solve_exact(Q.P, Q.q, Q.A, Q.l, Q.u)
        nu = U.shape[1]
        err = max(err, float(np.max(np.abs(U[b] - z[Q.NX:Q.NX + nu]))))
    return err


def make_controller(cfg, X0, Xref, B, device, **opts):
    from pympc_b200 import MPCController
    nu = cfg["Bd"].shape[1]
    K = MPCController(cfg["Ad"], cfg["Bd"], Np=cfg["Np"], x0=X0, xref=Xref, uminus1=np.zeros(nu), batch=B, device=device,
                      **{k: cfg[k] for k in SYS_KEYS if k in cfg}, **opts)
    K.setup(solve=False)
    return K


def side_config(torch, dist, dev, name, cfg, X0, Xref, steps, warmup, shape_key, peaks, flush, settle_steps=0):
    """one extra BASELINE config on rank 0 of a single-GPU run: device + e2e throughput, solver statistics, oracle spot check"""
    B = X0.shape[0]; nu = cfg["Bd"].shape[1]
    K = make_controller(cfg, X0, Xref, B, dev.index)
    t0 = time.perf_counter(); K.solve(); K.output(); torch.cuda.synchronize(dev)
    cold_ms = 1e3 * (time.perf_counter() - t0); cold = K.stats()
    G = Gather(K, torch, dist, dev, B, nu, 0, 1, True)
    tot_ms, acc, rounds, Xd = device_loop(torch, dist, K, cfg, X0, steps, warmup, dev, 1, G, flush)
    settled = None
    if settle_steps > 0:
        # the same closed loop continued until the transient is over: the regime a controller spends its life in
        s_ms, s_acc, s_rounds, Xd = device_loop(torch, dist, K, cfg, Xd.cpu().numpy(), steps, settle_steps, dev, 1, G, flush, t_off=steps + warmup)
        settled = {"after_steps": steps + warmup + settle_steps, "steps": steps, "value": B * steps / (s_ms * 1e-3), "unit": UNIT, "ms_per_step": s_ms / steps,
                   "solver": {"mean_rounds": float(np.mean(s_rounds)), "unsolved": int(s_acc["unsolved"]), "admm_iters_per_solve": s_acc["admm_iters"] / (B * steps),
                              "refinements_per_solve": s_acc["polish_steps"] / (B * steps)}}
    e2e_steps = min(steps, 200)
    K._L.bmpc_bind_output(K.handle, None)
    e2e_t, Xh, Uh = e2e_loop(torch, dist, K, cfg, X0, e2e_steps, warmup, dev, 1, G, flush)
    err = oracle_spot_check(K, cfg, Xh, Xref, Uh)
    K.close()
    kern, peak_tf, hbm = roofline_entries(shape_key, acc, steps, peaks)
    return {"workload": name, "batch": B, "steps": steps, "value": B * steps / (tot_ms * 1e-3), "unit": UNIT, "ms_per_step": tot_ms / steps,
            "e2e": {"value": B * e2e_steps / e2e_t, "unit": UNIT, "steps": e2e_steps, "ms_per_step": 1e3 * e2e_t / e2e_steps},
            "solver": {"mean_rounds": float(np.mean(rounds)), "unsolved": int(acc["unsolved"]), "admm_iters_per_solve": acc["admm_iters"] / (B * steps),
                       "refinements_per_solve": acc["polish_steps"] / (B * steps), "launches_per_step": acc["launches"] / steps},
            "cold_first_solve": {"ms": cold_ms, "rounds": cold["rounds"], "unsolved": cold["unsolved"]},
            "oracle_spot_check": {"instances": 8, "max_abs_err_u": err, "tol": 1e-6, "ok": bool(err < 1e-6)},
            "roofline": kern, **({"settled": settled} if settled else {})}


def gpu_arm(args, rank, world, local_rank):
    import torch
    import torch.distributed as dist
    from pympc_b200 import build
    from pympc_b200.dist import shard_range
    if rank == 0:
        build.build()
    if world > 1:
        dist.barrier()
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    # weak scaling (the contract's default): 65 536 instances per GPU; --scaling strong: BASELINE configs[4]'s 524 288 in total
    B = B_PER_GPU if args.scaling == "weak" else (8 * B_PER_GPU) // world
    Btot = B * world
    s, e = shard_range(Btot, rank, world)
    cfgp, X0all, Xrefall = pendulum_batch(Btot, args.workload)
    X0, Xref = X0all[s:e], Xrefall[s:e]
    K = make_controller(cfgp, X0, Xref, B, local_rank)
    torch.cuda.synchronize(dev)
    t0 = time.perf_counter()
    K.solve(); K.output()                                      # cold first solve (zero start), reported separately
    cold_ms = 1e3 * (time.perf_counter() - t0)
    cold = dict(K.stats(), ms=cold_ms)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)   # > 126 MB L2
    G = Gather(K, torch, dist, dev, B, 1, rank, world, args.nccl_gather)
    sampler = ClockSampler(local_rank) if rank == 0 else None
    tot_ms_max, acc, rounds, Xd = device_loop(torch, dist, K, cfgp, X0, args.steps, args.warmup, dev, world, G, flush, sampler)
    clocks = sampler.stop() if rank == 0 else None
    dumped = {"u": G.gathered().cpu().numpy()} if args.dump_outputs else None
    gather_ok = G.verify()
    # ---- end-to-end through the public API with pinned host buffers (H2D and D2H inside the timed region)
    e2e_t, Xh, Uh = e2e_loop(torch, dist, K, cfgp, X0, args.steps, args.warmup, dev, world, G, flush)
    gather_ok_e2e = G.verify()
    if dumped is not None:
        dumped["u_e2e"] = G.gathered().cpu().numpy() if world > 1 else Uh
    if world > 1 and not (gather_ok and gather_ok_e2e):
        raise SystemExit(f"rank {rank}: gathered u* buffer differs from the NCCL all-gather of the ranks' outputs")
    K.close()
    if rank != 0:
        return None
    if dumped is not None:
        dump_outputs(args.dump_outputs, dumped)
    peaks = load_json("MEASURED_PEAKS.json")
    shape_key = "pendulum_4_1_20_20"
    kern, peak_tf, hbm = roofline_entries(shape_key, acc, args.steps, peaks)
    top = kern[0] if kern else {}
    # secondary, SURVEY 8d's figure: "algorithmic" bytes of the reference's sparse ADMM iteration; the condensed iterate never
    # leaves the SM, so this is NOT a bound (kept for continuity with round 1 and labelled as such)
    alg = None
    if acc["ms_admm"] > 0 and acc["admm_iters"] > 0:
        a_gbs = acc["admm_iters"] * ALG_BYTES_PER_ITER / (acc["ms_admm"] * 1e-3) / 1e9
        alg = {"achieved_gbs": a_gbs, "frac_of_hbm_peak": a_gbs / hbm, "note": "on-chip, not a bound: 24(n+2m)=14544 B per instance-iteration of the reference-form QP"}
    value = Btot * args.steps / (tot_ms_max * 1e-3)
    par = f"batch-shard x{world}"
    if world > 1:
        par += (", u* gathered by peer stores fused into the solver epilogue (NVLink symmetric memory, double-buffered), arrival flags raised and awaited by the solver kernel's last warp (no collective, no extra launch)"
                if G.fused else ", 1 NCCL all-gather of u*/step")
    out = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": tot_ms_max / args.steps, "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None,
        "dtype": "f64", "data": "synthetic",
        "config": {"workload": f"inverted_pendulum nx=4 nu=1 Np=20, batch={B} per GPU ({args.workload} instances), "
                               "closed loop with the linear plant, warm start (BASELINE configs[1])",
                   "global_batch": Btot, "parallelism": par,
                   "l2": "flushed between timed steps (256 MiB write)", "parity": "u* within 1e-6 of the KKT-certified optimum (polish on)"},
        "e2e": {"value": Btot * args.steps / e2e_t, "unit": UNIT, "h2d_bytes_per_step": int(B * (4 + 1) * 8 * world),
                "d2h_bytes_per_step": int(B * 8 * world), "ms_per_step": 1e3 * e2e_t / args.steps,
                "note": "x0 + u_-1 fetched from pinned (device-mapped) host memory by the solver kernel itself while it computes, u* stored "
                        "straight into pinned host memory by its epilogue (N = 1; at N > 1 u* goes to the gathered device buffer and is "
                        "copied D2H): the PCIe bytes per step are the same as with explicit copies, there is no separate copy phase" + ("; the gather of u* across ranks is inside the timed region" if world > 1 else "") +
                        "; the 4-byte status per instance is read back only in steps where some instance was not KKT-verified"},
        "gpu_launches": int(acc["launches"]),
        "roofline": {"bound": top.get("bound", "fp64"), "kernel": top.get("kernel"), "achieved": top.get("achieved"), "peak": top.get("peak", peak_tf),
                     "unit": top.get("unit", "TFLOP/s"), "frac": top.get("frac"), "traffic": top.get("traffic"),
                     "peak_source": "profiles/fp64_peak.json: DFMA peak measured on this B200 pool by tools/ubench_fp64.cu (of measured); "
                                    "DRAM fractions against MEASURED_PEAKS.json hbm_gbs" + (" (of measured)" if peaks else " (fallback 6650 GB/s)"),
                     "note": "dominant kernel of the timed steps; achieved = fp64-pipe instructions (SASS count per refinement x refinements counted "
                             "on the device) x 2 flop / CUDA-event time of that kernel; ncu's sm__pipe_fp64_cycles_active of the same kernel is in profiles/",
                     "kernels": kern, "algorithmic_hbm_secondary": alg,
                     "ms_admm": acc["ms_admm"], "ms_polish": acc["ms_polish"]},
        "solver": {"mean_rounds": float(np.mean(rounds)), "unsolved": int(acc["unsolved"]),
                   "admm_iters_per_solve": acc["admm_iters"] / (B * args.steps), "refinements_per_solve": acc["polish_steps"] / (B * args.steps)},
        "cold_first_solve": {"ms": cold["ms"], "solves_per_sec": B / (cold["ms"] * 1e-3), "rounds": cold["rounds"],
                             "admm_iters_per_solve": cold["admm_iters"] / B, "unsolved": cold["unsolved"],
                             "note": "rank 0's shard, zero warm start, host wall clock around solve()+output(); not in value"},
        "clocks": clocks,
    }
    if world > 1:
        out["gather_verified"] = bool(gather_ok and gather_ok_e2e)
    if world == 1 and not args.no_configs:
        # BASELINE configs[2] and configs[3] next to the headline (same process, same GPU, < 60 s)
        cfgs = {}
        try:
            c3, X3, R3 = pendulum_batch(B_PER_GPU, "random")
            cfgs["random_1000"] = side_config(torch, dist, dev, "configs[2]: inverted pendulum, per-instance random x0/xref, 1000 warm closed-loop steps, B=65536",
                                              c3, X3, R3, 1000, 3, "pendulum_4_1_20_20", peaks, flush)
        except Exception as exc:                                   # pragma: no cover
            cfgs["random_1000"] = {"error": repr(exc)}
        try:
            c4, X4, R4 = mimo_batch(16384)
            cfgs["mimo_16384"] = side_config(torch, dist, dev, "configs[3]: MIMO reference-governor shape nx=8 nu=4 Np=40, B=16384, random x0; value = steps 4-13 of the transient from a cold start, settled = the same loop 60 steps later",
                                             c4, X4, R4, 10, 3, "mimo_8_4_40_40", peaks, flush, settle_steps=60)
        except Exception as exc:                                   # pragma: no cover
            cfgs["mimo_16384"] = {"error": repr(exc)}
        out["configs"] = cfgs
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="native", choices=["native", "reference"])
    ap.add_argument("--workload", default="identical", choices=["identical", "random"])
    ap.add_argument("--cpu-sample", type=int, default=4096)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-configs", action="store_true", help="skip the configs[2] / configs[3] side measurements")
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"], help="strong: 524 288 instances in total (configs[4])")
    ap.add_argument("--nccl-gather", action="store_true", help="use the NCCL all-gather instead of fused peer stores")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write u* of the last timed step to DIR/*.npy")
    args = ap.parse_args()
    if args.warmup < 3:
        args.warmup = 3
    rank = int(os.environ.get("RANK", "0")); world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))

    if args.impl == "reference":
        if rank != 0:
            return
        cb = cpu_arm(args.steps, args.warmup, args.cpu_sample, args.workload)
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, {"u": cb["u"]})
        line = {"impl": "reference", "metric": METRIC, "value": cb["value"], "unit": UNIT, "n_gpus": args.gpus,
                "steps": args.steps, "warmup": args.warmup, "ms_per_step": cb["ms_per_step"], "higher_is_better": True,
                "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
                "config": {"workload": f"inverted_pendulum nx=4 nu=1 Np=20 ({args.workload} instances), bounded sample of "
                                       f"{args.cpu_sample} instances per step on the host cores", "global_batch": args.cpu_sample,
                           "parallelism": f"openmp x{cb['cores']}"},
                "cpu_baseline": {k: cb[k] for k in ("value", "unit", "cores", "kind", "sample")},
                "e2e": {"value": cb["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                "gpu_launches": 0}
        print(json.dumps(line))
        return

    import torch
    import torch.distributed as dist
    # native libraries (NCCL's version banner, ...) write to file descriptor 1: park it on stderr while the run is in
    # progress so that stdout carries exactly the one JSON line of rank 0
    sys.stdout.flush()
    saved_stdout = os.dup(1); os.dup2(2, 1)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        if os.environ.get("NCCL_DEBUG", "VERSION").upper() == "VERSION":
            os.environ["NCCL_DEBUG"] = "WARN"                  # keep NCCL's version banner off stdout: rank 0 prints ONE JSON line
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    out = gpu_arm(args, rank, world, local_rank)
    if rank == 0:
        if not args.no_cpu_baseline and world == 1:
            cb = cpu_arm(3, 1, args.cpu_sample, args.workload)
            out["cpu_baseline"] = {k: cb[k] for k in ("value", "unit", "cores", "kind", "sample")}
        elif not args.no_cpu_baseline:
            out["cpu_baseline"] = None
    sys.stdout.flush(); os.dup2(saved_stdout, 1); os.close(saved_stdout)
    if rank == 0:
        print(json.dumps(out), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
