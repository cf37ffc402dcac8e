#!/usr/bin/env python
"""bench.py -- molecules/sec of PaiNN energy+forces (fwd + analytic bwd) on B200.

Contract (task statement): `python bench.py --gpus N --steps K --warmup W` prints ONE JSON
line on rank 0.  A "step" = one E+F pass of the hot path over one batch of 256 synthetic
drug-like conformations per GPU (BASELINE.json configs[1]); `value` = whole-job molecules/s
with inputs resident in HBM; `e2e` = the same through the reference-facing module with HOST
buffers (pinned H2D of z/pos/n_atoms and D2H of E,F inside the timed region every step).

`--impl reference` times the CPU oracle restatement of the reference path (the reference
itself cannot be imported on this image: schnetpack/PyG/e3nn absent) on all host cores.

`--dump-outputs DIR` writes the energies and forces of the last timed step as DIR/energy.npy and
DIR/forces.npy (float32).  Inputs and weights are seeded, so two builds run with the same arguments
can be compared output for output.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.path.insert(0, os.path.join(ROOT, "tests", "golden"))

METRIC = "molecules/sec (PaiNN E+F fwd+bwd)"
B_PER_GPU = 256
N_POOL = 4  # distinct synthetic batches cycled through the timed steps
CATS = ["neighbor_build", "radial_filter", "embedding", "node_gemm", "node_elementwise", "msg_fwd", "msg_bwd", "readout", "force_assembly"]


def load_peaks():
    """(HBM GB/s, dense TF32 TFLOP/s, source).  TF32 tensor peak = half the measured sustained bf16 cuBLAS throughput (the node kernels run
    inside a long step), the 3xTF32 pass factor is applied to the FLOP count, not to the peak."""
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            d = json.load(open(p))
            return float(d["hbm_gbs"]), float(d["bf16_tflops_sustained"]) / 2.0, "measured (MEASURED_PEAKS.json hbm_gbs, bf16_tflops_sustained / 2 for TF32)"
        except Exception:
            pass
    return 6650.0, 1125.0 / 2 * 1.0, "fallback (B200_PROFILING.md 6.65 TB/s; nominal dense TF32 = 2250 / 2 / 2 TFLOP/s)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""

    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, gpu_index):
        self.rows, self.proc, self.gpu = [], None, gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100", "-i", str(self.gpu)],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
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
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


def dump_outputs(directory, energy, forces):
    """What a caller of the timed path receives from one step: per-molecule energies [n_mol], per-atom forces [n_atoms, 3]."""
    import numpy as np

    os.makedirs(directory, exist_ok=True)
    for name, t in (("energy", energy), ("forces", forces)):
        np.save(os.path.join(directory, name + ".npy"), t.detach().cpu().float().numpy())


def build_model(kind, device):
    import torch
    from helpers import load_golden_weights

    if kind in ("painn", "schnet"):
        from nabladft_b200 import spk

        rep_cls = spk.PaiNN if kind == "painn" else spk.SchNet
        m = spk.NeuralNetworkPotential(
            representation=rep_cls(n_atom_basis=128, n_interactions=6, radial_basis=spk.GaussianRBF(n_rbf=100, cutoff=5.0),
                                   cutoff_fn=spk.CosineCutoff(cutoff=5.0)),
            input_modules=[spk.PairwiseDistances()], output_modules=[spk.Atomwise(n_in=128, output_key="energy"), spk.Forces()],
            postprocessors=[spk.AddOffsets(property="energy", add_mean=True)])
    else:
        from nabladft_b200.painn_oc import PaiNN

        m = PaiNN(hidden_channels=128, num_layers=6, num_rbf=100, cutoff=5.0, max_neighbors=100, direct_forces=False, use_pbc=False, num_elements=100)
    load_golden_weights(m, torch.float32)  # random-init weights of the reference architecture (seeded, name-keyed)
    return m.eval().to(device)


def build_oracle(kind, ours):
    import torch

    sd = {k: v.detach().cpu().float() for k, v in ours.state_dict().items()}
    if kind in ("painn", "schnet"):
        from oracle.spk import NeuralNetworkPotential as O
        from oracle.spk import SpkPaiNN, SpkSchNet

        ref = O(SpkPaiNN() if kind == "painn" else SpkSchNet())
        ref.load_state_dict({k: sd[k] for k in ref.state_dict()}, strict=True)
    else:
        from oracle.painn_oc import PaiNNOC

        ref = PaiNNOC(hidden_channels=128, num_layers=6, num_rbf=100, cutoff=5.0, max_neighbors=100, num_elements=100)
        ref.load_state_dict(sd, strict=True)
    return ref.eval()


def oracle_pass(kind, ref, b, n_mol, dtype=None):
    """One CPU E+F pass of the oracle over the first n_mol molecules of batch b (neighbour list inside)."""
    import torch
    from oracle.graph import ase_neighbor_list

    n_at = int(b["mol_ptr"][n_mol])
    z = torch.from_numpy(b["z"][:n_at]).long()
    pos = torch.from_numpy(b["pos"][:n_at]).to(dtype or torch.float32)
    batch = torch.from_numpy(b["batch"][:n_at])
    if kind in ("painn", "schnet"):
        ptr = torch.from_numpy(b["mol_ptr"][: n_mol + 1]).long()
        idx_i, idx_j = ase_neighbor_list(pos, ptr, 5.0)
        out = ref({"_atomic_numbers": z, "_positions": pos.clone(), "_idx_i": idx_i, "_idx_j": idx_j, "_idx_m": batch})
        return out["energy"], out["forces"]
    return ref(z, pos.clone(), batch)


def pick_threads(kind, ref, b):
    """Eager PyTorch on many-core hosts slows down when every tiny op fans out to all cores;
    give the CPU arm its best intra-op thread count (tried: 8, 16, 32, 64, all)."""
    import torch

    ncpu = os.cpu_count() or 1
    best, best_t = ncpu, float("inf")
    for n in sorted({min(c, ncpu) for c in (8, 16, 32, 64, ncpu)}):
        torch.set_num_threads(n)
        oracle_pass(kind, ref, b, 4)
        t0 = time.perf_counter()
        oracle_pass(kind, ref, b, 8)
        dt = time.perf_counter() - t0
        if dt < best_t:
            best, best_t = n, dt
    torch.set_num_threads(best)
    return best


def cpu_baseline(kind, ours, b, sample_mols, reps, gpu_e=None, gpu_f=None):
    """The oracle timed on the host cores (fp32, as the reference runs) + PARITY of the device outputs of the same bench batch against a
    float64 pass of the oracle over the same `sample_mols` molecules (north_star: 1e-5 Ha, 1e-4 Ha/A)."""
    import torch

    ref = build_oracle(kind, ours)
    cores = pick_threads(kind, ref, b)
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        oracle_pass(kind, ref, b, sample_mols)
        ts.append(time.perf_counter() - t0)
    out = {"value": sample_mols / statistics.median(ts), "unit": "molecules/s", "cores": cores, "kind": "port",
           "sample": f"{reps} E+F passes over the first {sample_mols} molecules of the bench batch, oracle restatement "
                     f"(fp32, torch {torch.__version__}, {cores} threads = best of 8/16/32/64/all on {os.cpu_count()} host cores), neighbour list inside the timed region"}
    if gpu_e is not None:
        e64, f64 = oracle_pass(kind, ref.double(), b, sample_mols, dtype=torch.float64)
        n_at = int(b["mol_ptr"][sample_mols])
        out["parity"] = {"max_dE": float((gpu_e[:sample_mols].double().cpu() - e64.detach()).abs().max()),
                         "max_dF": float((gpu_f[:n_at].double().cpu() - f64.detach()).abs().max()),
                         "n_mol": sample_mols, "n_atoms": n_at, "max_abs_E": float(e64.detach().abs().max()),
                         "against": "float64 pass of the oracle over the same molecules; tolerances 1e-5 Ha / 1e-4 Ha/A"}
    return out


def train_record(args, dev, rank, world, storage="f32"):
    """BASELINE configs[2] shape as a sub-record of the same line: PaiNN E+F TRAINING step on 256 synthetic conformations per GPU --
    forward, MSE(E) + MSE(F) (config/model/painn.yaml:30-46), backward through the engine (analytic parameter gradients incl. the force-loss
    double backward), ONE gradient all-reduce from a pre-flattened bucket on a side stream, AdamW step.  `storage`: "f32" (the reference
    trains in fp32) or "bf16" = configs[2]'s "bf16": per-edge arrays (filter rows, their distance derivative, per-edge filter gradients)
    stored as bf16, fp32 arithmetic everywhere.  Does not change the headline metric."""
    import torch

    from nabladft_b200.parallel import GradBucket, max_over_ranks
    from nabladft_b200.synth import synth_batch

    model = build_model(args.model, dev).train()
    model.train_edge_storage = storage
    bucket = GradBucket(model.parameters())
    opt = torch.optim.AdamW(model.parameters(), lr=1e-5)
    pool = []
    for k in range(2):
        b = synth_batch(1 + k, B_PER_GPU)
        n_atoms = torch.from_numpy(b["mol_ptr"][1:] - b["mol_ptr"][:-1]).to(dev)
        if args.model == "painn":
            inputs = {"_atomic_numbers": torch.from_numpy(b["z"]).to(dev), "_positions": torch.from_numpy(b["pos"]).to(dev),
                      "_idx_m": torch.from_numpy(b["batch"]).to(dev), "_n_atoms": n_atoms}
        else:
            class _D:
                pass
            inputs = _D()
            inputs.z, inputs.pos, inputs.batch, inputs.num_graphs = torch.from_numpy(b["z"]).to(dev), torch.from_numpy(b["pos"]).to(dev), torch.from_numpy(b["batch"]).to(dev), B_PER_GPU
        g = torch.Generator(device="cpu").manual_seed(k)
        pool.append((inputs, torch.randn(B_PER_GPU, generator=g).to(dev), (0.1 * torch.randn(b["pos"].shape[0], 3, generator=g)).to(dev)))
    ar_ms = []

    def step(k):
        inputs, target, f_target = pool[k % len(pool)]
        bucket.zero()
        out = model(inputs)
        en, fo = (out["energy"], out["forces"]) if isinstance(out, dict) else out
        loss = ((en - target) ** 2).mean() + ((fo - f_target) ** 2).mean()
        loss.backward()
        n = bucket.allreduce()
        opt.step()
        return n

    for k in range(2):
        n_grad = step(k)
    torch.cuda.synchronize()
    if world > 1:
        torch.distributed.barrier()
    steps = args.steps
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for k in range(steps):
        step(k)
    e1.record()
    torch.cuda.synchronize()
    t = bucket.last_allreduce_ms()  # the last step's all-reduce (CUDA events on the side stream)
    if t is not None:
        ar_ms.append(t)
    ms = max_over_ranks(e0.elapsed_time(e1) / steps, dev)
    return {"workload": "PaiNN E+F training step, MSE(E) + MSE(F), AdamW, 256 synthetic conformations per GPU (BASELINE configs[2] shape)",
            "ms_per_step": ms, "value": world * B_PER_GPU / (ms / 1e3), "unit": "molecules/s", "steps": steps,
            "dtype": "f32" if storage == "f32" else "bf16 storage of the per-edge arrays (W, dW/dd, per-edge filter gradients), f32 arithmetic / weights / gradients",
            "allreduce_elements": n_grad, "allreduce_us": (1e3 * sum(ar_ms) / len(ar_ms)) if ar_ms else None,
            "allreduce": "one flat fp32 bucket (GradBucket), NCCL on a side stream"}


def run_reference(args):
    import torch
    from nabladft_b200.synth import synth_batch

    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    kind = args.model
    b = synth_batch(1, B_PER_GPU)
    # weights: same seeded recipe as the CUDA arm, built on CPU (no CUDA needed for this arm)
    from helpers import load_golden_weights
    if kind in ("painn", "schnet"):
        from oracle.spk import NeuralNetworkPotential as O
        from oracle.spk import SpkPaiNN, SpkSchNet
        ref = load_golden_weights(O(SpkPaiNN() if kind == "painn" else SpkSchNet()), torch.float32).eval()
    else:
        from oracle.painn_oc import PaiNNOC
        ref = load_golden_weights(PaiNNOC(), torch.float32).eval()
    cores = pick_threads(kind, ref, b)
    sample = args.ref_sample
    for _ in range(max(1, min(args.warmup, 2))):
        oracle_pass(kind, ref, b, min(8, sample))
    t0 = time.perf_counter()
    for _ in range(args.steps):
        out = oracle_pass(kind, ref, b, sample)
    dt = time.perf_counter() - t0
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, *out)
    val = args.steps * sample / dt
    line = {
        "impl": "reference", "metric": METRIC, "value": val, "unit": "molecules/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": {"workload": f"PaiNN ({'config/painn.yaml, schnetpack semantics' if kind == 'painn' else 'config/painn-oc.yaml'}) "
                               f"energy+forces inference, 256-molecule synthetic batch (<=30 heavy atoms); each step = bounded sample of {sample} molecules",
                   "model": kind},
        "cpu_baseline": {"value": val, "unit": "molecules/s", "cores": cores, "kind": "port",
                         "sample": f"{args.steps} steps x {sample} molecules; CPU oracle restatement of the reference path (reference not importable: schnetpack/PyG absent)"},
        "e2e": {"value": val, "unit": "molecules/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--model", default="painn", choices=["painn", "painn-oc", "schnet"])
    ap.add_argument("--ref-sample", type=int, default=32, help="molecules per step of the CPU reference arm")
    ap.add_argument("--cpu-sample", type=int, default=32)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--streams", type=int, default=3, help="independent batches in flight on separate CUDA streams (value leg)")
    ap.add_argument("--batch", type=int, default=256, help="molecules per GPU per step (BASELINE config 2 = 256; other values are experiments)")
    ap.add_argument("--gemm", default="tc", choices=["tc", "cublas"], help="node GEMM backend: tcgen05 3xTF32 (default) or cuBLAS SGEMM")
    ap.add_argument("--node", default="fused", choices=["fused", "unfused"], help="per-atom part of a layer: fused tcgen05 kernels (default) or one launch per op (round 1)")
    ap.add_argument("--skip-e2e", action="store_true", help="profiling runs only (ncu): device-resident leg only")
    ap.add_argument("--no-train", action="store_true", help="skip the training sub-record (BASELINE configs[2] shape)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the energies and forces of the last timed step to DIR/energy.npy, DIR/forces.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3)
    global B_PER_GPU
    B_PER_GPU = args.batch
    if args.impl == "reference":
        return run_reference(args)

    import numpy as np
    import torch
    import torch.distributed as dist

    from nabladft_b200 import _lib
    from nabladft_b200.synth import synth_batch

    rank, world = int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    model = build_model(args.model, dev)
    post = True
    eng = model.engine(post) if args.model in ("painn", "schnet") else model.engine()
    _lib.check(eng.lib.nb200_engine_set_gemm_backend(eng._h, 1 if args.gemm == "tc" else 0), "set_gemm_backend")
    if args.model != "schnet":
        _lib.check(eng.lib.nb200_engine_set_node_backend(eng._h, 1 if args.node == "fused" else 0), "set_node_backend")
    # weak scaling: 256 conformations per GPU per step.  Every rank cycles the SAME seeded pool of synthetic batches, i.e. identical
    # atoms / edges per rank and step: the scaling curve then shows the machine (host threads, clocks, NCCL), not the luck of the draw
    # (round 1 used rank-dependent seeds and reported max over ranks of DIFFERENT batches; per-rank times are in the line now)
    pool_host = [synth_batch(1 + k, B_PER_GPU) for k in range(N_POOL)]
    pool_dev = [dict(z=torch.from_numpy(b["z"]).to(dev), pos=torch.from_numpy(b["pos"]).to(dev), mol_ptr=torch.from_numpy(b["mol_ptr"]).to(dev)) for b in pool_host]
    n_atoms = [int(b["z"].shape[0]) for b in pool_host]
    eng.e_cap = max(n_atoms) * 32

    def step_dev(k, e=None):
        d = pool_dev[k % N_POOL]
        return (e or eng).launch(d["z"], d["pos"], d["mol_ptr"], B_PER_GPU, with_forces=True)

    # ---- warm-up (also validates status once, grows capacity if the guess was short)
    for k in range(args.warmup):
        e, f, st = step_dev(k)
        sth = st.cpu()
        if int(sth[1]) == -4:
            eng.e_cap = int(int(sth[0]) * 1.1) + 1024
            e, f, st = step_dev(k)
            sth = st.cpu()
        eng.raise_on_status(sth)
    n_edges = []
    for k in range(N_POOL):
        _, _, st = step_dev(k)
        n_edges.append(int(st.cpu()[0]))
    barrier()

    # ---- timed region: K steps, inputs resident in HBM, no host sync inside
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
        time.sleep(0.3)
    # independent 256-conformation batches are pipelined over `--streams` CUDA streams (one engine = cuBLAS handle +
    # workspace per stream, shared weights): the tail of one step overlaps the head of the next.  Device time is
    # taken between an event all streams wait on and an event that waits on all streams.
    n_str = max(1, args.streams)
    engines = [eng] + [eng.clone_for_stream() for _ in range(n_str - 1)]
    for e_ in engines:
        _lib.check(e_.lib.nb200_engine_set_gemm_backend(e_._h, 1 if args.gemm == "tc" else 0), "set_gemm_backend")
        if args.model != "schnet":
            _lib.check(e_.lib.nb200_engine_set_node_backend(e_._h, 1 if args.node == "fused" else 0), "set_node_backend")
        e_.e_cap = eng.e_cap
    streams = [torch.cuda.Stream() for _ in range(n_str)]
    for i_, (e_, s_) in enumerate(zip(engines, streams)):  # allocate workspaces outside the timed region
        with torch.cuda.stream(s_):
            step_dev(i_, e_)
    barrier()
    launches0 = sum(e_.lib.nb200_engine_own_launches(e_._h) for e_ in engines)
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    ev0.record()
    for s_ in streams:
        s_.wait_event(ev0)
    last = [None] * n_str
    for k in range(args.steps):
        with torch.cuda.stream(streams[k % n_str]):
            last[k % n_str] = step_dev(k, engines[k % n_str])
    for s_ in streams:
        torch.cuda.current_stream().wait_stream(s_)
    ev1.record()
    barrier()
    ms = ev0.elapsed_time(ev1)
    launches = sum(e_.lib.nb200_engine_own_launches(e_._h) for e_ in engines) - launches0
    for r_ in last:
        if r_ is not None:
            eng.raise_on_status(r_[2].cpu())
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, *last[(args.steps - 1) % n_str][:2])
    e, f, st = step_dev(0)
    torch.cuda.synchronize()
    eng.raise_on_status(st.cpu())
    from nabladft_b200.parallel import max_over_ranks
    ms_max = max_over_ranks(ms, dev)  # device time of the job = slowest rank
    value = world * args.steps * B_PER_GPU / (ms_max / 1e3)
    per_rank_ms = [ms / args.steps]
    if world > 1:
        gathered = [torch.zeros(1, dtype=torch.float64, device=dev) for _ in range(world)]
        dist.all_gather(gathered, torch.tensor([ms / args.steps], dtype=torch.float64, device=dev))
        per_rank_ms = [float(g.item()) for g in gathered]

    # ---- e2e: reference-facing module call with HOST (pinned) buffers, H2D + D2H every step
    pinned = []
    for b in pool_host:
        nat = np.diff(b["mol_ptr"]).astype(np.int64)
        pinned.append(dict(z=torch.from_numpy(b["z"].astype(np.int64)).pin_memory(), pos=torch.from_numpy(b["pos"]).pin_memory(),
                           n_atoms=torch.from_numpy(nat).pin_memory(), batch=torch.from_numpy(b["batch"]).pin_memory()))

    class _D:
        pass

    # e2e: each step's inputs start in pinned HOST memory and its results end in pinned HOST memory; steps are
    # pipelined over the same `--streams` streams through the module's public async call, and a slot's buffers are
    # only reused after its stream has been synchronised (= that step's D2H read has completed).
    e2e_streams = streams if args.model in ("painn", "schnet") else streams[:1]
    model.eval()
    S2 = len(e2e_streams)
    out_e = [torch.empty(B_PER_GPU, dtype=torch.float32).pin_memory() for _ in range(S2)]
    out_f = [torch.empty(max(n_atoms), 3, dtype=torch.float32).pin_memory() for _ in range(S2)]
    out_st = [torch.zeros(4, dtype=torch.int32).pin_memory() for _ in range(S2)]

    def step_e2e(k):
        slot = k % S2
        h = pinned[k % N_POOL]
        e2e_streams[slot].synchronize()  # results of step k - S2 are now readable on the host
        with torch.cuda.stream(e2e_streams[slot]):
            z = h["z"].to(dev, non_blocking=True)
            pos = h["pos"].to(dev, non_blocking=True)
            if args.model in ("painn", "schnet"):
                # the reference-facing call: module.forward(batch_dict) (what AtomisticTaskFixed / the calculators call); asynchronous,
                # its status check is deferred to the next call on the same stream's engine and to model.check() below
                out = model({"_atomic_numbers": z, "_positions": pos, "_idx_m": h["batch"].to(dev, non_blocking=True),
                             "_n_atoms": h["n_atoms"].to(dev, non_blocking=True)})
                en, fo = out["energy"], out["forces"]
            else:
                d = _D()
                d.z, d.pos, d.batch, d.num_graphs = z, pos, h["batch"].to(dev, non_blocking=True), B_PER_GPU
                en, fo = model(d)
            out_e[slot].copy_(en, non_blocking=True)
            out_f[slot][: fo.shape[0]].copy_(fo, non_blocking=True)

    if args.skip_e2e:
        if rank == 0:
            sampler.stop()
            print(json.dumps({"profiling_only": True, "value": value, "ms_per_step": ms_max / args.steps}), flush=True)
        return
    for k in range(3 * S2):
        step_e2e(k)
    barrier()
    e2e_steps = args.steps
    ev0.record()
    for s_ in e2e_streams:
        s_.wait_event(ev0)
    for k in range(e2e_steps):
        step_e2e(k)
    for s_ in e2e_streams:
        torch.cuda.current_stream().wait_stream(s_)
    ev1.record()
    barrier()
    model.check()  # deferred status words of every asynchronous forward() above
    ms_e2e = ev0.elapsed_time(ev1)
    e2e_value = world * e2e_steps * B_PER_GPU / (max_over_ranks(ms_e2e, dev) / 1e3)
    navg = sum(n_atoms) / len(n_atoms)
    h2d = int(navg * (8 + 12 + 8) + B_PER_GPU * 8)  # z int64, pos f32x3, idx_m int64, n_atoms int64
    d2h = int(B_PER_GPU * 4 + navg * 12)
    clocks = sampler.stop() if rank == 0 else None

    # ---- per-category kernel timing (CUDA events on the launch stream) -> roofline of K_msg
    eng.lib.nb200_engine_set_timing(eng._h, 1)
    prof_steps = min(args.steps, 10)
    for k in range(prof_steps):
        step_dev(k)
    torch.cuda.synchronize()
    import ctypes
    ms_cat = (ctypes.c_float * 16)()
    n_cat = (ctypes.c_int32 * 16)()
    _lib.check(eng.lib.nb200_engine_read_timings(eng._h, ms_cat, n_cat, 16), "read_timings")
    eng.lib.nb200_engine_set_timing(eng._h, 0)
    breakdown = {CATS[i]: {"ms_per_step": ms_cat[i] / prof_steps, "launch_groups_per_step": n_cat[i] / prof_steps} for i in range(len(CATS))}

    train_rec = None
    if not (args.no_train or args.model == "schnet"):  # configs[2] names bf16: that variant is the record, the fp32 step rides along
        train_rec = train_record(args, dev, rank, world, "bf16")
        f32 = train_record(args, dev, rank, world, "f32")
        train_rec["f32"] = {k: f32[k] for k in ("ms_per_step", "value", "unit", "dtype")}

    if rank == 0:
        peak, tpeak, peak_src = load_peaks()
        L, F = 6, 128
        N_avg = sum(n_atoms[k % N_POOL] for k in range(prof_steps)) / prof_steps
        E_avg = sum(n_edges[k % N_POOL] for k in range(prof_steps)) / prof_steps
        ms = {k: v["ms_per_step"] for k, v in breakdown.items()}
        # SURVEY.md section 8d definition A: algorithmic bytes per launch (one layer) of the message kernels; the filter kernel writes W and dW/dd
        bytes_bwd = N_avg * 16 * F * 4 + E_avg * (6 * F * 4 + 32)
        bytes_fwd = N_avg * 10 * F * 4 + E_avg * (3 * F * 4 + 20)
        fused = args.node == "fused" and args.model != "schnet"
        # filter rows: fused path = ONE [W | dW/dd] record per undirected pair (E/2 rows of 6F floats per layer), else W and dW per directed edge
        bytes_filter = (E_avg / 2 * 16 + L * (E_avg / 2) * 6 * F * 4) if fused else (E_avg * 16 + 2 * L * E_avg * 3 * F * 4)
        # node kernels (painn_fused.cu): fp32-equivalent FLOPs of the Linear layers they contain, forward + input gradients
        #   fwd / layer: 2 (3*F*2F + 2F*F + F*3F + F*F + F*3F); bwd / layer: update 2 (3F*F + F*2F + 3*2F*F), message MLP (layers > 0) 2 (3F*F + F*F)
        flop_atom = L * 2 * (3 * F * 2 * F + 2 * F * F + F * 3 * F + F * F + F * 3 * F) + L * 2 * (3 * F * F + F * 2 * F + 3 * 2 * F * F) \
            + (L - 1) * 2 * (3 * F * F + F * F) + 2 * 2 * F * (F // 2)
        flops_node = N_avg * flop_atom            # fp32-equivalent per step
        t_node = (ms["node_gemm"] + ms["node_elementwise"]) * 1e-3
        n_node = breakdown["node_gemm"]["launch_groups_per_step"]
        node_name = "k_node_fwd + k_node_bwd (painn_fused.cu)" if fused else "k_gemm_tf32x3* + node elementwise kernels"
        ach_node = 3 * flops_node / t_node / 1e12  # three TF32 MMA passes per fp32-accurate product
        entries = {
            node_name: {"bound": "tensor", "achieved": ach_node, "peak": tpeak, "unit": "TFLOP/s", "frac": ach_node / tpeak, "ms_per_step": t_node * 1e3,
                        "launches_per_step": n_node, "algorithmic_flops_per_step_fp32": flops_node,
                        "note": "achieved = 3 x fp32-equivalent FLOPs (3xTF32: lo.hi + hi.lo + hi.hi) / time; peak = TF32 dense = bf16_tflops_sustained / 2"},
            "k_filter": {"bound": "hbm", "achieved": bytes_filter / (ms["radial_filter"] * 1e-3) / 1e9, "peak": peak, "unit": "GB/s",
                         "ms_per_step": ms["radial_filter"], "algorithmic_bytes_per_launch": bytes_filter},
            "k_painn_msg_bwd": {"bound": "hbm", "achieved": bytes_bwd / (ms["msg_bwd"] / L * 1e-3) / 1e9, "peak": peak, "unit": "GB/s",
                                "ms_per_step": ms["msg_bwd"], "avg_launch_ms": ms["msg_bwd"] / L, "algorithmic_bytes_per_launch": bytes_bwd},
            "k_painn_msg_fwd": {"bound": "hbm", "achieved": bytes_fwd / (ms["msg_fwd"] / L * 1e-3) / 1e9, "peak": peak, "unit": "GB/s",
                                "ms_per_step": ms["msg_fwd"], "avg_launch_ms": ms["msg_fwd"] / L, "algorithmic_bytes_per_launch": bytes_fwd},
        }
        for v in entries.values():
            v.setdefault("frac", v["achieved"] / v["peak"])
        t_sum = sum(ms.values())
        for v in entries.values():
            v["share_of_kernel_time"] = v["ms_per_step"] / t_sum
        dominant = max(entries, key=lambda k: entries[k]["ms_per_step"])
        traffic = None
        tpath = os.path.join(ROOT, "profiles", "traffic.json")
        if os.path.exists(tpath):
            try:
                traffic = json.load(open(tpath)).get(dominant.split(" ")[0])
            except Exception:
                traffic = None
        d = entries[dominant]
        roofline = {"kernel": dominant, "bound": d["bound"], "achieved": d["achieved"], "peak": d["peak"], "unit": d["unit"], "frac": d["frac"],
                    "traffic": traffic, "peak_source": peak_src, "share_of_kernel_time": d["share_of_kernel_time"],
                    "serial_kernel_ms_per_step": t_sum, "atoms": N_avg, "edges": E_avg,
                    "detail": {k: v for k, v in d.items() if k not in ("bound", "achieved", "peak", "unit", "frac")},
                    "also": {k: v for k, v in entries.items() if k != dominant and v["share_of_kernel_time"] >= 0.05}}
        line = {
            "metric": METRIC, "value": value, "unit": "molecules/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_max / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic",
            "config": {"workload": f"PaiNN ({'config/painn.yaml, schnetpack semantics' if args.model == 'painn' else 'config/painn-oc.yaml'}) "
                                   "energy+forces inference, 256-molecule synthetic batch per GPU (<=30 heavy atoms, seeded, random-init weights)",
                       "model": args.model, "node_gemm": ("fused tcgen05 3xTF32 node kernels (painn_fused.cu)" if args.node == "fused" and args.model != "schnet" else "tcgen05 3xTF32 GEMM per Linear (gemm_tc.cu)") if args.gemm == "tc" else "cuBLAS SGEMM", "molecules_per_gpu_per_step": B_PER_GPU, "atoms_per_step": N_avg, "edges_per_step": E_avg,
                       "parallelism": f"replicas x{world} (independent molecules, no data-path collective)", "streams_in_flight": max(1, args.streams),
                       "per_rank_batches": "same seeded pool on every rank (identical atoms / edges per rank and step)",
                       "l2": "per-step working set (filters W,dW = 2x6xEx1536 B ~ 3.5 GB) >> 126 MB L2; 4 distinct batches cycled"},
            "e2e": {"value": e2e_value, "unit": "molecules/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h, "steps": e2e_steps,
                    "streams_in_flight": S2,
                    "api": "nabladft_b200.spk.NeuralNetworkPotential.forward(batch_dict), one call per step, steps round-robin over the CUDA streams" if args.model in ("painn", "schnet") else "nabladft_b200.PaiNN.forward(data)"},
            "gpu_launches": int(launches), "clocks": clocks, "roofline": roofline, "kernel_breakdown_ms": breakdown,
            "per_rank_ms_per_step": per_rank_ms, "train": train_rec,
        }
        if not args.no_cpu_baseline and world == 1:
            line["cpu_baseline"] = cpu_baseline(args.model, model, pool_host[0], args.cpu_sample, 3, e, f)
            line["parity"] = line["cpu_baseline"].get("parity")
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
