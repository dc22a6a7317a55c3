#!/usr/bin/env python
"""bench.py -- DeepFM (dac_ctr) training throughput over the HBM parameter server.

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path
    python bench.py --impl reference --gpus N --steps K ...  # CPU restatement of the Go PS path

One step = one pass of the PS hot path over one synthetic Criteo-shaped batch
(BASELINE.json configs[1]): pull dense -> unique -> pull rows of 76 tables -> tower
fwd/bwd -> dedup-sum -> push with fused Adam -> version++.  Prints ONE JSON line.

`value`   : whole-job samples/s with inputs resident in HBM (CUDA events, max over ranks)
`e2e`     : same metric with the step's ids/features/labels copied from pinned host
            memory and the loss copied back every step, inside the timed region
`roofline`: the dominant PS kernel's algorithmic bytes / CUDA-event duration vs the
            measured HBM copy bandwidth (MEASURED_PEAKS.json)
`cpu_baseline`: the oracle's C restatement of the Go PS path on the host cores
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

ADAM_ARGS = "learning_rate=0.001;beta_1=0.9;beta_2=0.999;epsilon=1e-07;amsgrad=false;"  # dac_ctr/elasticdl_train.py:47-48
FALLBACK_HBM_GBS = 6650.0  # B200_PROFILING.md fallback


def ncu_traffic(kernel, world):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of the named kernel from the committed
    `ncu --set full` capture of this workload at N=1 (profiles/ncu_traffic.json); None when the capture
    does not cover the configuration (a number taken under ncu is never measured live by the bench)."""
    if world != 1:
        return None
    try:
        with open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "profiles", "ncu_traffic.json")) as f:
            k = json.load(f)["kernels"][kernel]
        return k["dram_read_bytes"] + k["dram_write_bytes"]
    except (OSError, KeyError, ValueError):
        return None


def measured_peak():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured"
    except Exception:
        return FALLBACK_HBM_GBS, "fallback"


class ClockSampler:
    FIELDS = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.FIELDS,
                 "--format=csv,noheader,nounits", "-lms", "100"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx.append(float(r[1]))
                for n, v in zip(names, r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(n)
            except Exception:
                pass
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


class _CpuWorkload:
    """Inputs of the CPU arm, generated once for the largest thread count and sliced per run."""

    def __init__(self, t_max, batch, dist_kind, seed=1234):
        import numpy as np

        from elasticdl_b200.workloads.deepfm import DEEP_DIM, GROUP_ROWS, synthetic_batch

        self.G, self.batch, self.t_max = len(GROUP_ROWS), batch, t_max
        ids = np.stack([synthetic_batch(batch, seed + t, "cpu", dist_kind)[0].numpy() for t in range(t_max)])  # [T, G, B]
        self.ids = np.ascontiguousarray(ids, dtype=np.int64)
        rng = np.random.RandomState(0)
        # one thread's gradient block, repeated for the others (the values do not affect the timing)
        self.grads = {dim: np.ascontiguousarray(np.broadcast_to(
            (rng.randn(1, self.G, batch, dim) * 1e-3).astype(np.float32), (t_max, self.G, batch, dim)))
            for dim in (1, DEEP_DIM)}

    def run(self, T, steps, warmup):
        import ctypes

        from oracle import ps_oracle as O

        G, batch, n_shards = self.G, self.batch, 1
        vp = ctypes.c_void_p
        ids = self.ids[:T]
        total = 0.0
        for dim, grads_all in self.grads.items():
            grads = grads_all[:T]
            tabs = [[O.OracleTable(dim, "zero") for _ in range(G * n_shards)] for _ in range(3)]
            arrs = [(vp * (G * n_shards))(*[t._h for t in fam]) for fam in tabs]
            rows = (ctypes.c_double * 2)()

            def run(n):
                return O.lib.oracle_bench_ps(T, G, n_shards, arrs[0], arrs[1], arrs[2], O._i64(ids.reshape(-1)),
                                             O._f32(grads.reshape(-1)), batch, dim, 1e-3, 0.9, 0.999, 1e-7, n, rows)

            if warmup:
                run(warmup)
            total += run(steps)
            del tabs
        return T * batch * steps / total


def cpu_reference(batch, steps, warmup, dist_kind, threads=None):
    """Times the oracle's C restatement of the Go PS path (oracle/ps_oracle.c
    oracle_bench_ps): T host threads, each a worker with its own batch, doing unique ->
    pull -> dedup -> scatter -> SparseAdam on in-process hash-map shards (RWMutex per table,
    go/pkg/common/embedding_table.go:22-58) for both table families (dim 1 and dim 8).
    gRPC/protobuf and the TF tower are NOT included, which flatters the reference.  The
    thread count is swept (lock contention on Zipf-hot rows can make fewer threads faster)
    and the best is reported.  Returns (samples_per_sec, threads, description)."""
    import ctypes

    from oracle import ps_oracle as O
    from oracle import ref_kernels

    ref = ref_kernels.lib()  # oracle/_ref: the reference's own kernel_api.cc, compiled unmodified (None if not built)
    O.lib.oracle_set_ref_adam(ctypes.cast(ref.Adam, ctypes.c_void_p) if ref is not None else None)
    ncpu = os.cpu_count() or 1
    cands = [threads] if threads else sorted({min(c, ncpu) for c in (8, 16, 32, 64, ncpu)})
    cands = [c for c in cands if c <= 128] or [min(ncpu, 128)]
    wl = _CpuWorkload(max(cands), batch, dist_kind)
    best = (0.0, cands[0])
    if len(cands) > 1:
        for T in cands:
            sps = wl.run(T, 1, 0 if batch >= 16384 else 1)
            if sps > best[0]:
                best = (sps, T)
    T = best[1]
    sps = wl.run(T, steps, warmup)
    O.lib.oracle_set_ref_adam(None)
    return sps, T, ("C restatement of the Go PS path (unique+pull+dedup+SparseAdam, 76 tables, no gRPC/protobuf, "
                    "no tower), row update by %s: best of thread counts %s = %d threads x batch %d x %d steps, %s ids, "
                    "%d host cores"
                    % ("the reference's own compiled Adam (oracle/_ref = kernel_api.cc built unmodified), one call per row "
                       "as kernel.go:119-138 does" if ref is not None else "the restated Adam (oracle/_ref not built)",
                       cands, T, batch, steps, dist_kind, ncpu))


def parity_check_multi(engine, group, rank, world, dev, lr=1e-3):
    """Post-timing self-check of the path N > 1 times (outside every timed region), on a fresh batch:
    (a) b200ps_xchg_pull == b200ps_pull_rows through the direct peer path, bit for bit, every group;
    (b) one b200ps_xchg_push on rows that are disjoint across ranks (groups with >= 4*world^2 rows;
        rank r draws ids with (id // world) % world == r, which still hit every owner), then the
        rows and both Adam slots read back through the direct path must equal the oracle's Adam
        (kernel_api.cc:40-77 restated, oracle.np_adam) applied to the state read before the push
        -- bit for bit (ids are unique, so no float reassociation is involved).  The ranks issue
        push_begin one after the other so that each knows its optimizer step on every shard.
    The oracle is the checker here, never the thing measured.  Returns the dict printed in the
    JSON line; raises SystemExit(3) on any mismatch (all ranks agree through an all-reduce)."""
    import numpy as np
    import torch
    import torch.distributed as dist

    from elasticdl_b200._lib import check
    from elasticdl_b200.workloads.deepfm import GROUP_ROWS
    from oracle import ps_oracle as O

    G, B, D = engine.G, engine.B, engine.D
    lib, h = group.lib, group._h
    gen = torch.Generator(device=dev).manual_seed(777 + rank)
    big = [g for g in range(G) if GROUP_ROWS[g] >= 4 * world * world]
    ids = torch.empty((G, B), dtype=torch.int64, device=dev)
    for g in range(G):
        R = GROUP_ROWS[g]
        u = torch.rand(B, generator=gen, device=dev, dtype=torch.float64)
        if g in big:
            blocks = R // (world * world)  # id = (q * world + rank) * world + owner
            q = torch.floor(u * blocks).to(torch.int64)
            owner = torch.randint(0, world, (B,), generator=gen, device=dev)
            ids[g] = (q * world + rank) * world + owner
        else:
            ids[g] = torch.floor(u * R).to(torch.int64)
    torch.cuda.synchronize(dev)
    dist.barrier()
    base_steps = [st for _, st, _ in group.snapshot()]
    engine._use(engine.cur)
    engine._unique_into(ids)
    st = group._stream()
    check(lib.b200ps_xchg_pull(h, engine.uniq.data_ptr(), engine.n_unique.data_ptr(), engine.bet_d.data_ptr(),
                               engine.bet_w.data_ptr(), st))
    torch.cuda.synchronize(dev)
    nu = engine.n_unique.cpu().numpy()
    uniq = engine.uniq.view(G, B)
    bet_d, bet_w = engine.bet_d.view(G, B, D), engine.bet_w.view(G, B)
    bad_pull, rows_pull = 0, 0
    pre = {}
    for g in range(G):
        u = int(nu[g])
        idg = uniq[g, :u].contiguous()
        d_direct, w_direct = group.pull_rows([(engine.deep_names[g], idg), (engine.wide_names[g], idg)])
        bad_pull += int((d_direct != bet_d[g, :u]).any().item()) + int((w_direct.view(-1) != bet_w[g, :u]).any().item())
        rows_pull += u
        if g in big:
            pre[g] = (idg, d_direct.cpu().numpy(), w_direct.cpu().numpy(),
                      [group.slot_rows(engine.deep_names[g], idg, k).cpu().numpy() for k in (1, 2)],
                      [group.slot_rows(engine.wide_names[g], idg, k).cpu().numpy() for k in (1, 2)])
    # gradients for the live rows
    engine.gsum_d.normal_(0.0, 1e-2, generator=gen)
    engine.gsum_w.normal_(0.0, 1e-2, generator=gen)
    gs_d, gs_w = engine.gsum_d.view(G, B, D).cpu().numpy(), engine.gsum_w.view(G, B).cpu().numpy()
    torch.cuda.synchronize(dev)
    dist.barrier()
    for r in range(world):  # ordered ApplyGradients: rank r is the (r+1)-th pusher on every shard
        if r == rank:
            group.push_begin(lr, [0] * world)
            torch.cuda.synchronize(dev)
        dist.barrier()
    check(lib.b200ps_xchg_push(h, engine.gsum_d.data_ptr(), engine.gsum_w.data_ptr(), st))
    group.push_end(sync=False)
    torch.cuda.synchronize(dev)
    dist.barrier()
    bad_push, rows_push = 0, 0
    for g in big:
        idg, p_d, p_w, s_d, s_w = pre[g]
        u = idg.numel()
        if u == 0:
            continue
        # every id of group g lives on shard id % world: the step this rank used there
        owners = (idg % world).cpu().numpy()
        got_d = group.pull_rows([(engine.deep_names[g], idg)])[0].cpu().numpy()
        got_w = group.pull_rows([(engine.wide_names[g], idg)])[0].cpu().numpy()
        got_sd = [group.slot_rows(engine.deep_names[g], idg, k).cpu().numpy() for k in (1, 2)]
        got_sw = [group.slot_rows(engine.wide_names[g], idg, k).cpu().numpy() for k in (1, 2)]
        for s_ in range(world):
            m = owners == s_
            if not m.any():
                continue
            step = int(base_steps[s_]) + rank + 1
            for p0, m0, v0, gr, got, gm, gv_ in ((p_d, s_d[0], s_d[1], gs_d[g, :u], got_d, got_sd[0], got_sd[1]),
                                                  (p_w, s_w[0], s_w[1], gs_w[g, :u, None], got_w, got_sw[0], got_sw[1])):
                pp, mm, vv = p0[m].copy(), m0[m].copy(), v0[m].copy()
                O.np_adam(np.ascontiguousarray(gr[m], dtype=np.float32), pp, mm, vv, lr, step, 0.9, 0.999, 1e-7)
                bad_push += int(not (np.array_equal(pp, got[m]) and np.array_equal(mm, gm[m]) and np.array_equal(vv, gv_[m])))
        rows_push += u
    group.check()
    t = torch.tensor([bad_pull, bad_push, rows_pull, rows_push], device=dev, dtype=torch.int64)
    dist.all_reduce(t)
    bad_pull, bad_push, rows_pull, rows_push = (int(x) for x in t.tolist())
    res = {"pull": "bit-exact" if bad_pull == 0 else "MISMATCH (%d groups)" % bad_pull,
           "push": "bit-exact" if bad_push == 0 else "MISMATCH (%d shard-groups)" % bad_push,
           "rows": rows_pull, "rows_push_checked": rows_push, "world": world,
           "what": "xchg_pull vs direct peer pull (all 76 tables); xchg_push (Adam, rank-disjoint rows) vs oracle.np_adam on "
                   "the pre-push state: params and both slots"}
    if bad_pull or bad_push:
        if rank == 0:
            print(json.dumps({"parity_check": res}), file=sys.stderr)
        raise SystemExit(3)
    return res


DUMP_ROWS_PER_GROUP = 4096
DUMP_MAX_BYTES = 64 << 20


def dump_outputs(out_dir, engine, group, ids, seed=0):
    """Writes what the last timed step computed as float32 / float64 .npy files under out_dir, so that two builds
    run with the same arguments (hence the same inputs) can be compared array by array:
      loss [1], logits [B] (fused towers only)   what the step returned / wrote for its batch
      dense_params [n]                           the tower parameters the PS holds after the step, flat order
      row_ids [K, 2] float64                     (id group, id): a fixed seeded sample of up to DUMP_ROWS_PER_GROUP
                                                 of the distinct ids of the step's batch in every group
      deep_rows [K, 8], wide_rows [K]            those rows of the deep / wide tables after the step
    Gradients are summed with atomics, so repeated runs of one build differ in the last bits: compare with a float
    tolerance (two runs at the defaults on a B200 at its 1000 W power limit: rows and dense parameters within 6e-8,
    logits within 6e-7).
    ids: the step's int64 [G, B] id batch (device)."""
    import numpy as np
    import torch

    torch.cuda.synchronize(engine.device)
    out = {"loss": engine.loss_buf.cpu().numpy().astype(np.float32)}
    if engine.tower_kind != "torch":  # the torch tower returns its logits to autograd, not into logits_buf
        out["logits"] = engine.logits_buf.cpu().numpy().astype(np.float32)
    dense = group.pull_dense([n for n, _ in engine.params])
    out["dense_params"] = torch.cat([dense[n].reshape(-1) for n, _ in engine.params]).cpu().numpy()
    picks, requests = [], []
    for g in range(engine.G):
        u = torch.unique(ids[g]).cpu().numpy()
        rng = np.random.RandomState(seed + g)
        sel = u[np.sort(rng.choice(u.size, min(u.size, DUMP_ROWS_PER_GROUP), replace=False))]
        picks.append(np.stack([np.full(sel.size, g), sel], 1).astype(np.float64))
        requests += [(engine.deep_names[g], sel), (engine.wide_names[g], sel)]
    rows = group.pull_rows(requests)
    out["row_ids"] = np.concatenate(picks)
    out["deep_rows"] = torch.cat(rows[0::2]).cpu().numpy()
    out["wide_rows"] = torch.cat(rows[1::2]).reshape(-1).cpu().numpy()
    total = sum(a.nbytes for a in out.values())
    if total > DUMP_MAX_BYTES:
        raise SystemExit("bench.py --dump-outputs: %d bytes exceed the %d-byte budget" % (total, DUMP_MAX_BYTES))
    os.makedirs(out_dir, exist_ok=True)
    for name, a in out.items():
        assert a.dtype in (np.float32, np.float64), (name, a.dtype)
        np.save(os.path.join(out_dir, name + ".npy"), a)


def api_path_leg(dev, batches, steps, warmup):
    """The same DeepFM step through the DROP-IN API instead of the engine: ParameterServerTrainer.train_minibatch
    over 76 elasticdl Embedding layers + PSClient (worker/ps_trainer.py), tower in eager torch.  Timed by wall
    clock around K steps (device idle on both sides); `batched` = the trainer's batched lookups, `per_layer` = one
    unique + pull per layer call as embedding_delegate.py:75-106 does."""
    import time
    import types

    import torch

    from elasticdl_b200.ps import PSGroup
    from elasticdl_b200.worker.ps_client import PSClient
    from elasticdl_b200.worker.ps_trainer import ParameterServerTrainer
    from elasticdl_b200.workloads.deepfm import DeepFMLayersModel

    out = {}
    for mode, batched, graphed, k in (("graphed", True, True, 4 * steps), ("batched", True, False, steps),
                                      ("per_layer", False, False, max(2, steps // 3))):
        group = PSGroup(1, "Adam", ADAM_ARGS, device=dev.index)
        client = PSClient(group)
        client.dense_output = "torch"
        model = DeepFMLayersModel().to(dev)
        trainer = ParameterServerTrainer(model, client, args=types.SimpleNamespace(
            get_model_steps=1, batched_embedding_lookups=batched, cuda_graph=graphed, cuda_graph_warmup=warmup))
        feats = [(DeepFMLayersModel.features_of(ids, dense), labels) for ids, dense, labels in batches]
        for i in range(warmup + (2 if graphed else 0)):  # graphed: `warmup` eager minibatches, the capture, one replay
            trainer.train_minibatch(*feats[i % len(feats)])
        torch.cuda.synchronize(dev)
        l0 = group.launch_count
        t0 = time.perf_counter()
        for i in range(k):
            accepted, version, loss = trainer.train_minibatch(*feats[(warmup + i) % len(feats)])
        torch.cuda.synchronize(dev)
        dt = (time.perf_counter() - t0) / k
        B = batches[0][0].shape[1]
        out[mode] = {"ms_per_step": dt * 1e3, "samples_per_s": B / dt, "ps_launches_per_step": (group.launch_count - l0) / k,
                     "steps": k, "final_loss": float(loss), "version": int(version)}
        if graphed:
            out[mode]["cuda_graph"] = isinstance(trainer._graph_state, dict)
            out[mode]["graph_fallback_reason"] = trainer.graph_fallback_reason
            out[mode]["per_step"] = "input copy (1 kernel per dtype) + ONE graph replay + error word / versions read on the host"
        group.close()
        del trainer, model, client, group
    out["what"] = ("ParameterServerTrainer.train_minibatch (pull_dense + 76 Embedding layers + torch tower + push_gradients), "
                   "1 shard, wall clock: `graphed` = args.cuda_graph (the whole minibatch replayed as one CUDA graph), "
                   "`batched` = eager with batched lookups, `per_layer` = one lookup per layer call as the reference does; "
                   "the engine path (`value`) additionally fuses the tower into one hand-written kernel")
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--batch", type=int, default=32768, help="samples per GPU per step")
    ap.add_argument("--dist", default="zipf", choices=["zipf", "uniform"])
    ap.add_argument("--pool", type=int, default=8, help="distinct pre-generated batches cycled through")
    ap.add_argument("--cpu-batch", type=int, default=0, help="per-thread batch of the CPU arm (0 = --batch: same config)")
    ap.add_argument("--cpu-steps", type=int, default=2)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--tower", default="tile", choices=["tile", "fused", "mma", "torch"])
    ap.add_argument("--no-graph", action="store_true", help="time eager launches instead of the captured CUDA graph")
    ap.add_argument("--profile-step", action="store_true",
                    help="run ONE eager step between cudaProfilerStart/Stop after the warm-up and exit "
                         "(for `ncu --profile-from-start off`; prints no bench line)")
    ap.add_argument("--lookahead", default="on", choices=["on", "off"],
                    help="deduplicate the ids of batch i+1 on a second stream while batch i trains (graph mode)")
    ap.add_argument("--paired", default="off", choices=["on", "off"],
                    help="store each group's deep+wide rows as one record per id")
    ap.add_argument("--exchange", default="auto", choices=["auto", "owner", "direct"],
                    help="multi-GPU row exchange: owner-computes bulk exchange (default for N>1) or direct peer access")
    ap.add_argument("--api-steps", type=int, default=6,
                    help="steps of the drop-in API path (ParameterServerTrainer) timed after the engine at N=1; 0 = skip")
    ap.add_argument("--no-parity-check", action="store_true", help="skip the post-timing N>1 parity self-check")
    ap.add_argument("--ids", default="narrow", choices=["narrow", "int32"],
                    help="id transport of the packed batches: 1/2/4 bytes per id by table size, or int32")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last timed step computed (loss, logits, dense "
                         "parameters, a fixed seeded sample of the embedding rows it trained) as DIR/<name>.npy")
    args = ap.parse_args()
    cpu_batch = args.cpu_batch or args.batch

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    config = {"workload": "DeepFM dac_ctr synthetic Criteo: 38 id groups x (wide dim1 + deep dim8) = 76 PS tables, "
                          "5549416 rows/family, Adam 1e-3, DNN[16,4]+FM tower",
              "batch_per_gpu": args.batch, "global_batch": args.batch * max(world, 1), "id_distribution": args.dist,
              "ps_shards": max(world, 1), "sharding": "id % N over GPUs (NVLink P2P)" if world > 1 else "1 shard",
              "step": "pull_dense+unique+pull(76 tables)+tower fwd/bwd+dedup-sum+push(dense+76 tables, Adam)+version++"}

    if args.impl == "reference":
        if rank != 0:
            return
        sps, T, desc = cpu_reference(cpu_batch, max(args.steps, 1), min(args.warmup, 2), args.dist)
        config["cpu_batch_per_thread"] = cpu_batch
        config["same_batch"] = cpu_batch == args.batch
        line = {"impl": "reference", "metric": "deepfm_train_samples_per_sec", "value": sps, "unit": "samples/s",
                "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": 1e3 * cpu_batch * T / sps, "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": config,
                "cpu_baseline": {"value": sps, "unit": "samples/s", "cores": T, "kind": "port", "sample": desc},
                "e2e": {"value": sps, "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                "gpu_launches": 0}
        print(json.dumps(line))
        return

    import torch
    import torch.distributed as dist

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- the product path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        if os.environ.get("NCCL_DEBUG", "").upper() in ("", "VERSION"):
            os.environ["NCCL_DEBUG"] = "WARN"  # keep NCCL's version banner off stdout: one JSON line only
        dist.init_process_group("nccl", device_id=dev)

    from elasticdl_b200 import _lib
    from elasticdl_b200.ps import PSGroup
    from elasticdl_b200.workloads.deepfm import DeepFMPSEngine, N_DENSE, pack_batch, synthetic_batch

    group = PSGroup(world, "Adam", ADAM_ARGS, device=local_rank,
                    local_shards=[rank] if world > 1 else None)
    engine = DeepFMPSEngine(group, args.batch, tower=args.tower, paired=args.paired == "on",
                            exchange=None if args.exchange == "auto" else args.exchange, id_transport=args.ids)
    config["record_layout"] = "paired deep+wide record per id" if engine.paired else "one record slab per table"
    config["exchange"] = engine.exchange
    use_graph = args.tower != "torch" and not args.no_graph
    lookahead = use_graph and args.lookahead == "on"
    config["pipeline"] = ("CUDA graph per step; id dedup of batch i+1 overlapped with step i on a second stream"
                          if lookahead else ("CUDA graph per step" if use_graph else "eager launches"))
    config["id_transport"] = (("ids cross PCIe / sit in HBM at 1 / 2 / 4 bytes by table size (<= 256 / <= 65536 / larger rows)"
                               if args.ids == "narrow" else "ids cross PCIe / sit in HBM as int32 (all tables < 2^31 rows)")
                              + ", widened to int64 inside the dedup kernel; one packed buffer per batch [ids|dense|labels]")
    if world > 1:
        dist.barrier()
    B = args.batch
    G = engine.G

    # pre-generated batches: packed pinned host copies (e2e) and packed device copies (kernel-resident timing)
    host, devb, devp = [], [], []
    for p in range(args.pool):
        ids, dense, labels = synthetic_batch(B, 1234 + p + 1000 * rank, dev, args.dist)
        devb.append((ids, dense, labels))
        devp.append(pack_batch(ids, dense, labels, widths=engine.widths))
        host.append(pack_batch(ids.cpu(), dense.cpu(), labels.cpu(), pin=True, widths=engine.widths))
    uniq_per_batch = []
    for ids, _, _ in devb:
        _, _, n = group.unique(ids.view(-1), G)
        uniq_per_batch.append(int(n.sum().item()))
    h2d = host[0].numel()
    u_mean = statistics.mean(uniq_per_batch)
    rows_mb = u_mean * (96 + 16) / 1e6  # Adam records touched per step: 96 B (dim 8) + 16 B (dim 1) per unique id
    config["l2_policy"] = ("pool of %d distinct batches cycled: a batch's rows (%.0f MB of records per step, plus "
                           "~%.0f MB of id / dedup / row buffers) recur after %d other steps, i.e. after > %.0f MB of "
                           "other traffic vs the 126 MB L2; Zipf-hot rows recur every step by construction of the workload"
                           % (args.pool, rows_mb, 12 * G * B * 4 / 1e6, args.pool - 1, (args.pool - 1) * rows_mb))

    def sync_all():
        torch.cuda.synchronize(dev)
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize(dev)

    def max_over_ranks(ms):
        if world > 1:
            t = torch.tensor([ms], device=dev, dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            return float(t.item())
        return ms

    def my_launches():
        return group.launch_count + _lib.lib().b200ps_launch_count(None) + _lib.lib().b200_deepfm_launch_count() + _lib.lib().b200_deepfm_mma_launch_count() + _lib.lib().b200_deepfm_tile_launch_count() + _lib.lib().b200feat_launch_count()

    # ---- eager pass: every kernel launched from the host, CUDA-event pairs around the PS kernels ----
    for i in range(args.warmup):
        engine.step(*devb[i % args.pool])
    sync_all()
    if args.profile_step:
        torch.cuda.cudart().cudaProfilerStart()
        engine.step(*devb[args.warmup % args.pool])
        torch.cuda.synchronize(dev)
        torch.cuda.cudart().cudaProfilerStop()
        group.check()
        return
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    launches0 = my_launches()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(args.steps):
        engine.step(*devb[i % args.pool])
    e1.record()
    sync_all()
    ms_eager = max_over_ranks(e0.elapsed_time(e1))
    launches = my_launches() - launches0
    group.check()
    # per-kernel device times: the same eager steps with CUDA-event pairs around the named kernels.  The host
    # needs ~10 us per launch, more than some of these kernels run, so each step is queued behind a spin
    # kernel (torch.cuda._sleep) that keeps the GPU busy while the host enqueues the whole step: the kernels
    # then execute back to back and an event pair brackets device time, not host time.
    ev = {}
    for i in range(args.steps):
        torch.cuda._sleep(4_000_000)
        engine.step(*devb[i % args.pool], ev=ev)
    sync_all()
    group.check()
    ms = ms_eager
    if use_graph:
        # ---- headline: the same step replayed from a CUDA graph (inputs resident in HBM) ----
        if lookahead:
            # batch i trains while the ids of batch i+1 are deduplicated on a second stream
            engine.capture_ahead()
            engine.prepare_packed(devp[0])

            def graph_step(i):
                return engine.step_ahead_graph(devp[(i + 1) % args.pool])
        else:
            engine.capture()

            def graph_step(i):
                return engine.step_graph(devp[i % args.pool])
        for i in range(args.warmup):
            graph_step(i)
        sync_all()
        e0.record()
        for i in range(args.warmup, args.warmup + args.steps):
            graph_step(i)
        e1.record()
        sync_all()
        ms = max_over_ranks(e0.elapsed_time(e1))
        group.check()
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        # step i of a timed loop trains batch i % pool: the graph loop ran steps warmup .. warmup+steps-1, the
        # eager path's last loop steps 0 .. steps-1
        last = (args.warmup + args.steps - 1 if use_graph else args.steps - 1) % args.pool
        dump_outputs(args.dump_outputs, engine, group, devb[last][0])

    # ---- per-kernel durations from the CUDA events recorded inside the timed region ----
    kern = engine.kernel_report(ev, [uniq_per_batch[i % args.pool] for i in range(args.steps)])

    # ---- end to end: host buffers in, loss out, every step ----------------------------
    sync_all()
    e2, e3 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ahead = 2 if lookahead else 1  # batches in flight ahead of the running step
    feeder = engine.host_feeder(ahead + 1, lookahead=lookahead) if use_graph else None
    # the link itself: one packed batch per copy, back to back on the copy stream
    probe = torch.empty_like(devp[0])
    cs = feeder.copy_stream if feeder is not None else torch.cuda.Stream(device=dev)
    p0, p1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with torch.cuda.stream(cs):
        probe.copy_(host[0], non_blocking=True)
        p0.record(cs)
        for j in range(8):
            probe.copy_(host[j % args.pool], non_blocking=True)
        p1.record(cs)
    sync_all()
    h2d_ms = p0.elapsed_time(p1) / 8
    with torch.cuda.stream(cs):  # second round: the first DMA from a freshly pinned buffer is slower
        p0.record(cs)
        for j in range(8):
            probe.copy_(host[j % args.pool], non_blocking=True)
        p1.record(cs)
    sync_all()
    h2d_ms = min(h2d_ms, p0.elapsed_time(p1) / 8)
    # W warm-up steps run through the feeder (untimed, like the device-resident arm's warm-up) and leave its
    # prefetch window full; then EXACTLY K steps are timed between two barrier + synchronize points: every timed
    # step enqueues the H2D copy of one batch from pinned host memory (the batch `ahead` steps in front of it,
    # like the reference's dataset.prefetch), runs one dedup + one train pass, and copies its loss D2H.
    n_e2e = args.warmup + args.steps
    if feeder is not None:
        for j in range(ahead):
            feeder.submit(host[j % args.pool])
    for i in range(n_e2e):
        if i == args.warmup:
            sync_all()  # barrier + synchronize: the prefetched batches have landed, nothing is in flight
            e2.record()
        if feeder is not None:
            feeder.submit(host[(i + ahead) % args.pool])
            feeder.run_next()
        else:
            hb = host[i % args.pool].to(dev, non_blocking=True)
            from elasticdl_b200.workloads.deepfm import packed_views
            engine.step(*packed_views(hb, G, B, engine.widths))
        # the D2H read of the step's loss: the last kernel of every step stores it into a ring in pinned host
        # memory (engine.loss_ring, 4 bytes over PCIe per step; b200_deepfm_publish_loss) -- a cudaMemcpyAsync of the
        # scalar between two graph launches put a copy-engine round trip on the critical path of every step
        # (tools/e2e_probe.py: 198 us per step without it, 222-237 us with it)
    e3.record()
    sync_all()
    ms_e2e = max_over_ranks(e2.elapsed_time(e3))
    group.check()

    parity = None
    if world > 1 and not args.no_parity_check and engine.exchange == "owner":
        parity = parity_check_multi(engine, group, rank, world, dev)

    if rank != 0:
        if world > 1:
            dist.barrier()
        return

    samples = args.steps * B * world
    value = samples / (ms * 1e-3)
    e2e_value = samples / (ms_e2e * 1e-3)
    peak, peak_kind = measured_peak()
    line = {"metric": "deepfm_train_samples_per_sec", "value": value, "unit": "samples/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": config,
            "clocks": clocks,
            "e2e": {"value": e2e_value, "unit": "samples/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": 4,
                    "d2h": "the step's loss, stored by the step's last kernel into a ring in pinned host memory",
                    "ms_per_step": ms_e2e / args.steps, "h2d_copy_ms_probe": h2d_ms,
                    "h2d_gbs_probe": h2d / h2d_ms / 1e6,
                    "id_narrowing": "ids int64 -> %s on the host side of the boundary (packed batch), widened on the device" % ("1/2/4-byte" if args.ids == "narrow" else "int32")},
            "gpu_launches": int(launches), "gpu_launches_per_step": launches / max(args.steps, 1),
            "launch_mode": "cuda_graph" if use_graph else "eager", "eager_ms_per_step": ms_eager / args.steps,
            "tower": args.tower,
            "final_loss": engine.loss_host(engine.steps - 1),
            "e2e_losses_read_on_host": [engine.loss_host(engine.steps - 1 - j) for j in range(min(3, args.steps))]}
    if parity is not None:
        line["parity_check"] = parity
    if kern:
        # the DOMINANT kernel of the step by CUDA-event time, whatever its name
        top = max((k for k in kern if "gbs" in kern[k]), key=lambda k: kern[k]["ms"])
        line["kernels"] = kern
        k = kern[top]
        step_bytes = sum(v["bytes"] for v in kern.values() if "bytes" in v)
        step_ms = ms / args.steps
        line["roofline"] = {"kernel": top, "bound": "hbm", "achieved": k["gbs"], "peak": peak, "unit": "GB/s",
                            "frac": k["gbs"] / peak,
                            "traffic": ncu_traffic(top, world) if (args.batch == 32768 and args.dist == "zipf") else None,
                            "peak_kind": peak_kind, "algorithmic_bytes_per_launch": k["bytes"], "us_per_launch": k["ms"] * 1e3,
                            "step_algorithmic_bytes": step_bytes, "step_gbs": step_bytes / step_ms / 1e6,
                            "step_frac": step_bytes / step_ms / 1e6 / peak,
                            "per_kernel_frac": {n: v["gbs"] / peak for n, v in kern.items() if "gbs" in v},
                            "note": "achieved = algorithmic bytes (SURVEY 8d) / CUDA-event time of the launch (eager pass, GPU kept "
                                    "busy so that the event pairs bracket device time); "
                                    "step_frac = sum of the step's algorithmic bytes / graph ms_per_step / peak"}
        # NOT measured in this run (labelled as such): where the row kernels sit once the launch is big enough to be
        # bandwidth-bound, and the roof a bare random-row gather / read-modify-write reaches on the same memory system
        line["roofline"]["row_kernels_at_scale"] = {
            "not_measured_in_this_run": True,
            "source": "profiles/r2_13_kernel_roofline_sweep_rows_final.jsonl (bench_kernels.py, graph-timed, 4 M unique "
                      "random rows, table >> L2) and profiles/r2_01_gather_roof.jsonl (tools/probes/gather_roof.cu)",
            "frac_of_copy_peak": {"pull_dim8": 0.376, "push_adam_dim8": 0.385, "pull_dim64": 0.675, "push_adam_dim64": 0.533,
                                  "pull_dim1": 0.131, "push_adam_dim1": 0.154},
            "bare_probe_frac_of_copy_peak": {"gather_dim8": 0.374, "rmw_adam_dim8": 0.465, "gather_dim64": 0.954,
                                             "gather_dim1": 0.108},
        }
        pk = "pull" if "pull" in kern else ("pull_deep" if "pull_deep" in kern else None)
        if pk:
            line["pull_gbs"] = kern[pk]["gbs"]
            line["pull_frac_of_peak"] = kern[pk]["gbs"] / peak
    line["unique_ids_per_step"] = u_mean
    if world == 1 and args.api_steps > 0 and not args.profile_step:
        try:  # a side leg: it must never cost the run its headline line
            line["api_path"] = api_path_leg(dev, devb, args.api_steps, 3)
            line["api_path"]["engine_over_batched_api"] = line["api_path"]["batched"]["ms_per_step"] / (ms / args.steps)
            line["api_path"]["engine_over_graphed_api"] = line["api_path"]["graphed"]["ms_per_step"] / (ms / args.steps)
        except Exception as err:
            line["api_path"] = {"error": "%s: %s" % (type(err).__name__, str(err)[:300])}
    if not args.no_cpu_baseline and world == 1:
        sps, T, desc = cpu_reference(cpu_batch, args.cpu_steps, 1, args.dist)
        line["cpu_baseline"] = {"value": sps, "unit": "samples/s", "cores": T, "kind": "port", "sample": desc,
                                "batch_per_thread": cpu_batch, "same_batch": cpu_batch == args.batch}
    print(json.dumps(line))
    if world > 1:
        dist.barrier()


if __name__ == "__main__":
    main()
