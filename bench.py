#!/usr/bin/env python
"""bench.py — broadcast fan-out throughput of the B200-native engine (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W            # our arm
    python bench.py --impl reference --gpus N --steps K ...  # CPU restatement of the reference path
    torchrun --nproc-per-node N bench.py --gpus N ...         # one rank per GPU (N>1)
    python bench.py ... --dump-outputs DIR                    # + the last timed step's outputs as DIR/*.npy

Workload (config.workload "C2", BASELINE.json configs[1]): 2^20 subscribers per GPU all subscribed to
one topic, batches of 8 broadcast messages with 1 KiB payloads (L=1080 B capnp frame, F=1084 B framed
delivery).  One *step* = one batch = 8 x 2^20 deliveries = 9.09 GB written into the per-connection
rings.  `value` is egress GB/s of the whole job with the batch already resident in HBM (submit_device
path).  For N>1 every rank opens the SAME sharded engine through the C ABI (pcdn_config.world_shards =
N, first_shard = rank, one shared ncclUniqueId): the LIBRARY replicates each batch from rank 0's GPU
with one ncclBroadcast per step on its ingest stream, inside the timed region, and every GPU fans
out to its own connection shard — weak scaling; nothing of that lives in this file any more.  `e2e` is the same
metric through pcdn_submit with HOST buffers (pinned staging + H2D inside) plus pcdn_poll (D2H of the
counters and the span table).  Outputs are far larger than L2 (9 GB per step), inputs are 8.7 KB.
"""
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
sys.dont_write_bytecode = True   # the benchmark may run from a read-only tree and writes nothing into it

METRIC = "broadcast fan-out egress GB/s (1 KiB x 2^20 subscribers per GPU, 1 topic); msgs/s and % of HBM peak alongside"
N_CONNS = 1 << 20
PAYLOAD = 1024
MSGS_PER_STEP = 8
KEY_LEN = 32
RING_RECORDS = 16


def broadcast_frame(topic: int, payload: bytes) -> bytes:
    """Single-segment cdn-proto Broadcast{topics:[topic], message:payload} (SURVEY Appendix B).
    Synthetic input generation only — routing never looks inside (R1)."""
    k = len(payload)
    words = 5 + 1 + (k + 7) // 8
    out = bytearray()
    out += (0).to_bytes(4, "little") + words.to_bytes(4, "little")
    out += bytes.fromhex("0000000001000100")            # root → Message (1 data, 1 ptr)
    out += (4).to_bytes(8, "little")                     # union tag: broadcast
    out += bytes.fromhex("0000000000000200")            # → Broadcast (0 data, 2 ptrs)
    out += (5).to_bytes(4, "little") + (2 | (1 << 3)).to_bytes(4, "little")   # topics: byte list, 1 elem
    out += (5).to_bytes(4, "little") + (2 | (k << 3)).to_bytes(4, "little")   # message: byte list, k elems
    out += bytes([topic]) + bytes(7)
    out += payload + bytes((-k) % 8)
    return bytes(out)


DUMP_SPANS = 1024           # --dump-outputs: spans sampled from the batch's span table
DUMP_RECORD_BYTES = 12 << 20  # ... and at most this many framed bytes of theirs (48 MB as float32)


def dump_outputs(eng, b, out_dir):
    """--dump-outputs: what a caller of the timed path receives for batch `b` (polled here, released by
    the caller afterwards), as .npy files that two builds can be compared by:
      batch.npy    float64 [n_msgs, n_spans, n_deliveries, bytes_out, n_overflow, n_direct_dropped, status]
      spans.npy    float64 (K, 4): conn, ring_off, len, n_records of a fixed seeded sample of the span
                   table (sorted by connection, then offset)
      records.npy  float32: the framed records (4-byte BE length + frame) of those spans, in that order;
                   the pad bytes up to the 32-byte record stride are unspecified and left out"""
    import numpy as np

    res = eng.poll(b)
    if res.runs:   # run-length table {conn0, n_conns, ring_off, len, n_records, off_stride}, expanded without a Python loop
        r = np.ctypeslib.as_array(C.cast(res.runs, C.POINTER(C.c_uint32)), shape=(res.n_runs, 6)).astype(np.int64)
        n = r[:, 1]
        k = np.arange(int(n.sum())) - np.repeat(np.cumsum(n) - n, n)
        t = np.stack([np.repeat(r[:, 0], n) + k, np.repeat(r[:, 2], n) + k * np.repeat(r[:, 5], n),
                      np.repeat(r[:, 3], n), np.repeat(r[:, 4], n)], axis=1)
    elif res.n_spans:
        t = np.ctypeslib.as_array(C.cast(res.spans, C.POINTER(C.c_uint32)), shape=(res.n_spans, 4)).astype(np.int64)
    else:
        t = np.zeros((0, 4), dtype=np.int64)
    t = t[np.lexsort((t[:, 1], t[:, 0]))]
    pick = np.sort(np.random.default_rng(0).choice(len(t), size=min(len(t), DUMP_SPANS), replace=False))
    spans, records, total = [], [], 0
    for conn, off, ln, nrec in t[pick].tolist():
        data = eng.read(conn, res.pool_base + off, ln)   # output pool: absolute 32-byte unit offset
        p, framed = 0, []
        for _ in range(nrec):
            n_rec = 4 + int.from_bytes(data[p:p + 4], "big")
            framed.append(data[p:p + n_rec])
            p += (n_rec + 31) // 32 * 32
        framed = b"".join(framed)
        if total + len(framed) > DUMP_RECORD_BYTES:
            break
        spans.append((conn, off, ln, nrec))
        records.append(framed)
        total += len(framed)
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "batch.npy"), np.array(
        [res.n_msgs, res.n_spans, res.n_deliveries, res.bytes_out, res.n_overflow, res.n_direct_dropped, res.status], dtype=np.float64))
    np.save(os.path.join(out_dir, "spans.npy"), np.array(spans, dtype=np.float64).reshape(-1, 4))
    np.save(os.path.join(out_dir, "records.npy"), np.frombuffer(b"".join(records), dtype=np.uint8).astype(np.float32))


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, dev):
        self.dev, self.proc, self.lines = dev, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-i", str(self.dev), "-lms", "100"], stdout=subprocess.PIPE, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for ln in self.proc.stdout:
            self.lines.append(ln.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx = float(f[2])
            except ValueError:
                continue
            for nm, v in zip(names, f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx, "samples": len(sm), "reasons": sorted(reasons)}


def run_cpu_reference(n_conns, payload, msgs, steps, warmup, threads=0, timeout=900, model=1):
    """oracle/cpu_broker_timed: the C++ restatement of the reference's CPU path (the reference is
    Rust and cannot be built here).  This is the ONLY place bench.py executes anything in oracle/."""
    from oracle import oracle as orc

    orc.build()
    out = subprocess.run([orc.TIMED_PATH, str(n_conns), str(payload), str(msgs), str(steps), str(warmup), str(threads), str(model)],
                         capture_output=True, text=True, timeout=timeout, check=True)
    return json.loads(out.stdout.strip().splitlines()[-1])


def pick_cpu_model(n_conns, payload, msgs, cores):
    """The port has two threading models (writer tasks after / concurrent with the receive loops); one
    step of each decides which is faster ON THIS BOX — the baseline is always the faster one."""
    cal = {}
    for model in (0, 1):
        try:
            cal[model] = run_cpu_reference(n_conns, payload, msgs, 1, 0, cores, model=model)["gbps"]
        except Exception:
            cal[model] = 0.0
    best = max(cal, key=lambda k: cal[k])
    return best, {"two_phases_GBps": cal[0], "overlapped_GBps": cal[1]}


def reference_arm(args, rank, world):
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    # default shape = config C2; `--conns 128 --msgs 1` is BASELINE config C1 (the reference's own
    # CPU-runnable broadcast bench scaled to 128 subscribers x 1 KiB), `--conns 2 --payload 10000` its
    # literal shape (cdn-broker/benches/broadcast.rs:58-62)
    n_conns, payload = args.conns, args.payload
    cores = min(cores, max(1, n_conns // 1024))  # the port starts its worker threads per step: tiny shapes run serially
    msgs = args.msgs            # the SAME batch as the GPU arm (same_config): a long run is cut in steps, never in the batch
    model, calib = pick_cpu_model(n_conns, payload, msgs, cores)
    per_step = n_conns * msgs * (4 + 8 * (7 + (payload + 7) // 8)) / 1e9 / max(max(calib.values()), 1e-3)
    budget = 200.0
    steps, warmup = args.steps, args.warmup
    while steps > 1 and per_step * (steps + warmup) > budget:
        steps = max(1, steps // 2)
        warmup = min(warmup, 1)
    r = run_cpu_reference(n_conns, payload, msgs, steps, warmup, cores, model=model)
    gbps = r["gbps"]
    line = {
        "impl": "reference", "metric": METRIC, "value": gbps, "unit": "GB/s", "n_gpus": args.gpus, "steps": steps,
        "warmup": warmup, "steps_requested": args.steps, "ms_per_step": 1e3 * r["seconds"] / max(1, steps), "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
        "deliveries_per_s": r["deliveries_per_s"],
        "config": {"workload": "C2: 2^20 subscribers, 1 topic, 1 KiB broadcast" if (n_conns, payload) == (N_CONNS, PAYLOAD) else
                   "%d subscribers, 1 topic, %d B broadcast" % (n_conns, payload), "n_conns": n_conns, "payload": payload,
                   "msgs_per_step": msgs, "frame_bytes": r["frame_bytes"],
                   "note": "C++ restatement of cdn-broker's CPU path (reference is Rust, not buildable here): %s (the faster of the "
                           "port's two threading models on this box); same batch as the GPU arm, %d of the %d requested steps timed" % (r.get("model"), steps, args.steps)},
        "cpu_baseline": {"value": gbps, "unit": "GB/s", "cores": r["threads"], "kind": "port",
                         "sample": "%d msgs x %d subscribers per step, %d steps" % (msgs, n_conns, steps),
                         "model": r.get("model"), "model_calibration": calib, "model_calibration": calib,
                         "median_step_value": r.get("gbps_median_step"), "router_threads": r.get("router_threads"),
                         "writer_threads": r.get("writer_threads"), "stage12_s": r["stage12_s"], "stage3_s": r["stage3_s"]},
        "e2e": {"value": gbps, "unit": "GB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--variant", type=int, default=int(os.environ.get("PCDN_PACK_VARIANT", "0")))
    ap.add_argument("--conns", type=int, default=N_CONNS)
    ap.add_argument("--payload", type=int, default=PAYLOAD)
    ap.add_argument("--msgs", type=int, default=MSGS_PER_STEP)
    ap.add_argument("--ring-records", type=int, default=RING_RECORDS)
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-verify", action="store_true")
    ap.add_argument("--pool", action="store_true", help="one shared output pool (PCDN_FLAG_OUTPUT_POOL, same bytes as the rings) instead of a ring per connection")
    ap.add_argument("--plain-spans", action="store_true", help="one 16-byte span per connection instead of the run-length span table (PCDN_FLAG_SPAN_RUNS)")
    ap.add_argument("--no-secondary", action="store_true", help="skip the secondary configs (C4 direct, C5 sparse, C3 mixed; N=1 only)")
    ap.add_argument("--sustain", type=float, default=2.0, help="seconds of the sustained window reported beside the K-step number (0 = skip)")
    ap.add_argument("--no-e2e-host", action="store_true", help="skip the e2e_host leg (egress drain of every byte to host memory)")
    ap.add_argument("--ingest", choices=["nccl", "host"], default="nccl",
                    help="N>1: how the library brings a batch to every GPU (pcdn_config.ingest). nccl = H2D on shard 0 + one "
                         "ncclBroadcast over NVLink per batch, issued by the library on its ingest stream; host = every shard "
                         "copies the batch from its process's pinned staging (host-buffer path only)")
    ap.add_argument("--host-rings", action="store_true",
                    help="egress hand-off mode: rings in mapped pinned host memory (PCDN_FLAG_HOST_RINGS); PCIe-bound, use with --conns <= 65536")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step computed (batch counters, a seeded sample of its span table and "
                         "framed records) as DIR/*.npy; with N>1, rank 0's shard")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        reference_arm(args, rank, world)
        return

    import numpy as np
    import torch
    import torch.distributed as dist

    import __graft_entry__ as ge

    pkg = ge.load_package()
    # build only when the library is missing (file times are meaningless on a copied snapshot, and a
    # rebuild by rank 0 would race with the other ranks' dlopen)
    if rank == 0 and not os.path.exists(pkg.LIB_PATH):
        pkg.build(force=True)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.barrier()
    stream = torch.cuda.Stream(device=dev)
    n_conns, M = args.conns, args.msgs
    frames = [broadcast_frame(0, bytes(((i * 131 + m * 7 + 1) & 0xFF) for i in range(args.payload))) for m in range(M)]
    L = len(frames[0]); F = 4 + L
    rec = (F + 31) // 32 * 32
    ring_bytes = args.ring_records * rec
    shard_kw = {}
    if world > 1:
        # one logical broker over `world` connection shards; this process drives shard `rank` on GPU `local`
        uid = [pkg.nccl_unique_id() if rank == 0 else None]
        dist.broadcast_object_list(uid, src=0)
        shard_kw = dict(devices=[local], world_shards=world, first_shard=rank, nccl_unique_id=uid[0],
                        ingest=pkg.INGEST_HOST if args.ingest == "host" else pkg.INGEST_NCCL)
    eng = pkg.Engine(device=local, stream=stream.cuda_stream, max_conns=n_conns, max_topics=256, max_keys=world * n_conns,
                     max_key_len=KEY_LEN, ring_bytes_per_conn=ring_bytes, max_batch_msgs=max(64, M), max_batch_bcast=max(16, M),
                     max_batch_bytes=max(1 << 20, 4 * M * (rec + 64)), max_batch_deliveries=M * n_conns + 1024, batch_slots=4,
                     pack_variant=args.variant,
                     flags=(pkg.FLAG_HOST_RINGS if args.host_rings else 0) | (0 if args.plain_spans else pkg.FLAG_SPAN_RUNS) |
                           (pkg.FLAG_OUTPUT_POOL if args.pool else 0), **shard_kw)
    # world x 2^20 subscribers, all on topic 0.  Every rank replays the same control plane (the SPMD
    # contract of a multi-process group): connections go to the least-loaded shard, i.e. round robin,
    # so each GPU ends up owning exactly n_conns of them.
    n_total = world * n_conns
    rng = np.random.default_rng(2)
    keys = rng.integers(0, 256, size=(n_total, KEY_LEN), dtype=np.uint8)
    keys[:, :8] = np.arange(n_total, dtype=np.uint64).view(np.uint8).reshape(n_total, 8)
    topics = np.zeros(n_total, dtype=np.uint16)
    offs = np.arange(n_total + 1, dtype=np.uint32)
    t0 = time.time()
    conn_ids = eng.add_users_bulk(keys, KEY_LEN, topics, offs)
    setup_s = time.time() - t0
    sd = eng.shard_info(0)
    assert sd.n_conns == n_conns and sd.global_index == rank, (sd.n_conns, sd.global_index)
    assert world == 1 or sd.nccl_ranks == world or args.ingest == "host", "ingest communicator does not span all ranks"
    del keys, topics, offs, conn_ids

    # ---- device-resident batch (slot = 16-byte aligned, raw at +4) --------------------------------
    slot = (4 + L + 15) // 16 * 16
    host_arena = np.zeros(M * slot + 64, dtype=np.uint8)
    for m, fr in enumerate(frames):
        host_arena[m * slot + 4: m * slot + 4 + L] = np.frombuffer(fr, dtype=np.uint8)
    pinned = torch.from_numpy(host_arena).pin_memory()
    with torch.cuda.stream(stream):
        d_arena = torch.zeros(M * slot + 64, dtype=torch.uint8, device=dev)
        if rank == 0:
            d_arena.copy_(pinned, non_blocking=True)
        d_kind = torch.full((M,), 4, dtype=torch.uint8, device=dev)
        d_flags = torch.zeros(M, dtype=torch.uint8, device=dev)
        d_slot = (torch.arange(M, dtype=torch.int64, device=dev) * (slot // 16)).to(torch.int32)
        d_len = torch.full((M,), L, dtype=torch.int32, device=dev)
        d_aoff = torch.arange(M, dtype=torch.int32, device=dev)
        d_alen = torch.ones(M, dtype=torch.int32, device=dev)
        d_topics = torch.zeros(M, dtype=torch.int16, device=dev)
        d_bidx = torch.arange(M, dtype=torch.int32, device=dev)
    db = pkg.DeviceBatch(M, M, d_arena.data_ptr(), d_arena.numel(), d_kind.data_ptr(), d_flags.data_ptr(), d_slot.data_ptr(),
                         d_len.data_ptr(), d_aoff.data_ptr(), d_alen.data_ptr(), d_topics.data_ptr(), M, d_bidx.data_ptr())

    # Batches are pipelined the way a broker streams them: batch n is released (its ring space
    # handed back by the consumer) right after batch n+1 has been submitted, so the engine can run
    # the match/plan/offsets kernels of n+1 while the pack of n is still streaming to HBM.  With
    # N>1 the ingest buffer is double-buffered so the NCCL broadcast of step n+1 never touches the
    # frames the pack of step n is reading.
    torch.cuda.synchronize(dev)
    with torch.cuda.stream(stream):
        d_arenas = [d_arena, d_arena.clone()]
    dbs = [db, pkg.DeviceBatch(M, M, d_arenas[1].data_ptr(), d_arenas[1].numel(), d_kind.data_ptr(), d_flags.data_ptr(),
                               d_slot.data_ptr(), d_len.data_ptr(), d_aoff.data_ptr(), d_alen.data_ptr(),
                               d_topics.data_ptr(), M, d_bidx.data_ptr())]
    for d_ in dbs:
        d_.hints = pkg.BATCH_READY      # the batch buffers are static and complete: the library may broadcast batch n+1 while batch n is packed
    db.hints = pkg.BATCH_READY
    state = {"i": 0}

    def step_device(release=True):
        # the engine double-buffers nothing of the CALLER's: two ingest buffers alternate so that the
        # broadcast of step i+1 (library, ingest stream) never touches the frames step i's pack reads
        k = state["i"] & 1
        state["i"] += 1
        b = eng.submit_device(dbs[k])
        if release:
            eng.release_batch(b)                 # the consumer (NIC hand-off) frees the ring space
        return b

    def drain_device():
        state["i"] = 0

    def sync_all():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    with torch.cuda.stream(stream):
        for _ in range(args.warmup):
            step_device()
        drain_device()
        sync_all()
        sampler = ClockSampler(local)
        sampler.start()
        launches0 = eng.stats().kernel_launches
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record(stream)
        for i in range(args.steps):
            # --dump-outputs: the last batch stays unreleased until its result has been read below (its
            # release, one small kernel, then runs after the timed window instead of inside it)
            last = step_device(release=not (args.dump_outputs and i == args.steps - 1))
        drain_device()                        # waits (on the stream) for the last pack
        ev1.record(stream)
        sync_all()
        if args.dump_outputs:
            if rank == 0:
                dump_outputs(eng, last, args.dump_outputs)
            eng.release_batch(last)
        gpu_launches = int(eng.stats().kernel_launches - launches0)   # counted by the library at every launch site
    ms = ev0.elapsed_time(ev1)
    t_ms = torch.tensor([ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t_ms, op=dist.ReduceOp.MAX)
    ms_max = float(t_ms.item())
    deliveries_step = M * n_conns
    egress_step = deliveries_step * F
    value = world * egress_step * args.steps / (ms_max * 1e-3) / 1e9

    # ---- sustained window: the same loop for >= 2 s (K steps take ~30 ms: too short to see clocks settle) ----
    sustained = None
    if args.sustain > 0:
        n_sus = max(args.steps, int(args.sustain * 1e3 / max(ms_max / args.steps, 1e-3)) + 1)
        with torch.cuda.stream(stream):
            sync_all()
            s2 = ClockSampler(local)
            s2.start()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            for _ in range(n_sus):
                step_device()
            drain_device()
            e1.record(stream)
            sync_all()
        t_s = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t_s, op=dist.ReduceOp.MAX)
        sus_ms = float(t_s.item())
        sustained = {"value": world * egress_step * n_sus / (sus_ms * 1e-3) / 1e9, "unit": "GB/s", "steps": n_sus,
                     "seconds": sus_ms * 1e-3, "ms_per_step": sus_ms / n_sus, "clocks": s2.stop()}
    # `clocks`: sampled from the start of the K-step region to the end of the sustained window (the same
    # loop, continuously under load; the K steps alone last ~30 ms = less than one nvidia-smi sample)
    clocks_timed = sampler.stop()
    sampler = ClockSampler(local)   # (the e2e legs below keep their own clock record)
    sampler.start()

    # ---- correctness of what was just timed: counters + every ring byte ----------------------------
    verify = "skipped"
    with torch.cuda.stream(stream):
        b = eng.submit_device(db)
        res = eng.poll(b)
        assert res.status == 0 and res.n_deliveries == deliveries_step and res.bytes_out == egress_step, \
            (res.status, res.n_deliveries, res.bytes_out)
        assert res.n_spans == n_conns and res.n_overflow == 0
        if not args.no_verify:
            base, rb, mc = eng.ring_info()
            image = bytearray()
            for fr in frames:
                image += L.to_bytes(4, "big") + fr + bytes(rec - F)
            # pad bytes are unspecified: compare only the F framed bytes of each record
            img = torch.from_numpy(np.frombuffer(bytes(image), dtype=np.uint8).copy()).to(dev).view(M, rec)[:, :F]
            ok = True
            if args.pool:
                # output pool: the batch is ONE region [pool_base, +n_conns * M * rec), connection after connection
                pb = int(res.pool_base) * 32

                class _Pool:
                    __cuda_array_interface__ = {"shape": (n_conns * M * rec,), "typestr": "|u1", "data": (base + pb, False), "version": 3}

                region = torch.as_tensor(_Pool(), device=dev).view(n_conns, M, rec)
                for c0 in range(0, n_conns, 1 << 16):
                    ok = ok and bool((region[c0:c0 + (1 << 16), :, :F] == img.unsqueeze(0)).all().item())
                runs = np.ctypeslib.as_array(C.cast(res.runs, C.POINTER(C.c_uint32)), shape=(res.n_runs, 6)).astype(np.int64)
                stride = M * rec // 32
                ok = ok and bool((runs[:, 2] == (runs[:, 0] - rank * sd.shard_stride) * stride).all()) and bool((runs[:, 3] == M * rec).all()) and \
                    bool((runs[:, 4] == M).all()) and bool((runs[:, 5] == stride).all()) and int(runs[:, 1].sum()) == n_conns
            else:
                class _Arr:
                    __cuda_array_interface__ = {"shape": (n_conns, rb), "typestr": "|u1", "data": (base, False), "version": 3}

                ring = torch.as_tensor(_Arr(), device=dev)
                off = res.runs[0].ring_off if res.runs else res.spans[0].ring_off
                for c0 in range(0, n_conns, 1 << 16):
                    blk = ring[c0:c0 + (1 << 16), off:off + M * rec].reshape(-1, M, rec)[:, :, :F]
                    ok = ok and bool((blk == img.unsqueeze(0)).all().item())
                if res.runs:   # run-length span table: {conn0, n_conns, ring_off, len, n_records, off_stride}
                    runs = np.ctypeslib.as_array(C.cast(res.runs, C.POINTER(C.c_uint32)), shape=(res.n_runs, 6))
                    covered = np.concatenate([np.arange(c0, c0 + n, dtype=np.int64) for c0, n in runs[:, :2]])
                    ok = ok and bool((runs[:, 2] == off).all()) and bool((runs[:, 3] == M * rec).all()) and \
                        bool((runs[:, 4] == M).all()) and len(np.unique(covered)) == n_conns == len(covered)
                else:
                    spans = np.ctypeslib.as_array(C.cast(res.spans, C.POINTER(C.c_uint32)), shape=(res.n_spans, 4))
                    ok = ok and bool((spans[:, 1] == off).all()) and bool((spans[:, 2] == M * rec).all()) and \
                        bool((spans[:, 3] == M).all()) and len(np.unique(spans[:, 0])) == n_conns
            assert ok, "ring contents differ from the expected framed records"
            verify = "all %d connections x %d records bit-exact" % (n_conns, M)
        eng.release_batch(b)

    # ---- per-kernel time for the roofline (CUDA events inside the engine, on the same stream) ------
    eng.set_timing(True)
    s0 = eng.stats()
    with torch.cuda.stream(stream):
        ids = []
        for _ in range(args.steps):
            b = eng.submit_device(db)
            eng.poll(b)
            eng.release_batch(b)
        torch.cuda.synchronize(dev)
    s1 = eng.stats()
    eng.set_timing(False)
    nb = max(1, s1.timed_batches - s0.timed_batches)
    ms_pack = (s1.ms_pack - s0.ms_pack) / nb
    ms_match = (s1.ms_match - s0.ms_match) / nb
    ms_plan = (s1.ms_plan - s0.ms_plan) / nb
    pack_bytes = M * (n_conns * F + L)          # algorithmic bytes of one pack launch: D*F stores + L read per message
    peak, peak_src = measured_peak()
    achieved = pack_bytes / (ms_pack * 1e-3) / 1e9
    traffic, traffic_source = None, None
    tp = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(tp):
        try:
            traffic = json.load(open(tp)).get("k_pack_dram_bytes_per_launch")
            traffic_source = "static ncu capture (profiles/traffic.json: dram__bytes_read.sum + dram__bytes_write.sum of one --set full launch)"
        except Exception:
            traffic = None

    # ---- e2e: host buffers through the C ABI, H2D + D2H inside the timed region ---------------------
    # (N>1: same call on every rank — the SPMD contract; only rank 0's bytes are used, the other ranks
    #  pass zero-filled frames of the same shape and receive the real ones over NVLink)
    host_msgs = [("b", [0], fr if rank == 0 else bytes(len(fr)), False) for fr in frames]
    e2e_steps = args.steps

    def step_e2e():
        b = eng.submit(host_msgs)                # pinned staging + H2D (+ library ncclBroadcast) + kernels
        r = eng.poll(b)                          # D2H: counters + span table
        eng.release_batch(b)
        return r

    with torch.cuda.stream(stream):
        for _ in range(3):
            step_e2e()
        sync_all()
        t0 = time.perf_counter()
        for _ in range(e2e_steps):
            r = step_e2e()
        torch.cuda.synchronize(dev)
        t1 = time.perf_counter()
    t_e2e = torch.tensor([t1 - t0], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t_e2e, op=dist.ReduceOp.MAX)
    e2e_value = world * egress_step * e2e_steps / float(t_e2e.item()) / 1e9
    # ---- e2e_host: the same step, and every framed byte made readable by a socket writer -----------
    # pcdn_egress_drain (SURVEY 8f-2): per batch a gather kernel packs the records of each chunk of
    # spans into one contiguous device buffer, one DMA per 64 MiB chunk brings it into pinned host
    # memory (double-buffered), where the sink — the writev writer in production — reads it.  This is
    # PCIe-bound; it is the number to hold against a CPU broker whose output lands in host memory.
    e2e_host = None
    if not args.no_e2e_host:
        eg = pkg.Egress(eng)
        nh = max(2, min(args.steps, 6))

        def step_host(sink=None):
            b = eng.submit(host_msgs)
            st = eg.drain(b, sink)               # poll + gather + chunked D2H of every record of the batch
            eng.release_batch(b)
            return st

        with torch.cuda.stream(stream):
            step_host()
            sync_all()
            t0 = time.perf_counter()
            for _ in range(nh):
                st = step_host()
            t1 = time.perf_counter()
        t_h = torch.tensor([t1 - t0], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t_h, op=dist.ReduceOp.MAX)
        assert st.spans == n_conns and st.bytes == n_conns * M * rec, (st.spans, st.bytes)
        host_verify = "skipped"
        if not args.no_verify:
            # one more batch through a checking sink: EVERY record of EVERY connection, read from the
            # host memory the sink is given, must be the expected framed bytes
            image = np.frombuffer(b"".join(L.to_bytes(4, "big") + fr + bytes(rec - F) for fr in frames), dtype=np.uint8)
            keep = np.ones(M * rec, dtype=bool)
            for m in range(M):
                keep[m * rec + F:(m + 1) * rec] = False      # pad bytes are unspecified
            seen = {"spans": 0, "bad": 0}

            def check(ch):
                n = ch.n_spans
                flat = np.ctypeslib.as_array(C.cast(ch.data, C.POINTER(C.c_uint8)), shape=(ch.bytes,))
                offs = np.ctypeslib.as_array(ch.data_off, shape=(n,))
                # the spans of a chunk lie at a constant stride: back to back in a staged chunk, one ring apart when
                # the sink reads host rings in place
                so = np.sort(offs.astype(np.int64))          # (in-place host rings: the span table is in CTA order, not address order)
                st = int(so[1] - so[0]) if n > 1 else M * rec
                ap = st >= M * rec and bool((so == so[0] + np.arange(n, dtype=np.int64) * st).all()) and int(so[-1]) + M * rec <= ch.bytes
                if not ap:
                    seen["bad"] += 1
                    return
                a = np.lib.stride_tricks.as_strided(flat[int(so[0]):], shape=(n, M * rec), strides=(st, 1), writeable=False)
                sp = np.ctypeslib.as_array(C.cast(ch.spans, C.POINTER(C.c_uint32)), shape=(n, 4))
                ok = bool((a[:, keep] == image[keep]).all()) \
                    and bool((sp[:, 2] == M * rec).all()) and bool((sp[:, 3] == M).all())
                seen["spans"] += n
                seen["bad"] += 0 if ok else 1

            with torch.cuda.stream(stream):
                step_host(check)
            assert seen["spans"] == n_conns and seen["bad"] == 0, seen
            host_verify = "all %d connections x %d records bit-exact in host memory" % (n_conns, M)
        e2e_host = {"value": world * egress_step * nh / float(t_h.item()) / 1e9, "unit": "GB/s", "steps": nh,
                    "d2h_bytes_per_step": n_conns * M * rec + (16 * n_conns if args.plain_spans else 24 * int(r.n_runs)) + 64, "h2d_bytes_per_step": M * slot + 64 + 22 * M + 64 + 24 * n_conns,
                    "chunks_per_step": int(st.chunks), "verify": host_verify,
                    "note": "pcdn_submit (host buffers) -> pcdn_egress_drain: every framed record lands in pinned host memory "
                            "(gather kernel + one DMA per 64 MiB chunk, double-buffered); PCIe-bound"}
        eg.close()
    clocks = sampler.stop()  # sampled from the start of the timed region to the end of the e2e loop (all under load)
    h2d = M * slot + 64 + 22 * M + 64 if (world == 1 or rank == 0) else 0
    d2h = 64 + (16 * n_conns if args.plain_spans else 24 * int(r.n_runs))

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu:
        try:
            cores = os.cpu_count() or 1
            cmodel, calib = pick_cpu_model(n_conns, args.payload, M, cores)
            r = run_cpu_reference(n_conns, args.payload, M, 3, 1, cores, timeout=600, model=cmodel)
            cpu = {"value": r["gbps_median_step"], "unit": "GB/s", "cores": r["threads"], "kind": "port",
                   "sample": "%d msgs x %d subscribers per step, median of 3 steps after 1 warm-up (mean over the 3: %.3f GB/s)" % (M, n_conns, r["gbps"]),
                   "model": r.get("model"), "model_calibration": calib,
                   "deliveries_per_s": r["deliveries_per_s"], "stage12_s": r["stage12_s"], "stage3_s": r["stage3_s"]}
        except Exception as ex:  # the baseline is reported, never required for our number
            cpu = {"value": None, "unit": "GB/s", "cores": os.cpu_count(), "kind": "port", "sample": "failed: %r" % (ex,)}

    # ---- secondary configs (BASELINE.json C4 / C5 sparse / C3) so that the driver's run covers them ----
    secondary = None
    if rank == 0 and world == 1 and not args.no_secondary:
        eng.close()          # the C2 engine's 18 GB of rings go back before the next engines are built
        eng = None
        secondary = {}
        for wl, extra in (("C4", []), ("C5sparse", []), ("C3", [])):
            try:
                out = subprocess.run([sys.executable, "-B", os.path.join(ROOT, "bench_configs.py"), "--workload", wl, "--steps", "10", "--warmup", "3"] + extra,
                                     capture_output=True, text=True, timeout=420, check=True)
                d = json.loads(out.stdout.strip().splitlines()[-1])
                secondary[wl] = {"workload": d["config"]["workload"], "value": d["value"], "unit": d["unit"], "ms_per_step": d["ms_per_step"],
                                 "msgs_per_s": d["msgs_per_s"], "deliveries_per_s": d["deliveries_per_s"],
                                 "algorithmic_GBps": d["algorithmic_GBps"], "frac": d["frac_of_hbm_peak"],
                                 "frac_note": "ALGORITHMIC bytes of the whole step (SURVEY 8d) / step time / measured HBM peak",
                                 "stage_ms": d["roofline"]["stage_ms"], "verify": d["verify"], "clocks": d["clocks"]}
            except Exception as ex:
                secondary[wl] = {"error": repr(ex)[:300]}

    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": "GB/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_max / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "u8", "data": "synthetic",
            "deliveries_per_s": world * deliveries_step * args.steps / (ms_max * 1e-3),
            "ingress_msgs_per_s": M * args.steps / (ms_max * 1e-3),
            "frac_of_hbm_peak": value / world / peak,
            "config": {"workload": ("C2: 2^20 subscribers/GPU, 1 topic, 1 KiB broadcast, batches of %d" % M) if n_conns == N_CONNS and not args.host_rings
                       else "%d subscribers/GPU, 1 topic, %d B broadcast, batches of %d%s" % (n_conns, args.payload, M, ", rings in mapped pinned HOST memory (PCIe-bound egress hand-off)" if args.host_rings else ""),
                       "n_conns_per_gpu": n_conns, "payload": args.payload, "frame_bytes": F, "msgs_per_step": M,
                       "ring_bytes_per_conn": ring_bytes, "parallelism": ("connection shards x%d behind one sharded engine (pcdn_config.world_shards), " % world +
                                                                          ("every shard copies the batch from host memory" if args.ingest == "host" else
                                                                           "library-issued ncclBroadcast ingest over NVLink (%d ranks)" % sd.nccl_ranks))
                       if world > 1 else "single GPU", "l2": "outputs 9.1 GB/step >> L2; inputs 8.7 KB (algorithmically resident)",
                       "output": "shared output pool (PCDN_FLAG_OUTPUT_POOL)" if args.pool else "per-connection rings",
                       "pack_variant": args.variant, "verify": verify, "setup_s": round(setup_s, 2)},
            "roofline": {"bound": "hbm", "kernel": "k_pack (connection-major phase)" if not (args.variant & 2) else "k_pack (message-major phase)", "achieved": achieved, "peak": peak, "unit": "GB/s",
                         "frac": achieved / peak, "traffic": traffic, "traffic_source": traffic_source, "peak_source": peak_src,
                         "algorithmic_bytes_per_launch": pack_bytes, "ms_per_launch": ms_pack,
                         "stage_ms": {"match": ms_match, "plan_offsets": ms_plan, "pack": ms_pack}},
            "cpu_baseline": cpu,
            "e2e": {"value": e2e_value, "unit": "GB/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "timing": "wall clock between device synchronisations, max over ranks",
                    "output": "HBM-resident",
                    "note": "HBM-RESIDENT OUTPUT: the framed bytes stay in the HBM rings (NIC hand-off by GPUDirect, SURVEY 8f-2); the "
                            "host reads back counters + span table only.  e2e_host below is the same step with every byte brought "
                            "to host memory"},
            "e2e_host": e2e_host,
            "clocks": clocks_timed, "clocks_e2e": clocks,
            "gpu_launches": gpu_launches,
            "gpu_launches_note": "kernels launched by libpcdn_fanout.so inside the timed region (library-side counter at every launch site): "
                                 "k_match, k_plan_a, k_offsets, k_pack, k_release per step",
            "sustained": sustained,
            "secondary": secondary,
        }
        print(json.dumps(line), flush=True)
    if eng is not None:
        eng.close()
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
