#!/usr/bin/env python
"""bench.py — headline benchmark of the B200 block-compression engine (contract: see the task statement / DESIGN.md).

Default workload at N=1 = the configuration BASELINE.json's `metric` is quoted on: a 200,000,000-byte silesia.tar-shaped
slab (kanzi-go_b200/synth.py: silesia_shaped, SURVEY.md §8d C3), 4 MiB blocks (48 blocks), compressed and decompressed at
kanzi `-l 3` (TEXT+UTF+PACK+MM+LZX & HUFFMAN) AND `-l 5` (TEXT+UTF+BWT+RANK+ZRLT & ANS0) (app/BlockCompressor.go:665-700).
A "step" is one pass of the hot path over that slab: compress + decompress at -l 3 and compress + decompress at -l 5. The
two round trips belong to two contexts (one CUDA stream each) driven by two host threads: -l 5 compresses, and while it
decompresses - its serial RANK inverse chains occupy 48 of the 148 SMs for most of that time - the -l 3 round trip runs beside
it on the other SMs; a step ends when both have ended.

  value  = uncompressed bytes through the four passes per second (MB = 1e6 B), inputs resident in HBM (device API);
           "sequential" = the same steps with the levels one after the other (the schedule of the lines before r02_h);
           "levels" holds encode / decode / combined MB/s of each level on its own, and inside the side-by-side steps
  e2e    = the same through the host-buffer C ABI (kz_compress_stream / kz_decompress_stream) from pinned host
           memory, host<->device copies inside the timed region
  roofline: the kernel with the largest share of the step; achieved = algorithmic bytes of its stage (stage input +
           stage output bytes over the batch, SURVEY §8d) / CUDA-event time of the launch
  cpu_baseline / --impl reference: the C++ restatement of the reference path (oracle/, "port": no Go toolchain here)
           with one worker per block on all host cores, same slab, same levels.
With N > 1 ranks: see --mode. "weak" (default): every rank processes its own slab (no data-path collective: blocks are
independent, SURVEY.md §8e); "sharded": ONE slab on rank 0, block ranges scattered over NCCL, encoded shards gathered and
committed in order on rank 0 (and the mirror for decode) — reported inside the same line under "sharded".
Other workloads (--workload) are single-pass lines used for profiles/ (configs[1], configs[4] points, sub-pipelines).
"""
import argparse
import importlib
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

L3 = ("l3", "TEXT+UTF+PACK+MM+LZX", "HUFFMAN")
L5 = ("l5", "TEXT+UTF+BWT+RANK+ZRLT", "ANS0")
# name: (passes [(label, transform, entropy)], block size, bytes per GPU, data generator, metric label)
WORKLOADS = {
    "silesia": ([L3, L5], 4 << 20, 200_000_000, "silesia",
                "encode+decode MB/s, 200 MB silesia-shaped slab, kanzi -l 3 and -l 5, 4 MiB blocks"),
    "silesia_l3": ([L3], 4 << 20, 200_000_000, "silesia", "encode+decode MB/s, 200 MB silesia-shaped slab, kanzi -l 3"),
    "silesia_l5": ([L5], 4 << 20, 200_000_000, "silesia", "encode+decode MB/s, 200 MB silesia-shaped slab, kanzi -l 5"),
    "enwik_l5": ([L5], 32 << 20, 256 << 20, "enwik", "encode+decode MB/s, 256 MiB enwik-shaped text, kanzi -l 5 -b 32m (configs[3] shape, 8 blocks)"),
    "ans0": ([("ans0", "NONE", "ANS0")], 4 << 20, 64 * (4 << 20), "zipf1", "encode+decode MB/s (ANS0/NONE, 64x4MiB Zipf(1.0) blocks per GPU; BASELINE.json configs[1])"),
    "huffman": ([("huffman", "NONE", "HUFFMAN")], 4 << 20, 64 * (4 << 20), "zipf1", "encode+decode MB/s (HUFFMAN/NONE, 64x4MiB Zipf(1.0) blocks per GPU)"),
    "ans1": ([("ans1", "NONE", "ANS1")], 4 << 20, 64 * (4 << 20), "text", "encode+decode MB/s (ANS1/NONE, 64x4MiB order-1 text blocks per GPU; configs[4] at 4 MiB)"),
    "l3core": ([("l3core", "LZX", "HUFFMAN")], 4 << 20, 48 * (4 << 20), "text", "encode+decode MB/s (-t LZX -e HUFFMAN, 48x4MiB text blocks)"),
    "l5core": ([("l5core", "BWT+RANK+ZRLT", "ANS0")], 32 << 20, 4 * (32 << 20), "text", "encode+decode MB/s (-t BWT+RANK+ZRLT -e ANS0, 4x32MiB text blocks)"),
    "l5core4m": ([("l5core4m", "BWT+RANK+ZRLT", "ANS0")], 4 << 20, 16 * (4 << 20), "text", "encode+decode MB/s (-t BWT+RANK+ZRLT -e ANS0, 16x4MiB text blocks)"),
    "l2": ([("l2", "DNA+LZ", "HUFFMAN")], 4 << 20, 48 * (4 << 20), "text", "encode+decode MB/s (kanzi -l 2 = -t DNA+LZ -e HUFFMAN, 48x4MiB text blocks)"),
    "l1": ([("l1", "LZX", "NONE")], 4 << 20, 200_000_000, "silesia", "encode+decode MB/s, 200 MB silesia-shaped slab, kanzi -l 1"),
    "l4": ([("l4", "TEXT+UTF+EXE+PACK+MM+ROLZ", "NONE")], 4 << 20, 200_000_000, "silesia", "encode+decode MB/s, 200 MB silesia-shaped slab, kanzi -l 4"),
    "l3": ([L3], 4 << 20, 48 * (4 << 20), "text", "encode+decode MB/s (kanzi -l 3, 48x4MiB markov text blocks)"),
    "l5": ([L5], 4 << 20, 16 * (4 << 20), "text", "encode+decode MB/s (kanzi -l 5, 16x4MiB markov text blocks)"),
    "tiny": ([L3, L5], 256 << 10, 2_000_000, "silesia", "encode+decode MB/s, 2 MB silesia-shaped slab, kanzi -l 3 and -l 5, 256 KiB blocks (contract test of the line, not a measurement)"),
}
for _bs in (1, 2, 4, 8, 16, 32, 64):  # BASELINE.json configs[4]: ANS1 block-size sweep over 256 MiB of order-1 text
    WORKLOADS["ans1_%dm" % _bs] = ([("ans1", "NONE", "ANS1")], _bs << 20, 256 << 20, "text",
                                   "encode+decode MB/s (ANS1/NONE, 256 MiB order-1 text, %d MiB blocks; configs[4])" % _bs)

# kernel name -> (stage the kernel belongs to, as kz_stage_bytes names it) for the roofline's algorithmic bytes
STAGE_OF = {"lz_parse": "fwd:16", "lz_gather": "fwd:16", "lz_hash": "fwd:16", "lz_sort": "fwd:16", "lz_link": "fwd:16", "lz_spec": "fwd:16", "lz_stitch": "fwd:16", "lz_emit": "fwd:16", "lz_inverse": "inv:16", "text_forward": "fwd:10", "text_inverse": "inv:10", "utf_forward": "fwd:17",
            "utf_inverse": "inv:17", "bwt_forward": "fwd:1", "bwt_inverse": "inv:1", "sbrt_rank": "fwd:8", "sbrt_inverse": "inv:8", "zrlt_forward": "fwd:6",
            "zrlt_inverse": "inv:6", "alias_forward": "fwd:18", "alias_inverse": "inv:18", "fsd_forward": "fwd:15", "fsd_inverse": "inv:15",
            "rolz_forward": "fwd:11", "rolz_inverse": "inv:11", "exe_forward": "fwd:9", "exe_inverse": "inv:9"}


def make_data(kind, n, seed):
    synth = importlib.import_module("kanzi-go_b200.synth")
    if kind == "zipf1":
        return synth.zipf_bytes(n, 1.0, seed=seed)
    if kind == "text":
        return synth.markov_text(n, seed=seed)
    if kind == "silesia":
        return synth.silesia_shaped(n, seed=seed)
    if kind == "enwik":
        return synth.enwik_shaped(n, seed=seed)
    raise ValueError(kind)


def measured_traffic(kernel):
    """dram__bytes_read.sum + dram__bytes_write.sum of `kernel` from the newest committed `ncu --set full` summary
    (profiles/*ncu*summary.json, written by tools/ncu_summary.py): per launch of the default workload, or None."""
    import glob

    best = None
    files = sorted(glob.glob(os.path.join(ROOT, "profiles", "r02*ncu*summary*.json")), key=lambda f: ("final" in os.path.basename(f), os.path.basename(f)))
    for f in files:  # the capture named "final" wins, otherwise the highest generation
        try:
            for k in json.load(open(f)).get("kernels", []):
                if kernel in k.get("kernel", "") and k.get("dram_traffic_bytes"):
                    best = (float(k["dram_traffic_bytes"]), os.path.basename(f))
        except Exception:
            pass
    return best


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler(threading.Thread):
    def __init__(self, index):
        super().__init__(daemon=True)
        self.index = index
        self.samples = []
        self.reasons = set()
        self.stop_flag = False
        self.max_mhz = None

    def run(self):
        q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        while not self.stop_flag:
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q, "--format=csv,noheader,nounits"], capture_output=True,
                                     text=True, timeout=5).stdout.strip().split("\n")[0]
                f = [x.strip() for x in out.split(",")]
                self.samples.append(float(f[0]))
                self.max_mhz = float(f[1])
                for nme, v in zip(names, f[2:6]):
                    if v.lower().startswith("active"):
                        self.reasons.add(nme)
            except Exception:
                pass
            time.sleep(0.1)

    def summary(self):
        return {"sm_mhz": float(np.median(self.samples)) if self.samples else None, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(self.samples)}


def cpu_reference(steps, warmup, workload, max_seconds=60.0):
    """Times the CPU restatement of the reference path (oracle) with one worker per block on all host cores: the same slab and the
    same passes as the GPU arm. Bounded: stops taking further steps once max_seconds of CPU work were spent."""
    from oracle import pyoracle

    synth = importlib.import_module("kanzi-go_b200.synth")
    passes, BLOCK, n, kind, _ = WORKLOADS[workload]
    cores = os.cpu_count() or 1
    jobs = min(64, cores)
    x = make_data(kind, n, synth.SEED + 1)
    times, per, outputs = [], {}, {}
    t_all = time.perf_counter()
    for it in range(warmup + steps):
        tot = 0.0
        for label, transform, entropy in passes:
            te, td = [], []
            s = pyoracle.compress(x, transform, entropy, block_size=BLOCK, jobs=jobs, input_size=n, timing=te)
            y = pyoracle.decompress(s, n + 64, jobs=jobs, timing=td)
            if it == 0:
                assert np.array_equal(y, x)
            tot += te[0] + td[0]
            outputs[label] = (s, y)
            if it >= warmup or it == warmup + steps - 1:
                per[label] = {"encode_MBps": n / te[0] / 1e6, "decode_MBps": n / td[0] / 1e6, "MBps": 2 * n / (te[0] + td[0]) / 1e6, "compressed_bytes": int(len(s))}
        if it >= warmup:
            times.append(tot)
        if time.perf_counter() - t_all > max_seconds and times:
            break
    t = float(np.mean(times))
    return {"value": 2 * n * len(passes) / t / 1e6, "unit": "MB/s", "cores": jobs, "kind": "port",
            "sample": "the whole workload (%d bytes of %s data, %d-byte blocks; %s), compress+decompress in memory, %d worker threads, %d timed step(s); "
                      "C++ restatement of kanzi-go (no Go toolchain in this image)"
                      % (n, kind, BLOCK, " and ".join("-t %s -e %s" % (p[1], p[2]) for p in passes), jobs, len(times)),
            "ms_per_step": t * 1e3, "levels": per, "steps": len(times), "outputs": outputs}


def static_config(workload, passes, block, nblocks, n, world):
    """The workload description, identical in the b200 arm and in the reference arm (nothing measured in here)."""
    cfg = {"workload": workload_label(workload), "block_size": block, "blocks": nblocks, "uncompressed_bytes": n,
           "levels": {p[0]: {"transform": p[1], "entropy": p[2]} for p in passes},
           "l2": "slab (%d MB) and compressed streams larger than the 126 MB L2" % (n // 1000000)}
    if world == 1:
        cfg["parallelism"] = "1 process, 1 GPU"
    else:
        cfg["parallelism"] = ("%d ranks, ONE slab: contiguous block ranges per rank (%d blocks each), NCCL scatter of the input / gather-v of the encoded "
                              "fragments, ordered commit on rank 0; the replicas measurement of the same run is under \"weak\"" % (world, (nblocks + world - 1) // world))
    return cfg


def workload_label(name):
    passes, block, n, kind, _ = WORKLOADS[name]
    data = {"zipf1": "Zipf(1.0) bytes", "text": "order-1 markov text", "silesia": "silesia.tar-shaped mix (synth.silesia_shaped: 35% text, 25% x86-like, 15% records, 10% 16-bit walks, 10% XML, 5% random)",
            "enwik": "enwik9-shaped text (synth.enwik_shaped)"}[kind]
    lv = " and ".join("%s (-t %s -e %s)" % (p[0], p[1], p[2]) for p in passes)
    return "%d bytes of %s, %d blocks of %d MiB, %s" % (n, data, (n + block - 1) // block, block >> 20, lv) + \
        (" (BASELINE.json metric configuration)" if name == "silesia" else "")


DUMP_BYTES = 48 << 20  # all arrays of --dump-outputs together, in float32
DUMP_SEED = 0x44554D50


def dump_outputs(directory, outputs):
    """--dump-outputs: for every level, the stream the last timed step wrote (<label>_compressed) and the bytes it decoded from it
    (<label>_decompressed), as float32 .npy files, and their lengths in bytes (<label>_sizes, float64). An array larger than its
    share of DUMP_BYTES is written as its elements at a fixed, seeded sample of positions (sorted): two builds that compute the
    same bytes write the same files."""
    os.makedirs(directory, exist_ok=True)
    cap = DUMP_BYTES // 4 // (2 * len(outputs))
    for label, (compressed, decompressed) in outputs.items():
        np.save(os.path.join(directory, label + "_sizes.npy"), np.array([len(compressed), len(decompressed)], dtype=np.float64))
        for kind, a in (("compressed", compressed), ("decompressed", decompressed)):
            if len(a) > cap:
                a = a[np.sort(np.random.default_rng(DUMP_SEED).integers(0, len(a), cap))]
            np.save(os.path.join(directory, "%s_%s.npy" % (label, kind)), np.asarray(a, dtype=np.float32))


def emit(line):
    """Writes the one JSON line to the real stdout (fd 1 is pointed at stderr during the run so that library chatter such
    as "NCCL version ..." cannot end up in front of it)."""
    os.write(_REAL_STDOUT, (json.dumps(line) + "\n").encode())


_REAL_STDOUT = os.dup(1)
os.dup2(2, 1)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--mode", default="auto", choices=["auto", "weak", "sharded"])
    ap.add_argument("--workload", default="silesia", choices=sorted(WORKLOADS))
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step computed to DIR/<name>.npy (see dump_outputs)")
    args = ap.parse_args()
    passes, BLOCK, n, kind, METRIC = WORKLOADS[args.workload]
    NBLOCKS = (n + BLOCK - 1) // BLOCK
    args.warmup = max(args.warmup, 3) if args.impl != "reference" else max(args.warmup, 1)

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))

    if args.impl == "reference":
        if rank != 0:
            return 0
        # K steps and W warm-up steps as asked (every step = the whole workload, 2-3 s on the box's 64 cores); a wall-clock cap of 4 minutes keeps a
        # large K within "a few minutes" and is reported through `steps`
        r = cpu_reference(max(args.steps, 1), max(args.warmup, 1), args.workload, max_seconds=240.0)
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, r["outputs"])
        line = {"impl": "reference", "metric": METRIC, "value": r["value"], "unit": "MB/s", "n_gpus": args.gpus, "steps": r["steps"], "warmup": max(args.warmup, 1),
                "ms_per_step": r["ms_per_step"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
                "config": static_config(args.workload, passes, BLOCK, NBLOCKS, n, world), "levels": r["levels"],
                "schedule": "levels one after the other, every pass on all %d worker threads (side by side they would only share the same cores)" % r["cores"],
                "cpu_baseline": {k: r[k] for k in ("value", "unit", "cores", "kind", "sample")},
                "e2e": {"value": r["value"], "unit": "MB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0}
        emit(line)
        return 0

    import torch

    dist = None
    if world > 1:
        import torch.distributed as dist

        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    kz = importlib.import_module("kanzi-go_b200")
    synth = importlib.import_module("kanzi-go_b200.synth")
    torch.cuda.set_device(local_rank)
    ctx = kz.Context(local_rank)
    x = make_data(kind, n, synth.SEED + 1 + rank)
    cap = int(ctx.lib.kz_max_stream_output(n, BLOCK))
    P = [(label, kz.transform_type(tr), kz.entropy_type(en)) for label, tr, en in passes]

    # ---------------- device-resident pass (value) ----------------
    # one context (= one CUDA stream + its workspaces) and one host thread per level: the round trips of a step run side by side, the way two
    # callers of the C ABI would drive one GPU; the same steps with the levels one after the other are timed as well ("sequential")
    ctxs = [ctx] + [kz.Context(local_rank) for _ in P[1:]]
    ext = [torch.cuda.ExternalStream(c.cuda_stream()) for c in ctxs]
    d_src = torch.empty(n + 256, dtype=torch.uint8, device="cuda")
    d_cmp = [torch.zeros(cap + 256, dtype=torch.uint8, device="cuda") for _ in P]
    d_dec = [torch.empty(n + 256, dtype=torch.uint8, device="cuda") for _ in P]
    d_src[:n].copy_(torch.from_numpy(x))
    torch.cuda.synchronize()

    def barrier():
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    m = [0] * len(P)

    def device_round_trip(i, enc, dec, before=None, between=None):
        label, t48, et = P[i]
        with torch.cuda.stream(ext[i]):
            a, b, c = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            if before:
                before()
            a.record()
            m[i] = ctxs[i].compress_device(d_src.data_ptr(), n, d_cmp[i].data_ptr(), cap, t48, et, BLOCK, 0, n)
            b.record()
            if between:
                between()
            k = ctxs[i].decompress_device(d_cmp[i].data_ptr(), m[i], d_dec[i].data_ptr(), n)
            c.record()
            c.synchronize()
        assert k == n, "decoded %d of %d bytes at %s" % (k, n, label)
        enc[i] += a.elapsed_time(b)
        dec[i] += b.elapsed_time(c)

    def timed_region(steps, one, side_by_side):
        """`steps` steps of one(i, enc, dec) for every level i; device milliseconds of the whole region and per level."""
        enc, dec = [0.0] * len(P), [0.0] * len(P)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        errors = []
        barrier()
        t0 = time.perf_counter()
        e0.record(ext[0])
        if side_by_side and len(P) > 1:
            gate = threading.Barrier(len(P))
            coded = [threading.Event() for _ in range(steps)]  # step k: the anchor level has written its stream

            def worker(i):
                try:
                    torch.cuda.set_device(local_rank)
                    for k in range(steps):
                        gate.wait()  # a step starts when every level finished the previous one
                        if i == anchor:
                            one(i, enc, dec, None, coded[k].set)
                        else:  # beside the anchor's decode
                            one(i, enc, dec, lambda: coded[k].wait(120.0) or gate.abort(), None)
                except BaseException as e:  # noqa: B902 - reported by the main thread
                    errors.append(e)
                    gate.abort()
                    for ev in coded:
                        ev.set()

            th = [threading.Thread(target=worker, args=(i,)) for i in range(len(P))]
            for t in th:
                t.start()
            for t in th:
                t.join()
        else:
            for _ in range(steps):
                for i in range(len(P)):
                    one(i, enc, dec)
        e1.record(ext[0])  # every level synchronised its own stream at the end of its round trip: the streams are idle here
        barrier()
        if errors:
            raise errors[0]
        return e0.elapsed_time(e1), (time.perf_counter() - t0) * 1e3, enc, dec

    anchor = 0
    seq_steps = max(1, min(args.steps, 3))
    for w in range(args.warmup):
        for d in d_dec:
            d.zero_()
        _, _, _, w_dec = timed_region(1, device_round_trip, w > 0)
        for i, (label, t48, et) in enumerate(P):
            assert torch.equal(d_dec[i][:n], d_src[:n]), "round trip mismatch at %s" % label
        if w == 0:
            # the level with the longest decode (-l 5: the serial RANK inverse chains on 48 SMs) is the anchor of a step: the other levels run their
            # round trips beside its decode, after its encode
            anchor = max(range(len(P)), key=lambda i: w_dec[i])

    def profiling(on):
        for c in ctxs:
            c.profile(on)
            c.profile_reset()
            c.launch_count(reset=True)

    def collect(steps):
        """CUDA-event times of the kernels and byte counts of the stages since profiling(True), over all contexts."""
        kern, stages = {}, {}
        for c in ctxs:
            for name in c.profile_names():
                if name.startswith("stage:"):
                    cnt, bi, bo = c.stage_bytes(name)
                    if cnt:
                        st = stages.setdefault(name[6:], {"bytes_in": 0.0, "bytes_out": 0.0, "batches_per_step": 0.0})
                        st["bytes_in"] += bi
                        st["bytes_out"] += bo
                        st["batches_per_step"] += cnt
                    continue
                cnt, ms = c.kernel_time(name)
                if cnt:
                    kk = kern.setdefault(name, {"launches": 0, "ms_avg": 0.0, "ms_per_step": 0.0})
                    kk["launches"] += cnt
                    kk["ms_per_step"] += ms
        for kk in kern.values():
            kk["ms_avg"] = kk["ms_per_step"] / kk["launches"]
            kk["ms_per_step"] /= steps
        for st in stages.values():
            cnt = st["batches_per_step"]
            st["bytes_in"] /= cnt
            st["bytes_out"] /= cnt
            st["batches_per_step"] = cnt / steps
        return kern, stages

    profiling(True)
    seq_ms, _, seq_enc, seq_dec = timed_region(seq_steps, device_round_trip, False)
    seq_kern, _ = collect(seq_steps)
    sampler = ClockSampler(local_rank)
    sampler.start()
    profiling(True)
    dev_ms, _, enc_ms, dec_ms = timed_region(args.steps, device_round_trip, True)
    launches = sum(c.launch_count(reset=True) for c in ctxs)
    kern, stages = collect(args.steps)
    profiling(False)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {label: (d_cmp[i][:m[i]].cpu().numpy(), d_dec[i][:n].cpu().numpy()) for i, (label, _, _) in enumerate(P)})

    # ---------------- end-to-end pass through the host-buffer C ABI (pinned host memory) ----------------
    e2e_ms, e2e_wall_ms, e2e_steps = 0.0, 0.0, 0
    if not args.no_e2e:
        h_src = torch.empty(n, dtype=torch.uint8).pin_memory()
        h_cmp = [torch.empty(cap, dtype=torch.uint8).pin_memory() for _ in P]
        h_dec = [torch.empty(n + 64, dtype=torch.uint8).pin_memory() for _ in P]
        h_src.numpy()[:] = x
        e2e_steps = max(1, min(args.steps, 3))

        def host_round_trip(i, enc, dec, before=None, between=None):
            label, t48, et = P[i]
            if before:
                before()
            mm = ctxs[i].compress_host(h_src.data_ptr(), n, h_cmp[i].data_ptr(), cap, t48, et, BLOCK, 0, n)
            if between:
                between()
            kk = ctxs[i].decompress_host(h_cmp[i].data_ptr(), mm, h_dec[i].data_ptr(), n + 64)
            assert kk == n and mm == m[i], "e2e round trip: %d bytes coded, %d decoded at %s" % (mm, kk, label)

        timed_region(1, host_round_trip, True)
        for i, (label, t48, et) in enumerate(P):
            assert np.array_equal(h_dec[i].numpy()[:n], x), "e2e round trip mismatch at %s" % label
        e2e_ms, e2e_wall_ms, _, _ = timed_region(e2e_steps, host_round_trip, True)
    sampler.stop_flag = True
    sampler.join(timeout=2)

    # ---------------- sharded: ONE slab (rank 0's), block ranges scattered over NCCL, fragments gathered and committed on rank 0 ----------------
    sharded = None
    if dist is not None and args.mode != "weak":
        par = importlib.import_module("kanzi-go_b200.parallel")
        sh = par.ShardedStream(par.GpuEngine(ctx, torch), dist, torch)
        slab = d_src if rank == 0 else None
        same_stream = True
        for w in range(2):
            for i, (label, t48, et) in enumerate(P):
                stream, nb = sh.compress(slab, n, t48, et, BLOCK, 0, n)
                back, mm = sh.decompress(stream, nb, n + 4096)
                if rank == 0 and w == 0:
                    same_stream = same_stream and nb == m[i] and bool(torch.equal(stream[:nb], d_cmp[i][:nb]))  # the bytes one GPU writes
                    assert mm == n and torch.equal(back[:n], d_src[:n]), "sharded round trip mismatch at %s" % label
        sh.t_exchange = sh.t_codec = 0.0
        s_steps = max(1, min(args.steps, 5))
        barrier()
        g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s_enc = [0.0] * len(P)
        s_dec = [0.0] * len(P)
        xbytes = 0
        g0.record()
        for _ in range(s_steps):
            for i, (label, t48, et) in enumerate(P):
                t_a = time.perf_counter()
                stream, nb = sh.compress(slab, n, t48, et, BLOCK, 0, n)
                xbytes += sh.exchanged_bytes
                torch.cuda.synchronize()
                t_b = time.perf_counter()
                sh.decompress(stream, nb, n + 4096)
                xbytes += sh.exchanged_bytes
                torch.cuda.synchronize()
                t_c = time.perf_counter()
                s_enc[i] += (t_b - t_a) * 1e3
                s_dec[i] += (t_c - t_b) * 1e3
        g1.record()
        barrier()
        sv = torch.tensor([g0.elapsed_time(g1), sh.t_exchange * 1e3, sh.t_codec * 1e3] + s_enc + s_dec, dtype=torch.float64, device="cuda")
        dist.all_reduce(sv, op=dist.ReduceOp.MAX)
        sv = [float(v) for v in sv.tolist()]
        xb = torch.tensor([float(xbytes)], dtype=torch.float64, device="cuda")
        dist.all_reduce(xb, op=dist.ReduceOp.SUM)
        if rank == 0:
            s_ms = sv[0] / s_steps
            se, sd = sv[3:3 + len(P)], sv[3 + len(P):]
            sharded = {"value": 2.0 * n * len(P) * s_steps / (sv[0] / 1e3) / 1e6, "unit": "MB/s", "ms_per_step": s_ms, "steps": s_steps,
                       "stream_identical_to_1gpu": bool(same_stream),
                       "exchange_ms_per_step_max_rank": sv[1] / s_steps, "codec_ms_per_step_max_rank": sv[2] / s_steps,
                       "nccl_bytes_per_step": float(xb.item()) / 2.0 / s_steps,  # every byte is counted by its sender and its receiver
                       "levels": {P[i][0]: {"encode_MBps": n * s_steps / (se[i] / 1e3) / 1e6, "decode_MBps": n * s_steps / (sd[i] / 1e3) / 1e6} for i in range(len(P))},
                       "how": "one %d-byte slab on rank 0; contiguous block ranges scattered with grouped NCCL send/recv; kz_compress_fragment_device on every rank; "
                              "all_gather of the bit lengths + gather-v of the fragments; ordered bit-granular commit on rank 0 (kz_concat_bits_device); the mirror "
                              "for decompression (kz_stream_index_device, windows scattered, kz_decompress_fragment_device, decoded ranges gathered)" % n}

    # ---------------- max over ranks ----------------
    vals = torch.tensor([dev_ms, e2e_ms, seq_ms] + enc_ms + dec_ms + seq_enc + seq_dec, dtype=torch.float64, device="cuda")
    if dist is not None:
        dist.all_reduce(vals, op=dist.ReduceOp.MAX)
    vals = [float(v) for v in vals.tolist()]
    dev_ms, e2e_ms, seq_ms = vals[0], vals[1], vals[2]
    L = len(P)
    enc_ms, dec_ms, seq_enc, seq_dec = vals[3:3 + L], vals[3 + L:3 + 2 * L], vals[3 + 2 * L:3 + 3 * L], vals[3 + 3 * L:3 + 4 * L]
    if rank != 0:
        if dist is not None:
            dist.destroy_process_group()
        return 0

    npass = len(P)
    total_bytes = 2.0 * n * npass * world  # uncompressed bytes through encode and through decode of every level, all ranks
    ms_per_step = dev_ms / args.steps
    value = total_bytes * args.steps / (dev_ms / 1e3) / 1e6
    e2e_value = total_bytes * e2e_steps / (e2e_ms / 1e3) / 1e6 if e2e_steps else None
    peak, peak_src = peaks()
    levels = {}
    for i, (label, t48, et) in enumerate(P):
        # a level's own rates: timed with the levels one after the other (nothing else on the GPU); "side_by_side" = inside the timed steps of `value`
        levels[label] = {"transform": passes[i][1], "entropy": passes[i][2], "compressed_bytes": int(m[i]), "ratio": m[i] / n,
                         "encode_MBps": n * world * seq_steps / (seq_enc[i] / 1e3) / 1e6, "decode_MBps": n * world * seq_steps / (seq_dec[i] / 1e3) / 1e6,
                         "MBps": 2.0 * n * world * seq_steps / ((seq_enc[i] + seq_dec[i]) / 1e3) / 1e6}
        if npass > 1:
            levels[label]["side_by_side"] = {"encode_MBps": n * world * args.steps / (enc_ms[i] / 1e3) / 1e6, "decode_MBps": n * world * args.steps / (dec_ms[i] / 1e3) / 1e6}
    schedule = ("one context (CUDA stream + workspaces) and one host thread per level; a step = %s compress, then %s decompress with the round trip(s) of %s beside "
                "it on the GPU; the step ends when all of them have" % (P[anchor][0], P[anchor][0], ", ".join(P[i][0] for i in range(npass) if i != anchor))) \
        if npass > 1 else "one context, one level"
    sequential = {"value": total_bytes * seq_steps / (seq_ms / 1e3) / 1e6, "unit": "MB/s", "ms_per_step": seq_ms / seq_steps, "steps": seq_steps,
                  "what": "the same steps with the levels one after the other on the GPU (the schedule of the earlier bench lines)"}
    # dominant kernel of the step = largest ms_per_step among device kernels
    roof = None
    dev_kern = {k: v for k, v in kern.items() if not k.startswith("host:")}
    if dev_kern:
        top = max(dev_kern, key=lambda k: dev_kern[k]["ms_per_step"])
        st = stages.get(STAGE_OF.get(top, ""))
        if st is not None:
            # a stage runs once per pass that contains it; per launch of the kernel = stage bytes of one batch / launches per batch
            per_batch_launches = max(1.0, dev_kern[top]["launches"] / args.steps / max(st["batches_per_step"], 1e-9))
            alg = (st["bytes_in"] + st["bytes_out"]) / per_batch_launches
            how = "stage input + output bytes of one batch (%s) / launches per batch" % STAGE_OF[top]
        else:
            alg = float(n + sum(m) / max(len(m), 1))
            how = "uncompressed + compressed bytes of the batch"
        ach = alg / (dev_kern[top]["ms_avg"] / 1e3) / 1e9
        roof = {"bound": "hbm", "kernel": top, "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak, "traffic": None, "peak_source": peak_src,
                "algorithmic_bytes_per_launch": alg, "algorithmic_bytes": how, "ms_per_launch": dev_kern[top]["ms_avg"],
                "share_of_step": dev_kern[top]["ms_per_step"] / ms_per_step}
        if npass > 1 and top in seq_kern:
            # with the levels one after the other (how a profiler's serialised launch list sees the step): the kernel alone on the GPU
            roof["sequential"] = {"ms_per_launch": seq_kern[top]["ms_avg"], "achieved": alg / (seq_kern[top]["ms_avg"] / 1e3) / 1e9,
                                  "share_of_step": seq_kern[top]["ms_per_step"] / (seq_ms / seq_steps)}
        t = measured_traffic(top)
        if t:
            roof["traffic"] = t[0]
            roof["traffic_source"] = "dram__bytes_read.sum + dram__bytes_write.sum per launch, ncu --set full, profiles/" + t[1]
    line = {
        "metric": METRIC, "value": value, "unit": "MB/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_per_step,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
        "config": static_config(args.workload, passes, BLOCK, NBLOCKS, n, world), "levels": levels,
        "schedule": schedule, "sequential": sequential,
        "clocks": sampler.summary(),
        "gpu_launches": int(launches),
        "kernels": dict(sorted(kern.items(), key=lambda kv: -kv[1]["ms_per_step"])),
        "stages": stages,
    }
    if e2e_steps:
        line["e2e"] = {"value": e2e_value, "unit": "MB/s", "h2d_bytes_per_step": int(n * npass + sum(m)), "d2h_bytes_per_step": int(sum(m) + n * npass),
                       "steps": e2e_steps, "ms_per_step": e2e_ms / e2e_steps, "wall_ms_per_step": e2e_wall_ms / e2e_steps,
                       "api": "kz_compress_stream + kz_decompress_stream per level, pinned host buffers; same schedule as `value`"}
    if roof:
        line["roofline"] = roof
    if sharded is not None:
        # N > 1: the headline is the sharded job (strong scaling: the same slab whatever N); the replicas measurement stays as "weak"
        line["weak"] = {"value": value, "unit": "MB/s", "ms_per_step": ms_per_step, "scaling": "weak", "levels": levels,
                        "what": "every rank compresses + decompresses its own %d-byte slab, no data-path collective" % n}
        if "e2e" in line:
            line["weak"]["e2e"] = line["e2e"]
        line["sharded"] = sharded
        line["value"] = sharded["value"]
        line["ms_per_step"] = sharded["ms_per_step"]
        line["steps"] = sharded["steps"]
        line["scaling"] = "strong"
    if world == 1 and not args.no_cpu_baseline:
        try:
            r = cpu_reference(1, 1, args.workload, max_seconds=30.0)
            line["cpu_baseline"] = {k: r[k] for k in ("value", "unit", "cores", "kind", "sample", "levels")}
        except Exception as e:  # the checker is absent: report, never substitute
            line["cpu_baseline"] = {"value": None, "unit": "MB/s", "cores": 0, "kind": "port", "sample": "unavailable: %s" % e}
    emit(line)
    if dist is not None:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
