#!/usr/bin/env python3
"""bench.py -- the driver's measurement contract for agrep-b200.

One "step" = one pass of the scan path over the whole synthetic corpus:
    agrep -2 'because each' <64 GiB newline-delimited text>      (BASELINE.json configs[1])
i.e. stage 1 (k_front, the HBM-bound kernel) + stage 2 (k_records) + the ordered list of matching records;
with N > 1 the 64 GiB are sharded by byte range over the ranks -- cut inside records, at multiples of 512 bytes -- and
every rank calls agb_scan_sharded(): the cut rule runs on the device, the match lists are gathered with NCCL inside the
library (C ABI, include/agrep_b200.h).

  python bench.py --gpus N --steps K --warmup W            our arm (one rank per GPU under torchrun)
  python bench.py --impl reference ...                      the reference's own CPU scan on the host cores
  python bench.py ... --dump-outputs DIR                    also write what the last timed step returned, as DIR/*.npy

Prints ONE JSON line (rank 0).  `value` = corpus bytes / device time (inputs resident in HBM);
`e2e` = the same scan through agb_scan_host() on pinned HOST buffers, H2D and result D2H inside the timing;
`roofline` = k_front's algorithmic bytes / its CUDA-event duration against MEASURED_PEAKS.json;
`cpu_baseline` = the unmodified reference binary (oracle/_ref/agrep, built from /root/reference) on a
bounded sample of the same corpus on the box's host cores.
"""
import argparse, ctypes, json, os, shutil, statistics, subprocess, sys, tempfile, threading, time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

PATTERN = "because each"          # 12-char literal made of two adjacent vocabulary words (SURVEY 8d)
K = 2
TOTAL_GIB = float(os.environ.get("AGB_BENCH_GIB", "64"))
E2E_GIB = float(os.environ.get("AGB_BENCH_E2E_GIB", "4"))
CPU_SAMPLE_MIB = int(os.environ.get("AGB_BENCH_CPU_MIB", "1024"))
NEEDLE_EVERY = 4096               # one planted line per 16 MiB, with 0..3 substitutions
REF_BIN = os.path.join(ROOT, "oracle", "_ref", "agrep")
PAGE = 4096


def peaks():
    try:
        p = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        return float(p["hbm_gbs"]), "MEASURED_PEAKS.json hbm_gbs (of measured)"
    except Exception:
        return 6650.0, "fallback 6.65 TB/s (of fallback)"


def host_cores():
    """the cores this process may actually use: scheduler affinity, cut by the cgroup CPU quota when there is one"""
    try:
        n = len(os.sched_getaffinity(0))
    except AttributeError:
        n = os.cpu_count() or 1
    quota = None
    for path in ("/sys/fs/cgroup/cpu.max", "/sys/fs/cgroup/cpu/cpu.cfs_quota_us"):
        try:
            f = open(path).read().split()
            if path.endswith("cpu.max"):
                if f[0] != "max":
                    quota = float(f[0]) / float(f[1])
            else:
                q = float(f[0])
                if q > 0:
                    quota = q / float(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
            break
        except Exception:
            continue
    usable = n if quota is None else max(1, min(n, int(quota + 0.5)))
    return {"os_cpu_count": os.cpu_count(), "affinity": n, "cgroup_quota_cpus": quota, "usable": usable}


def all_core_reference(ag, cores, shard_mib, steps=2):
    """`cores` unmodified reference processes at once, each over its own shard of the synthetic corpus (the program is
    single-threaded by construction, SURVEY 5): GB/s of the whole box, (matches, bytes) of one pass"""
    shard = (shard_mib << 20) // PAGE * PAGE
    base = "/dev/shm" if os.path.isdir("/dev/shm") and shutil.disk_usage("/dev/shm").free > cores * shard * 1.2 else tempfile.gettempdir()
    tmp = tempfile.mkdtemp(prefix="agb_ref_", dir=base)
    try:
        files = [os.path.join(tmp, "shard%03d.txt" % i) for i in range(cores)]

        def gen(i):
            data = ag.corpus_host(shard, first_page=i * (shard // PAGE), needle=PATTERN, needle_every=NEEDLE_EVERY, needle_maxedits=3)
            with open(files[i], "wb") as f:
                f.write(data)
        th = [threading.Thread(target=gen, args=(i,)) for i in range(cores)]
        [t.start() for t in th]; [t.join() for t in th]
        best, matched = None, 0
        for _ in range(steps):
            t0 = time.perf_counter()
            ps = [subprocess.Popen([REF_BIN, "-V0", "-c", "-n", "-%d" % K, PATTERN, f], stdout=subprocess.PIPE,
                                   stderr=subprocess.DEVNULL) for f in files]
            matched = sum(int((p.communicate()[0] or b"0").split()[0]) if p.wait() is not None else 0 for p in ps)
            dt = time.perf_counter() - t0
            best = dt if best is None else min(best, dt)
        return shard * cores / best / 1e9, matched, shard * cores
    finally:
        shutil.rmtree(tmp, ignore_errors=True)


class ClockSampler:
    """SM clock and throttle reasons DURING the timed region (B200_PROFILING.md's clocks line): NVML polled every 2 ms from a
    thread of this process (the timed region of a sharded run is a few tens of milliseconds, shorter than `nvidia-smi`
    takes to start), `nvidia-smi -lms` as the fallback; only the samples between begin() and end() count."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
    REASONS = ((0x8, "hw_slowdown"), (0x40, "hw_thermal_slowdown"), (0x20, "sw_thermal_slowdown"), (0x4, "sw_power_cap"))

    def __init__(self, gpu_index, uuid=None):
        self.idx, self.uuid, self.proc, self.lines = gpu_index, uuid, None, []
        self.samples, self.stop_flag, self.t0, self.t1, self.nvml, self.mx = [], False, None, None, None, None

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            h = None
            if self.uuid:
                try:
                    h = pynvml.nvmlDeviceGetHandleByUUID(self.uuid if isinstance(self.uuid, bytes) else str(self.uuid).encode())
                except Exception:
                    h = None
            if h is None:
                vis = os.environ.get("CUDA_VISIBLE_DEVICES")
                phys = self.idx
                if vis:
                    ent = vis.split(",")[self.idx].strip()
                    phys = int(ent) if ent.isdigit() else None
                h = pynvml.nvmlDeviceGetHandleByIndex(phys) if phys is not None else pynvml.nvmlDeviceGetHandleByUUID(ent.encode())
            self.mx = float(pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM))
            reasons = getattr(pynvml, "nvmlDeviceGetCurrentClocksEventReasons", None) or pynvml.nvmlDeviceGetCurrentClocksThrottleReasons
            self.nvml = (pynvml, h, reasons)
            self.t = threading.Thread(target=self._poll, daemon=True)
            self.t.start()
            return
        except Exception:
            self.nvml = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.idx), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._pump, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _poll(self):
        pynvml, h, reasons = self.nvml
        while not self.stop_flag:
            try:
                self.samples.append((time.perf_counter(), float(pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM)), int(reasons(h))))
            except Exception:
                pass
            time.sleep(0.002)

    def _pump(self):
        for ln in self.proc.stdout:
            self.lines.append((time.perf_counter(), ln))

    def begin(self):
        self.t0 = time.perf_counter()

    def end(self):
        self.t1 = time.perf_counter()

    def stop(self):
        if self.nvml:
            self.stop_flag = True
            self.t.join(timeout=1)
            inside = [x for x in self.samples if self.t0 is None or (self.t0 <= x[0] <= (self.t1 or x[0]))]
            mask = 0
            for x in inside:
                mask |= x[2]
            return {"sm_mhz": statistics.median([x[1] for x in inside]) if inside else None, "sm_max_mhz": self.mx,
                    "reasons": sorted(name for bit, name in self.REASONS if mask & bit), "samples": len(inside), "source": "nvml, 2 ms period"}
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvml and nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            pass
        sm, mx, reasons = [], None, set()
        for ts, ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 8:
                continue
            try:
                sm.append(float(f[1])); mx = float(f[2])
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm), "source": "nvidia-smi -lms 100"}


DUMP_LIMIT = 64 << 20


def dump_outputs(out_dir, n_matched, records=None):
    """What a caller of the timed path receives from its last step, as float64 .npy files (byte offsets up to 2^53 are exact):
    n_matched.npy = [matching records], records.npy = their ordered (begin, end) rows.  A list larger than DUMP_LIMIT is cut to
    a fixed sample of rows (seed 0, kept in order), records_rows.npy says which.  The corpus, and so the answer, depends only
    on the arguments and AGB_BENCH_GIB: two builds can be compared file by file."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "n_matched.npy"), np.array([n_matched], dtype=np.float64))
    if records is None:
        return
    if records.nbytes > DUMP_LIMIT - (1 << 20):
        keep = (DUMP_LIMIT - (1 << 20)) // (records.shape[1] * 8 + 8)
        rows = np.sort(np.random.default_rng(0).choice(records.shape[0], keep, replace=False))
        records = records[rows]
        np.save(os.path.join(out_dir, "records_rows.npy"), rows.astype(np.float64))
    np.save(os.path.join(out_dir, "records.npy"), records.astype(np.float64))


# ----------------------------------------------------------------------------------------------------
def run_reference(args):
    """The reference's own CPU implementation of the path, all host threads: one unmodified `agrep -c -n -2`
    process per core, each over its own record-aligned shard of the same synthetic corpus (the program is
    single-threaded by construction, SURVEY 5).  -n forces the asearch() automaton (SURVEY 8c)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    import agrep_b200 as ag
    hc = host_cores()
    cores = hc["usable"]
    kind = "reference" if os.path.exists(REF_BIN) else "port"
    shard = (256 << 20) // PAGE * PAGE      # large enough that process start-up is noise next to the scan
    base = "/dev/shm" if os.path.isdir("/dev/shm") and shutil.disk_usage("/dev/shm").free > cores * shard * 1.2 else tempfile.gettempdir()
    tmp = tempfile.mkdtemp(prefix="agb_ref_", dir=base)
    try:
        files = [os.path.join(tmp, "shard%03d.txt" % i) for i in range(cores)]

        def gen(i):
            data = ag.corpus_host(shard, first_page=i * (shard // PAGE), needle=PATTERN, needle_every=NEEDLE_EVERY, needle_maxedits=3)
            with open(files[i], "wb") as f:
                f.write(data)
        th = [threading.Thread(target=gen, args=(i,)) for i in range(cores)]
        [t.start() for t in th]; [t.join() for t in th]
        total = shard * cores

        def step():
            if kind == "reference":
                ps = [subprocess.Popen([REF_BIN, "-V0", "-c", "-n", "-%d" % K, PATTERN, f], stdout=subprocess.PIPE,
                                       stderr=subprocess.DEVNULL) for f in files]
                return sum(int((p.communicate()[0] or b"0").split()[0]) if p.wait() is not None else 0 for p in ps)
            sys.path.insert(0, os.path.join(ROOT, "tests"))
            import _oracle
            a = _oracle.compile(PATTERN, k=K, linenum=1)
            res = [0] * cores

            def one(i):
                res[i] = _oracle.scan(a, open(files[i], "rb").read(), want_records=False)[0]
            th = [threading.Thread(target=one, args=(i,)) for i in range(cores)]
            [t.start() for t in th]; [t.join() for t in th]
            return sum(res)
        for _ in range(args.warmup):
            matched = step()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            matched = step()
        dt = (time.perf_counter() - t0) / max(1, args.steps)
        val = total / dt / 1e9
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, matched)
        sample = ("%d shards x %d MiB = %.1f GiB of the same synthetic corpus per step (a bounded sample of the %.0f GiB workload; GB/s is "
                  "size-normalised), one `agrep -V0 -c -n -%d` process per usable host core" % (cores, shard >> 20, total / (1 << 30), TOTAL_GIB, K))
        print(json.dumps({
            "impl": "reference", "metric": "text_scan_throughput", "value": val, "unit": "GB/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt * 1e3, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "u32 bitwise", "data": "synthetic",
            "config": workload_config(args.gpus), "matches_per_step": matched, "scanned_bytes_per_step": total, "host_cores": hc,
            "cpu_baseline": {"value": val, "unit": "GB/s", "cores": cores, "kind": kind, "sample": sample},
            "e2e": {"value": val, "unit": "GB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))
    finally:
        shutil.rmtree(tmp, ignore_errors=True)
    return 0


def workload_config(n_gpus):
    return {"workload": "agrep -%d '%s' over %.0f GiB synthetic newline-delimited ASCII (BASELINE.json configs[1]%s)"
                        % (K, PATTERN, TOTAL_GIB, "" if n_gpus == 1 else ", sharded as configs[4]"),
            "pattern": PATTERN, "k": K, "records": "newline", "corpus_gib": TOTAL_GIB,
            "parallelism": "1 GPU" if n_gpus == 1 else ("%d byte-range shards cut inside records (512-byte multiples), cut rule on the device, "
                                                           "ncclAllGather of 256-byte headers + match lists inside libagrepb200.so (agb_scan_sharded)" % n_gpus),
            "l2": "input per GPU is far larger than the 126 MB L2; no flush needed",
            "output": "count + ordered (begin,end) list of matching records"}


# ----------------------------------------------------------------------------------------------------
def cpu_baseline(ag, corpus_t, n_local):
    """rank 0, N=1: the unmodified reference binary on a bounded sample of the SAME corpus (one core: the
    program is single-threaded), `-n` forcing the asearch() automaton whose semantics we reproduce."""
    import torch
    nbytes = min(CPU_SAMPLE_MIB << 20, n_local) // PAGE * PAGE
    base = "/dev/shm" if os.path.isdir("/dev/shm") and shutil.disk_usage("/dev/shm").free > nbytes * 1.5 else tempfile.gettempdir()
    path = os.path.join(base, "agb_cpu_sample_%d.txt" % os.getpid())
    try:
        with open(path, "wb") as f:
            step = 256 << 20
            for off in range(0, nbytes, step):
                f.write(corpus_t[off:min(off + step, nbytes)].cpu().numpy().tobytes())
        best, count = None, None
        if os.path.exists(REF_BIN):
            kind = "reference"
            for _ in range(2):
                t0 = time.perf_counter()
                out = subprocess.run([REF_BIN, "-V0", "-c", "-n", "-%d" % K, PATTERN, path], capture_output=True).stdout
                dt = time.perf_counter() - t0
                best = dt if best is None else min(best, dt)
                count = int(out.split()[0]) if out.split() else 0
        else:
            kind = "port"
            sys.path.insert(0, os.path.join(ROOT, "tests"))
            import _oracle
            a = _oracle.compile(PATTERN, k=K, linenum=1)
            data = open(path, "rb").read()
            t0 = time.perf_counter()
            count = _oracle.scan(a, data, want_records=False)[0]
            best = time.perf_counter() - t0
        ordinals = None
        if kind == "reference":
            # the matching lines themselves, not just how many: -n prints j - 1 in front of every record (agrep.c:3878)
            import re
            out = subprocess.run([REF_BIN, "-V0", "-n", "-%d" % K, PATTERN, path], capture_output=True).stdout
            ordinals = [int(m.group(1)) for m in re.finditer(rb"^(\d+): ", out, re.M)]
        hc = host_cores()
        res = {"value": nbytes / best / 1e9, "unit": "GB/s", "cores": 1, "kind": kind,
               "sample": "first %d MiB of the benchmark corpus, `agrep -V0 -c -n -%d '%s'`, page-cached, best of 2" % (nbytes >> 20, K, PATTERN),
               "matched_in_sample": count, "host_cores": hc}
        if kind == "reference" and hc["usable"] > 1:
            v, m, b = all_core_reference(ag, hc["usable"], 128)
            res["all_cores"] = {"value": v, "unit": "GB/s", "cores": hc["usable"], "kind": kind,
                                "sample": "%d reference processes at once, %d MiB of the same corpus each, best of 2" % (hc["usable"], 128)}
        return res, nbytes, count, ordinals
    finally:
        try:
            os.unlink(path)
        except OSError:
            pass


def secondary_workloads(ag, torch, corpus, n_local, stream, peak):
    """The other BASELINE.json configs at the full corpus size, measured on the side (not the headline): device scans,
    best of 3, CUDA-event stage times from the library, each with its own roofline fraction (corpus bytes / time against
    the measured HBM figure).  configs[0] at scale: 'the' (sgrep/bm semantics, one line in three matches); configs[3]:
    -i -B best match; the headline query with -n; configs[2] last, because its paragraph corpus overwrites the text:
    32-char pattern, -3 -w, paragraph records."""
    out = []

    def roof(n, ms):
        return {"bound": "hbm", "achieved": n / ms / 1e6, "peak": peak, "unit": "GB/s", "frac": n / ms / 1e6 / peak}

    def timed(pat, data_ptr, n, **kw):
        p = ag.Pattern(pat, **kw)
        p.scan_device(data_ptr, n, stream=stream)
        best = None
        for _ in range(3):
            r = p.scan_device(data_ptr, n, stream=stream)
            t = r.ms_front + r.ms_records
            if best is None or t < best[0]:
                best = (t, r)
        t, r = best
        d = p.desc
        return {"pattern": pat, "options": {k: (v if isinstance(v, (int, str)) else int(v)) for k, v in kw.items()},
                "bytes": n, "ms": t, "gb_s": n / t / 1e6, "ms_stage1": r.ms_front, "matched": int(r.n_matched),
                "plan": "anchors" if d.plan == 1 else "all", "n_anchors": int(d.n_anchors), "roofline": roof(n, t)}
    try:
        o = timed("the", corpus.data_ptr(), n_local)
        o["config"] = "configs[0] at scale: agrep -c the (sgrep/bm semantics)"
        out.append(o)
        # the headline query with -n: the ordered list plus every record's ordinal (j), counted on the device
        cap = 1 << 22
        rec = torch.empty((cap, 4), dtype=torch.int64, device=corpus.device)
        pn = ag.Pattern(PATTERN, k=K, linenum=True)
        pn.scan_device(corpus.data_ptr(), n_local, stream=stream, d_records=rec.data_ptr(), capacity=cap, ordinals=True)
        bestn = None
        for _ in range(3):
            r = pn.scan_device(corpus.data_ptr(), n_local, stream=stream, d_records=rec.data_ptr(), capacity=cap, ordinals=True)
            t = r.ms_front + r.ms_records
            if bestn is None or t < bestn[0]:
                bestn = (t, r)
        t, r = bestn
        nr = int(r.n_records)
        ords = rec[:nr, 2]
        out.append({"config": "the headline query with -n (AGB_WANT_RECORDS | AGB_WANT_ORDINALS): list + ordinals (stage 1 also counts the delimiters of every 512-byte block)",
                    "pattern": PATTERN, "bytes": n_local, "ms": t, "gb_s": n_local / t / 1e6, "matched": int(r.n_matched),
                    "n_closes": int(r.n_closes), "ordinals_increasing": bool(nr < 2 or bool((ords[1:] > ords[:-1]).all().item())),
                    "roofline": roof(n_local, t)})
        # configs[3]: the -B sweep as ONE pass at the largest level: best level, its count and its ordered record list
        bestb = None
        for _ in range(3):
            t0 = time.perf_counter()
            best, res = ag.bestmatch_device("Becuase Each Just Th", corpus.data_ptr(), n_local, stream=stream, nocase=1,
                                            d_records=rec.data_ptr(), capacity=cap)
            torch.cuda.synchronize()
            dt = (time.perf_counter() - t0) * 1e3
            if bestb is None or dt < bestb[0]:
                bestb = (dt, best, res)
        dt, best, res = bestb
        out.append({"config": "configs[3]: -i -B best match (agrep.c:3582-3728), 20-char mixed-case pattern: best level + its records",
                    "pattern": "Becuase Each Just Th", "bytes": n_local, "ms": dt, "gb_s": n_local / dt / 1e6,
                    "best_k": int(best), "matched": int(res.n_matched), "records_returned": int(res.n_records),
                    "timing": "wall clock around the call (it may run more than one device pass)", "roofline": roof(n_local, dt)})
        del rec
        # configs[2] on the whole corpus size: the paragraph variant overwrites the text (nothing needs it after this)
        p32 = "business give group toward young"
        ag.corpus_device(corpus.data_ptr(), n_local, stream=stream, paragraphs=True, needle=p32, needle_every=NEEDLE_EVERY, needle_maxedits=4)
        torch.cuda.synchronize()
        o = timed(p32, corpus.data_ptr(), n_local, k=3, wordbound=True, linenum=True, delim="$$")
        o["config"] = "configs[2]: 32-char pattern, -3 -w -d '$$', paragraph records (M = 37: 64-bit rows; the reference refuses it)"
        out.append(o)
    except Exception as e:      # a secondary measurement must never take the headline down
        out.append({"error": repr(e)})
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step returned to DIR/*.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else max(args.warmup, 1)
    if args.impl == "reference":
        return run_reference(args)

    import torch
    import agrep_b200 as ag
    from agrep_b200 import _lib, shard
    L = _lib.lib()                      # raises if the CUDA library is missing: there is no fallback
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback)")
    torch.cuda.set_device(local)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    dev = torch.device("cuda", local)

    total = int(TOTAL_GIB * (1 << 30)) // (PAGE * world) * (PAGE * world)
    per = total // world
    # The shards: cut at multiples of 512 bytes that are NOT record boundaries (the corpus is made of independent 4 KiB
    # pages; a cut 1536 bytes into a page falls inside a line), so that the device-side cut rule of the sharded scan
    # (a record belongs to the shard that holds the last byte of the delimiter that opened it) is what decides.
    SKEW = 1536
    cut = lambda r: 0 if r == 0 else (total if r == world else r * per + SKEW)
    off, n_local = cut(rank), cut(rank + 1) - cut(rank)
    HL, HR = _lib.HALO_LEFT, _lib.HALO_RIGHT
    lead = off - rank * per                                     # bytes of the page-aligned range in front of the shard (0 or SKEW)
    pages = (lead + n_local + PAGE - 1) // PAGE
    buf = torch.empty(max(lead, HL) - lead + pages * PAGE + HR + 4096, dtype=torch.uint8, device=dev)
    gen0 = max(lead, HL) - lead                                  # where the generated pages start inside buf
    stream = torch.cuda.current_stream().cuda_stream
    ag.corpus_device(buf.data_ptr() + gen0, pages * PAGE, stream=stream, first_page=rank * (per // PAGE), needle=PATTERN,
                     needle_every=NEEDLE_EVERY, needle_maxedits=3)
    buf[gen0 + lead + n_local:].zero_()
    torch.cuda.synchronize()
    shard_ptr = buf.data_ptr() + gen0 + lead                     # 16-byte aligned: torch allocations are, gen0 + lead is a multiple of 512
    assert shard_ptr % 16 == 0
    corpus = buf[gen0 + lead:]                                   # the shard as a tensor (N = 1: the whole corpus)

    pat = ag.Pattern(PATTERN, k=K)
    CAP = 1 << 22
    recs = torch.zeros((CAP, 4), dtype=torch.int64, device=dev)       # agb_record = 4 x int64 (level+pad packed in the last)
    comm = None
    if world > 1:
        comm = shard.Comm(dist)                                  # NCCL communicator inside libagrepb200.so (the unique id travels over torch.distributed)
        comm.halo(shard_ptr, n_local, stream=stream)             # once per text: 64.5 KiB from each neighbour

    def step():
        if world == 1:
            res = pat.scan_device(shard_ptr, n_local, stream=stream, d_records=recs.data_ptr(), capacity=CAP)
        else:
            # every rank scans its shard (cut rule on the device), then ncclAllGather of the headers and of the match lists:
            # the ordered list of the whole corpus ends up in recs on every rank (agb_scan_sharded, csrc/shard.cu)
            res = comm.scan(pat, shard_ptr, n_local, off, d_records=recs.data_ptr(), capacity=CAP, stream=stream)
        if res.truncated:
            raise SystemExit("the record list did not fit")
        return res, int(res.n_records)

    if world > 1:
        # the sharded answer against the same corpus cut at page boundaries (where no record is cut): same total
        r0 = pat.scan_device(buf.data_ptr() + gen0, per, stream=stream)
        tt = torch.tensor([int(r0.n_matched)], dtype=torch.int64, device=dev)
        dist.all_reduce(tt)
        rs, _ = step()
        if int(tt.item()) != int(rs.n_matched):
            raise SystemExit("PARITY FAILURE: sharded scan counted %d records, the page-aligned scans %d" % (rs.n_matched, int(tt.item())))

    for _ in range(args.warmup):
        res, gathered = step()
    launches0 = L.agb_kernel_launches()
    try:
        uuid = "GPU-" + str(torch.cuda.get_device_properties(local).uuid)
    except Exception:
        uuid = None
    sampler = ClockSampler(local, uuid)
    if rank == 0:
        sampler.start()
    if dist:
        dist.barrier()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    front_ms, rec_ms = [], []
    sampler.begin()
    e0.record()
    for _ in range(args.steps):
        res, gathered = step()
        front_ms.append(res.ms_front); rec_ms.append(res.ms_records)
    e1.record()
    torch.cuda.synchronize()
    sampler.end()
    if dist:
        dist.barrier()
    ms_total = e0.elapsed_time(e1)
    t = torch.tensor([ms_total], dtype=torch.float64, device=dev)
    if dist:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_step = float(t.item()) / args.steps
    launches = L.agb_kernel_launches() - launches0
    clocks = sampler.stop() if rank == 0 else None
    matched_total = gathered
    if args.dump_outputs and rank == 0:
        # before anything else writes into recs; with N > 1 the gathered list of the whole corpus is on every rank
        dump_outputs(args.dump_outputs, int(res.n_matched), recs[:gathered, :2].cpu().numpy())

    # ---- end to end through the host-buffer entry point (pinned host memory, H2D + result D2H inside the timing)
    n_e2e = min(int(E2E_GIB * (1 << 30)), n_local - HR) // PAGE * PAGE
    host = torch.empty(n_e2e, dtype=torch.uint8, pin_memory=True)
    host.copy_(corpus[:n_e2e])
    torch.cuda.synchronize()
    E2E_CAP = max(1 << 20, n_e2e // 4096)       # (the 4 GiB slice holds about 96 k matching records)
    hrec = (_lib.Record * E2E_CAP)()
    hres = _lib.Result()

    def e2e_step():
        rc = L.agb_scan_host(pat._h, ctypes.c_void_p(host.data_ptr()), n_e2e, _lib.WANT_RECORDS, hrec, E2E_CAP, ctypes.byref(hres))
        if rc != 0:
            raise RuntimeError(L.agb_last_error().decode())
        if hres.truncated:
            raise RuntimeError("e2e: the record list did not fit (%d matches)" % hres.n_matched)
        return hres.n_records
    for _ in range(2):
        e2e_step()
    if dist:
        dist.barrier()
    t0 = time.perf_counter()
    E2E_STEPS = 3
    for _ in range(E2E_STEPS):
        nrec = e2e_step()
    dt = (time.perf_counter() - t0) / E2E_STEPS
    t = torch.tensor([dt], dtype=torch.float64, device=dev)
    if dist:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    e2e_val = n_e2e * world / float(t.item()) / 1e9

    # ---- the same through a file descriptor (agb_scan_fd: what replaces the fill_buf()/read(2) loop, bitap.c:450-477):
    # a page-cached temporary file -> pread(2) by 4 threads into the pinned ring -> H2D -> scan -> list back
    e2e_fd = None
    if rank == 0 and world == 1:
        import tempfile
        n_fd = min(n_e2e, 2 << 30)
        try:
            with tempfile.NamedTemporaryFile(prefix="agb_bench_", dir=os.environ.get("TMPDIR", "/tmp")) as tf:
                view = host[:n_fd].numpy()
                tf.write(memoryview(view)); tf.flush()
                fd = os.open(tf.name, os.O_RDONLY)
                try:
                    ts = []
                    for it in range(3):
                        os.lseek(fd, 0, os.SEEK_SET)
                        t0 = time.perf_counter()
                        rc = L.agb_scan_fd(pat._h, fd, _lib.WANT_RECORDS, hrec, E2E_CAP, ctypes.byref(hres))
                        ts.append(time.perf_counter() - t0)
                        if rc != 0:
                            raise RuntimeError(L.agb_last_error().decode())
                    e2e_fd = {"value": n_fd / min(ts[1:]) / 1e9, "unit": "GB/s", "bytes": n_fd, "records": int(hres.n_records),
                              "what": "agb_scan_fd() on a page-cached temporary file (first %.1f GiB of the corpus): pread(2) by 4 host threads into "
                                      "the pinned ring, H2D and stage 1 overlapped, list read back; best of 2 after a warm-up" % (n_fd / (1 << 30))}
                finally:
                    os.close(fd)
        except (OSError, RuntimeError) as e:
            e2e_fd = {"value": None, "error": str(e)[:200]}

    cpu = None
    if rank == 0 and world == 1:
        cpu, nsample, cpu_count, cpu_ordinals = cpu_baseline(ag, corpus, n_local)
        # the same sample through the CUDA path must agree with the reference binary, bit for bit: the count and which
        # lines they are (the ordinals the device computes against the reference's -n prefixes)
        pn = ag.Pattern(PATTERN, k=K, linenum=True)
        r = pn.scan_device(corpus.data_ptr(), nsample, stream=stream, d_records=recs.data_ptr(), capacity=CAP, ordinals=True)
        cpu["gpu_matched_in_sample"] = int(r.n_matched)
        if cpu_count is not None and int(r.n_matched) != cpu_count:
            raise SystemExit("PARITY FAILURE: reference counted %d records in the sample, CUDA path %d" % (cpu_count, r.n_matched))
        if cpu_ordinals is not None:
            got = (recs[:int(r.n_records), 2] - 1).cpu().tolist()
            if got != cpu_ordinals:
                raise SystemExit("PARITY FAILURE: the matching lines of the sample differ from the reference's (-n ordinals)")
            cpu["ordinals_checked"] = len(got)

    secondary = None
    if rank == 0 and world == 1 and os.environ.get("AGB_BENCH_SECONDARY", "1") != "0":
        secondary = secondary_workloads(ag, torch, corpus, n_local, stream, peaks()[0])

    if rank == 0:
        peak, peak_src = peaks()
        fm = statistics.mean(front_ms)
        achieved = n_local / (fm * 1e-3) / 1e9
        traffic = None
        try:
            traffic = json.load(open(os.path.join(ROOT, "profiles", "k_front_traffic.json")))
        except Exception:
            pass
        value = total / (ms_step * 1e-3) / 1e9
        step_traffic = None
        try:
            step_traffic = json.load(open(os.path.join(ROOT, "profiles", "step_traffic.json")))
        except Exception:
            pass
        roofline_step = {"bound": "hbm", "what": "the whole step (stage 1 + stage 1.5 + record stage + ordered list), per GPU",
                         "achieved": n_local / (ms_step * 1e-3) / 1e9, "peak": peak, "unit": "GB/s",
                         "frac": n_local / (ms_step * 1e-3) / 1e9 / peak, "algorithmic_bytes_per_step": n_local,
                         "traffic": (step_traffic or {}).get("dram_bytes_per_step"),
                         "traffic_note": (step_traffic or {}).get("note", "no ncu capture of a whole step yet")}
        out = {
            "metric": "text_scan_throughput", "value": value, "unit": "GB/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "u32 bitwise", "data": "synthetic", "config": workload_config(world),
            "matching_records": matched_total, "matching_records_per_s": matched_total / (ms_step * 1e-3),
            "roofline": {"bound": "hbm", "kernel": "k_front (stage 1, anchor filter)", "achieved": achieved, "peak": peak,
                         "unit": "GB/s", "frac": achieved / peak, "peak_source": peak_src,
                         "algorithmic_bytes_per_launch": n_local, "ms_per_launch": fm,
                         "stage2_ms_per_step": statistics.mean(rec_ms),
                         "traffic": (traffic or {}).get("dram_bytes_per_launch") if traffic else None,
                         "traffic_note": (traffic or {}).get("note") if traffic else "no ncu --set full capture yet"},
            "roofline_step": roofline_step,
            "e2e": {"value": e2e_val, "unit": "GB/s", "h2d_bytes_per_step": n_e2e, "d2h_bytes_per_step": 128 + 32 * int(nrec),
                    "what": "agb_scan_host() on a pinned host buffer holding the first %.1f GiB of each rank's shard; "
                            "64 MiB H2D slices overlapped with stage 1; wall clock incl. result read-back" % (n_e2e / (1 << 30))},
            "gpu_launches": int(launches), "clocks": clocks,
        }
        if e2e_fd:
            out["e2e"]["fd"] = e2e_fd
        if cpu:
            out["cpu_baseline"] = cpu
        if secondary:
            out["secondary_workloads"] = secondary
        print(json.dumps(out))
    if dist:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
