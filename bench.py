#!/usr/bin/env python
"""bench.py -- audio samples/sec of the VITS2 inference path (BASELINE.json metric) on N B200s.

One "step" = one pass of the hot path (SynthesizerTrn.infer) over one batch: BASELINE.json configs[1], a single
128-phoneme utterance (tokens = randint(0,62,(128,), seed 0), sid 2, scales [0.8, 1.0, 0.8], fp32), synthetic seeded
weights of the mb_istft_vits2_multi architecture (no checkpoint exists on the box).  N > 1: one process per GPU,
each rank synthesises its own copy of the workload (utterances share nothing -> weak scaling, no collective on the
utterance path; the packed weights are broadcast once from rank 0 over NCCL at init).

  value    : samples/s with inputs resident in HBM (device-pointer C-ABI), CUDA-event timed per step, L2 flushed
             between steps, max over ranks.
  e2e      : same metric through the reference-facing call (VitsSession.run with HOST numpy feeds, host->device and
             device->host copies inside the timed region, wall clock bracketed by synchronisation).
  e2e_cold : the same call on utterances that were NEVER seen before (other tokens, other lengths in 100..128, engine-drawn
             noise with a fresh seed per call) after the length buckets have been warmed by OTHER utterances -- what a
             stream of distinct texts gets (CUDA graphs are keyed on length buckets, not on lengths).
  extra    : N = 1 only -- BASELINE configs[2] (64 utterances in one call) with its own roofline, configs[4] (2000-phoneme
             streaming: time to first chunk / total) and the fp32-exact mode (precision 0) of the headline workload.
  --impl reference : the CPU path (oracle restatement of the reference's PyTorch graph) on the host cores.
  --dump-outputs DIR : after the timed steps, writes what the last timed step returned to its caller (DIR/wav.npy float32
             [1, frames * 256], DIR/y_lengths.npy float64), so that two builds can be compared output for output on the
             same seeded inputs and weights.
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

SR = 22050
METRIC = "audio samples/sec @22.05kHz, 128-phoneme utterance"
FRAMES_OF_WORKLOAD = 162        # data dependent; asserted at run time (seeded inputs and weights)


def workload(cfg):
    import torch
    g = torch.Generator().manual_seed(0)
    tok = torch.randint(0, cfg["n_vocab"], (1, 128), generator=g).numpy().astype(np.int64)
    eps_dp = torch.randn(1, 2, 128, generator=g).numpy()
    eps_z = torch.randn(1, cfg["inter_channels"], 24 * 128 + 8, generator=g).numpy()
    return dict(tok=tok, lens=np.array([128], np.int64), sid=np.array([2], np.int64),
                scales=np.array([0.8, 1.0, 0.8], np.float32), eps_dp=eps_dp, eps_z=eps_z)


def config_dict():
    """Identical in both arms (--impl ours / reference): names the workload, nothing else."""
    return {"workload": "BASELINE configs[1]: one 128-phoneme utterance (randint seed 0), sid=2, scales [0.8,1.0,0.8], "
                        "mb_istft_vits2_multi architecture, seeded synthetic weights", "batch_per_gpu": 1, "phonemes": 128,
            "frames": FRAMES_OF_WORKLOAD, "samples_per_step": FRAMES_OF_WORKLOAD * 256,
            "parallelism": "replicas (one utterance stream per GPU, weights broadcast once)", "l2": "flushed between timed steps"}


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm=d["hbm_gbs"], bf16=d["bf16_tflops"], bf16_sustained=d.get("bf16_tflops_sustained", d["bf16_tflops"]), src="measured")
    return dict(hbm=6650.0, bf16=1590.0, bf16_sustained=1400.0, src="fallback")


class ClockSampler(threading.Thread):
    """SM clock and throttle reasons sampled DURING the timed region (NVML, 5 ms period; nvidia-smi as a fallback)."""
    Q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.rows, self.stop_flag = index, [], False
        self.nvml = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nvml = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
        except Exception:
            self.nvml = None

    def run(self):
        while not self.stop_flag:
            if self.nvml is not None:
                try:
                    n = self.nvml
                    sm = n.nvmlDeviceGetClockInfo(self.h, n.NVML_CLOCK_SM)
                    mx = n.nvmlDeviceGetMaxClockInfo(self.h, n.NVML_CLOCK_SM)
                    try:
                        r = n.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                    except Exception:
                        r = n.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                    bits = {"hw_slowdown": 0x8, "sw_power_cap": 0x4, "sw_thermal_slowdown": 0x20, "hw_thermal_slowdown": 0x40}
                    self.rows.append((float(sm), float(mx), [k for k, b in bits.items() if r & b]))
                except Exception:
                    self.nvml = None
                time.sleep(0.005)
                continue
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    c = [x.strip() for x in out.split(",")]
                    names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
                    self.rows.append((float(c[0]), float(c[1]), [n for i, n in enumerate(names) if c[2 + i].lower().startswith("active")]))
            except Exception:
                pass
            time.sleep(0.05)

    def summary(self):
        self.stop_flag = True
        self.join(timeout=6)
        if not self.rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
        sm = sorted(r[0] for r in self.rows)
        reasons = sorted({x for r in self.rows for x in r[2]})
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": self.rows[0][1], "reasons": reasons, "samples": len(self.rows),
                "source": "nvml" if self.nvml is not None else "nvidia-smi"}


def host_cores():
    """Cores this process may actually use (affinity mask and cgroup quota), not the machine's core count."""
    try:
        n = len(os.sched_getaffinity(0))
    except Exception:
        n = os.cpu_count() or 1
    try:
        q, p = open("/sys/fs/cgroup/cpu.max").read().split()
        if q != "max":
            n = max(1, min(n, int(float(q) / float(p) + 0.5)))
    except Exception:
        pass
    return n


def pin_to_gpu_numa(index):
    """Bind this rank to the host cores next to its GPU (NVML's ideal CPU affinity): the per-utterance path has two graph
    launches and one synchronisation on the host side, and a rank running on the far socket is the straggler of a
    max-over-ranks timing.  Returns the number of cores bound, or None."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(index)
        ncpu = os.cpu_count() or 1
        words = (ncpu + 63) // 64
        mask = pynvml.nvmlDeviceGetCpuAffinity(h, words)
        cpus = {w * 64 + b for w, m in enumerate(mask) for b in range(64) if (int(m) >> b) & 1}
        cpus &= set(os.sched_getaffinity(0))
        if cpus:
            os.sched_setaffinity(0, cpus)
            return len(cpus)
    except Exception:
        pass
    return None


def ncu_traffic(family):
    """dram read+write bytes per launch of the dominant kernel from this round's committed `ncu --set full` capture
    (profiles/r2_conv_tc_traffic.json, made by the command in profiles/README.md), or None."""
    for name in ("r2_conv_tc_traffic.json", "r1_conv_tc_traffic.json"):
        path = os.path.join(ROOT, "profiles", name)
        if family == "tc" and os.path.exists(path):
            try:
                with open(path) as f:
                    return float(json.load(f)["dram_bytes_per_launch_mean"]), "profiles/" + name
            except Exception:
                pass
    return None, None


def pick_threads(cfg, w, cores):
    """PyTorch's intra-op pool is at its best well below the core count on these tiny convs (128 threads ran 300x
    slower than 8 on the B200 host): probe a short utterance at a few thread counts and keep the fastest, so that
    the CPU arm is the reference at ITS best, not a strawman."""
    import torch
    from oracle import vits_oracle as vo
    g = torch.Generator().manual_seed(1)
    T = 24
    tok = torch.randint(0, cfg["n_vocab"], (1, T), generator=g)
    e1, e2 = torch.randn(1, 2, T, generator=g), torch.randn(1, cfg["inter_channels"], 24 * T, generator=g)
    cands = sorted({c for c in (cores, 64, 32, 16, 8, 4) if 1 <= c <= cores}, reverse=True)
    best, best_t = cands[-1], float("inf")
    for c in cands[::-1]:                      # small counts first: a pathological large count is cut short
        torch.set_num_threads(c)
        ts = []
        with torch.no_grad():
            for _ in range(3):
                t0 = time.perf_counter()
                vo.infer(w, cfg, tok, torch.tensor([T]), torch.tensor([2]), (0.8, 1.0, 0.8), e1, e2)
                ts.append(time.perf_counter() - t0)
                if ts[-1] > 3.0:
                    break
        t = min(ts)
        if t < best_t:
            best, best_t = c, t
        if t > 4 * best_t:
            break
    return best


def cpu_reference_run(cfg, wl, steps, warmup, threads=None):
    """Times the oracle port of the reference's CPU graph (the only place bench.py executes oracle/)."""
    import torch
    from oracle import vits_oracle as vo
    from vosk_tts_b200 import synthetic, weights
    w = weights.fold_weight_norm(synthetic.make_random_checkpoint(cfg, 1234))
    cores = threads or pick_threads(cfg, w, host_cores())
    torch.set_num_threads(cores)
    tok, lens, sid = torch.as_tensor(wl["tok"]), torch.as_tensor(wl["lens"]), torch.as_tensor(wl["sid"])
    eps_dp, eps_z = torch.as_tensor(wl["eps_dp"]), torch.as_tensor(wl["eps_z"])
    times, n = [], 0
    with torch.no_grad():
        for i in range(warmup + steps):
            t0 = time.perf_counter()
            o = vo.infer(w, cfg, tok, lens, sid, wl["scales"], eps_dp, eps_z)
            wav = o["o"][0, 0].numpy()
            pcm = np.clip(wav * 32767.0, -32767.0, 32767.0).astype("int16")   # as vosk_tts/synth.py:127-130
            dt = time.perf_counter() - t0
            if i >= warmup:
                times.append(dt)
            n = pcm.shape[-1]
    return n, times, cores


def cpu_worker_main(threads, steps):
    """`bench.py --cpu-worker T S`: one process of the all-cores CPU throughput figure (prints samples and seconds)."""
    from vosk_tts_b200 import config as C
    cfg = C.DEFAULT_CONFIG
    n, times, _ = cpu_reference_run(cfg, workload(cfg), steps, 1, threads=threads)
    print(json.dumps({"samples": n, "steps": len(times), "seconds": sum(times)}))


def cpu_throughput_all_cores(threads, steps=3):
    """The CPU path at its best THROUGHPUT: k = host_cores // threads independent processes of `threads` intra-op threads
    each, all running the headline utterance at the same time (machine vs machine, next to the single-stream latency)."""
    cores = host_cores()
    k = max(1, min(cores // max(threads, 1), 16))
    t0 = time.perf_counter()
    procs = [subprocess.Popen([sys.executable, os.path.abspath(__file__), "--cpu-worker", str(threads), str(steps)],
                              stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True) for _ in range(k)]
    res = []
    for p in procs:
        try:
            out, _ = p.communicate(timeout=240)
            res.append(json.loads(out.strip().splitlines()[-1]))
        except Exception:
            p.kill()
    if not res:
        return None
    # every process times its own steps while the others run: aggregate rate = sum of the per-process rates
    rate = sum(r["samples"] * r["steps"] / r["seconds"] for r in res)
    return {"value": rate, "unit": "samples/s", "processes": len(res), "threads_per_process": threads, "host_cores": cores,
            "wall_s": time.perf_counter() - t0}


def extras(cfg, blob, manifest, eng, dev, pk):
    """Secondary BASELINE configs on the same GPU (N = 1 only); each is bounded to a few seconds."""
    import torch
    from vosk_tts_b200.engine import Engine
    out = {}
    est = torch.cuda.ExternalStream(eng.stream(), device=dev)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    # ---- configs[2]: 64 utterances of 64..256 phonemes in ONE call (ragged, packed), engine-drawn noise
    try:
        B = 64
        g = torch.Generator().manual_seed(1)
        lens = torch.randint(64, 257, (B,), generator=g).numpy().astype(np.int64)
        ids = torch.randint(0, cfg["n_vocab"], (B, int(lens.max())), generator=g).numpy().astype(np.int64)
        sid = torch.randint(0, 5, (B,), generator=g).numpy().astype(np.int64)
        d_ids, d_sid = torch.as_tensor(ids, device=dev), torch.as_tensor(sid, device=dev)
        scales = np.array([0.8, 1.0, 0.8], np.float32)
        yl = eng.durations_dev(d_ids.data_ptr(), lens, d_sid.data_ptr(), B, ids.shape[1], scales, 0, seed=7)
        maxf = int(yl.max())
        d_wav = torch.zeros(B, maxf * eng.hop, device=dev)
        eng.synthesize_dev(d_wav.data_ptr(), maxf * eng.hop)

        def step():
            return eng.infer_dev(d_ids.data_ptr(), lens, d_sid.data_ptr(), B, ids.shape[1], scales, d_wav.data_ptr(), maxf * eng.hop, seed=7)
        for _ in range(3):
            step()
        ms = []
        for _ in range(5):
            flush.fill_(1)
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(est)
            yl = step()
            e1.record(est)
            e1.synchronize()
            ms.append(e0.elapsed_time(e1))
        eng.profile(True)
        for _ in range(2):
            step()
        prof = eng.profile_read()
        stage = eng.stage_timings()
        eng.profile(False)
        n = int(yl.sum()) * eng.hop
        t = sum(ms) / len(ms)
        ach = prof["tc_flops"] / (prof["tc_ms"] / 1e3) / 1e12 if prof["tc_ms"] else 0.0
        out["configs2_batch64"] = {"workload": "BASELINE configs[2]: 64 utterances, 64-256 phonemes (seed 1), one call, precision mode 1",
                                   "ms_per_step": t, "samples_per_step": n, "value": n / (t / 1e3), "unit": "samples/s",
                                   "frames": int(yl.sum()), "phonemes": int(lens.sum()), "rtf": (t / 1e3) / (n / SR), "stage_ms_eager": stage,
                                   "roofline": {"kernel": "conv_tc_kernel<128> (machine-filling launches)", "bound": "tensor", "achieved": ach,
                                                "peak": pk["bf16_sustained"], "unit": "TFLOP/s", "frac": ach / pk["bf16_sustained"],
                                                "ms_per_step": prof["tc_ms"] / 2, "launches_per_step": prof["tc_launches"] / 2,
                                                "note": "algorithmic FLOPs; the split-bf16 kernel issues 3 MMAs per MAC (ceiling = peak/3)"}}
        del d_wav
    except Exception as ex:      # noqa: BLE001
        out["configs2_batch64"] = {"error": repr(ex)}
    # ---- configs[4]: one 2000-phoneme utterance, 256-frame chunks with a 24-frame halo (streaming) vs monolithic
    try:
        T = 2000
        ids = np.random.RandomState(9).randint(0, cfg["n_vocab"], size=(1, T)).astype(np.int64)
        res = []
        for rep in range(3):
            t0 = time.perf_counter()
            first, n = None, 0
            for c in eng.synthesize_stream(ids, 2, (0.8, 1.0, 0.8), chunk_frames=256, seed=3):
                if first is None:
                    first = time.perf_counter() - t0
                n += c.size
            tot = time.perf_counter() - t0
            t1 = time.perf_counter()
            eng.infer(ids, [T], [2], (0.8, 1.0, 0.8), seed=3)
            res.append((first, tot, time.perf_counter() - t1, n))
        first, tot, mono, n = min(res)
        out["configs4_longform"] = {"workload": "BASELINE configs[4]: 2000 phonemes, 256-frame chunks, 24-frame halo, host buffers",
                                    "samples": n, "audio_s": n / SR, "time_to_first_chunk_ms": first * 1e3, "streamed_total_ms": tot * 1e3,
                                    "monolithic_ms": min(r[2] for r in res) * 1e3, "rtf_streamed": tot / (n / SR),
                                    "rtf_monolithic": min(r[2] for r in res) / (n / SR)}
    except Exception as ex:      # noqa: BLE001
        out["configs4_longform"] = {"error": repr(ex)}
    return out


def sharded_batch(cfg, eng, dev, rank, world, steps=16):
    """BASELINE configs[3]: 64 utterances per GPU (64-256 phonemes), one global list sharded over the ranks by
    parallel.lpt_shards, every rank synthesises its shard in one batched call per step; no collective on the data path.
    Timed with CUDA events on the engine stream, max over ranks.  Every rank reaches the two collectives at the end
    whatever happened before them (a failure on one rank is reported, not waited for)."""
    import torch
    import torch.distributed as dist
    from vosk_tts_b200 import parallel
    err, mine_ms, n, B = None, 0.0, 0.0, 0
    n_all = 64 * world
    try:
        g = torch.Generator().manual_seed(3)
        lens_all = torch.randint(64, 257, (n_all,), generator=g).numpy().astype(np.int64)
        ids_all = torch.randint(0, cfg["n_vocab"], (n_all, 256), generator=g).numpy().astype(np.int64)
        sid_all = torch.randint(0, 5, (n_all,), generator=g).numpy().astype(np.int64)
        mine = parallel.lpt_shards(lens_all, world)[rank]
        lens, sid = lens_all[mine], sid_all[mine]
        ids = np.ascontiguousarray(ids_all[mine][:, : int(lens.max())])
        B = len(mine)
        d_ids, d_sid = torch.as_tensor(ids, device=dev), torch.as_tensor(sid, device=dev)
        scales = np.array([0.8, 1.0, 0.8], np.float32)
        yl = eng.durations_dev(d_ids.data_ptr(), lens, d_sid.data_ptr(), B, ids.shape[1], scales, 0, seed=11)
        maxf = int(yl.max())
        d_wav = torch.zeros(B, maxf * eng.hop, device=dev)
        eng.synthesize_dev(d_wav.data_ptr(), maxf * eng.hop)
        est = torch.cuda.ExternalStream(eng.stream(), device=dev)
        flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)

        def step():
            return eng.infer_dev(d_ids.data_ptr(), lens, d_sid.data_ptr(), B, ids.shape[1], scales, d_wav.data_ptr(), maxf * eng.hop, seed=11)
        for _ in range(3):
            yl = step()
        ms = []
        for _ in range(steps):
            flush.fill_(1)
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(est)
            yl = step()
            e1.record(est)
            e1.synchronize()
            ms.append(e0.elapsed_time(e1))
        torch.cuda.synchronize()
        mine_ms = float(sum(ms))
        n = float(int(yl.sum()) * eng.hop * steps)
        del d_wav, flush
    except Exception as ex:      # noqa: BLE001
        err = repr(ex)
    t = torch.tensor([mine_ms, -mine_ms if err is None else -1e30, 1.0 if err else 0.0], device=dev, dtype=torch.float64)
    tn = torch.tensor([n], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dist.all_reduce(tn, op=dist.ReduceOp.SUM)
    worst, best, failed = float(t[0]), -float(t[1]), float(t[2]) > 0
    if failed or worst <= 0:
        return {"error": err or "another rank failed"}
    return {"workload": "BASELINE configs[3]: %d utterances (64-256 phonemes, seed 3) sharded %d ways by parallel.lpt_shards, one batched call per "
                        "rank and step, weights from the one NCCL broadcast, no data-path collective" % (n_all, world),
            "steps": steps, "utterances_rank0": B, "value": float(tn[0]) / (worst / 1e3), "unit": "samples/s",
            "ms_per_step_slowest_rank": worst / steps, "ms_per_step_fastest_rank": best / steps, "timed_region_s": worst / 1e3}


def main():
    if len(sys.argv) >= 4 and sys.argv[1] == "--cpu-worker":
        cpu_worker_main(int(sys.argv[2]), int(sys.argv[3]))
        return 0
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--cpu-steps", type=int, default=5)
    ap.add_argument("--precision", type=int, default=1, help="0: fp32 FFMA everywhere; 1: flow+decoder on tcgen05 (split-bf16 x3); 2: encoder too; 3: encoder on tcgen05 with the exact 3-way split")
    ap.add_argument("--no-extras", action="store_true", help="skip the secondary configs (configs[2], configs[4], fp32-exact mode)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the outputs of the last timed step to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3)
    from vosk_tts_b200 import config as C
    cfg = C.DEFAULT_CONFIG
    wl = workload(cfg)
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    conf = config_dict()

    if args.impl == "reference":
        if rank != 0:
            return 0
        n, times, threads = cpu_reference_run(cfg, wl, args.steps, args.warmup)
        assert n == conf["samples_per_step"], (n, conf["samples_per_step"])
        tot = sum(times)
        v = n * len(times) / tot
        thr = cpu_throughput_all_cores(threads, steps=3)
        line = {"impl": "reference", "metric": METRIC, "value": v, "unit": "samples/s", "n_gpus": args.gpus, "steps": len(times),
                "warmup": args.warmup, "ms_per_step": 1e3 * tot / len(times), "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": "fp32", "data": "synthetic", "config": conf,
                "rtf": (tot / len(times)) / (n / SR),
                "cpu_baseline": {"value": v, "unit": "samples/s", "cores": threads, "threads": threads, "host_cores": host_cores(), "kind": "port",
                                 "sample": "%d timed runs of the same 128-phoneme utterance, one stream, PyTorch-CPU restatement of "
                                           "SynthesizerTrn.infer (onnxruntime/model.onnx unavailable) at its fastest intra-op thread count, "
                                           "incl. float->int16" % len(times),
                                 "throughput_all_cores": thr},
                "e2e": {"value": v, "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
        print(json.dumps(line))
        return 0

    import torch
    import torch.distributed as dist
    from vosk_tts_b200 import parallel, synthetic, weights
    from vosk_tts_b200.engine import Engine
    from vosk_tts_b200.session import VitsSession
    torch.cuda.set_device(local)
    pinned = pin_to_gpu_numa(local) if world > 1 else None
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    # ---- weights: packed on rank 0 (only the tensors this precision mode reads), ONE broadcast, engine created from the device blob
    t0 = time.perf_counter()
    blob = manifest = None
    folded = None
    if rank == 0:
        folded = weights.fold_weight_norm(synthetic.make_random_checkpoint(cfg, 1234))
        blob, manifest = weights.pack(folded, cfg, precision=args.precision)
    bcast_ms = 0.0
    if world > 1:
        torch.cuda.synchronize()
        dist.barrier()                          # (communicator setup is not part of the broadcast time)
        torch.cuda.synchronize()
        tb = time.perf_counter()
        tblob, manifest = parallel.broadcast_packed(blob, manifest, src=0, device="cuda:%d" % local)
        torch.cuda.synchronize()
        bcast_ms = (time.perf_counter() - tb) * 1e3
        eng = Engine(cfg, (tblob.data_ptr(), tblob.numel()), manifest, device=local, precision=args.precision)
        nblob = int(tblob.numel())
        del tblob
    else:
        eng = Engine(cfg, blob, manifest, device=local, precision=args.precision)
        nblob = int(blob.size)
    sess = VitsSession.__new__(VitsSession)
    sess.cfg, sess.engine, sess._lock, sess._seed, sess._calls = cfg, eng, threading.Lock(), 0, 0
    sess.last_y_lengths = sess.last_wav_lengths = None
    init_s = time.perf_counter() - t0

    dev = torch.device("cuda", local)
    d_ids = torch.as_tensor(wl["tok"], device=dev)
    d_sid = torch.as_tensor(wl["sid"], device=dev)
    d_eps_dp = torch.as_tensor(wl["eps_dp"], device=dev).contiguous()
    # frames of this workload (data dependent): one probe call
    ylen = eng.durations_dev(d_ids.data_ptr(), wl["lens"], d_sid.data_ptr(), 1, 128, wl["scales"], d_eps_dp.data_ptr())
    Ty = int(ylen[0])
    assert Ty == FRAMES_OF_WORKLOAD, Ty
    hop = eng.hop
    d_eps_z = torch.as_tensor(wl["eps_z"][:, :, :Ty], device=dev).contiguous()
    d_wav = torch.zeros(1, (Ty + 64) * hop, device=dev)
    eng.synthesize_dev(d_wav.data_ptr(), (Ty + 64) * hop, d_eps_z.data_ptr(), Ty)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)     # > 126 MB L2
    estream = torch.cuda.ExternalStream(eng.stream(), device=dev)

    def step_dev():
        yl = eng.infer_dev(d_ids.data_ptr(), wl["lens"], d_sid.data_ptr(), 1, 128, wl["scales"], d_wav.data_ptr(), (Ty + 64) * hop,
                           d_eps_dp.data_ptr(), d_eps_z.data_ptr(), Ty)
        return int(yl[0])

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(args.warmup):
        step_dev()
    sampler = ClockSampler(local) if rank == 0 else None
    if sampler:
        sampler.start()
    barrier()
    launches0 = eng.kernel_launches()
    step_ms = []
    for _ in range(args.steps):
        flush.fill_(1)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(estream)
        last_frames = step_dev()
        e1.record(estream)
        e1.synchronize()
        step_ms.append(e0.elapsed_time(e1))
    barrier()
    if args.dump_outputs and rank == 0:
        os.makedirs(args.dump_outputs, exist_ok=True)
        np.save(os.path.join(args.dump_outputs, "wav.npy"), d_wav[:, : last_frames * hop].cpu().numpy().astype(np.float32))
        np.save(os.path.join(args.dump_outputs, "y_lengths.npy"), np.array([last_frames], np.float64))
    launches = eng.kernel_launches() - launches0
    total_ms = float(sum(step_ms))
    # roofline pass: same steps with every conv launch bracketed by CUDA events on the engine stream (eager launches,
    # so this pass is slower than the timed one; only per-kernel durations are taken from it)
    eng.profile(True)
    prof_ms = []
    for _ in range(args.steps):
        flush.fill_(1)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(estream)
        step_dev()
        e1.record(estream)
        e1.synchronize()
        prof_ms.append(e0.elapsed_time(e1))
    prof = eng.profile_read()
    stage = eng.stage_timings()
    eng.profile(False)
    prof_total_ms = float(sum(prof_ms))
    # ---- e2e through the reference-facing call with host buffers
    feeds = {"input": wl["tok"], "input_lengths": wl["lens"], "scales": wl["scales"], "sid": wl["sid"], "bert": None,
             "phone_duration_extra": None}
    noise = {"dp": wl["eps_dp"], "z": np.ascontiguousarray(wl["eps_z"][:, :, :Ty])}
    for _ in range(3):
        sess.run(None, feeds, noise=noise)
    e2e_t = []
    for _ in range(args.steps):
        flush.fill_(1)
        torch.cuda.synchronize()
        t1 = time.perf_counter()
        audio = sess.run(None, feeds, noise=noise)[0]
        e2e_t.append(time.perf_counter() - t1)
    barrier()
    clocks = sampler.summary() if sampler else None
    e2e_total = float(sum(e2e_t))
    # ---- e2e_cold: utterances never seen before (buckets warmed by OTHER utterances)
    g = torch.Generator().manual_seed(4242 + rank)

    def fresh():
        T = int(torch.randint(100, 129, (1,), generator=g))
        return {"input": torch.randint(0, cfg["n_vocab"], (1, T), generator=g).numpy().astype(np.int64), "input_lengths": np.array([T], np.int64),
                "scales": wl["scales"], "sid": np.array([2], np.int64), "bert": None,
                "phone_duration_extra": None}
    # what a service does at start-up: size the workspace for the largest request it will take (here: <= 128 phonemes, <= 768
    # frames), so that no later call moves a buffer and invalidates the length buckets' CUDA graphs
    reserved_frames = sess.reserve(128, 768)
    r0 = eng.graph_replays()
    first_seen = []
    N_COLD_WARM, N_COLD = 150, 40
    def frame_bucket(n):         # engine.cu::bucket_frm
        return (n + 31) // 32 * 32 if n <= 256 else ((n + 63) // 64 * 64 if n <= 1024 else (n + 127) // 128 * 128)
    seen_buckets = set()
    for i in range(N_COLD_WARM):
        f = fresh()
        t1 = time.perf_counter()
        sess.run(None, f)
        first_seen.append(time.perf_counter() - t1)
        seen_buckets.add(((int(f["input_lengths"][0]) + 15) // 16 * 16, frame_bucket(int(sess.last_y_lengths[0]))))
    n_warm_buckets = len(seen_buckets)
    new_in_timed = []
    cold_t, cold_n = [], 0
    r1 = eng.graph_replays()
    h1, m1 = eng.speculation_stats()
    for _ in range(N_COLD):
        f = fresh()
        flush.fill_(1)
        torch.cuda.synchronize()
        t1 = time.perf_counter()
        a = sess.run(None, f)[0]
        cold_t.append(time.perf_counter() - t1)
        cold_n += int(sess.last_wav_lengths[0])
        key = ((int(f["input_lengths"][0]) + 15) // 16 * 16, frame_bucket(int(sess.last_y_lengths[0])))
        if key not in seen_buckets:
            seen_buckets.add(key)
            new_in_timed.append([key[0], key[1], round(1e3 * cold_t[-1], 2)])
    r2 = eng.graph_replays()
    h2, m2 = eng.speculation_stats()
    barrier()
    sharded = None
    if world > 1 and not args.no_extras:
        sharded = sharded_batch(cfg, eng, dev, rank, world)
    n_samples = Ty * hop
    if world > 1:
        t = torch.tensor([total_ms, e2e_total, float(sum(cold_t))], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        total_ms, e2e_total, cold_total = float(t[0]), float(t[1]), float(t[2])
        tn = torch.tensor([float(cold_n)], device=dev, dtype=torch.float64)
        dist.all_reduce(tn, op=dist.ReduceOp.SUM)
        cold_n_all = float(tn[0])
    else:
        cold_total, cold_n_all = float(sum(cold_t)), float(cold_n)
    if rank == 0:
        pk = peaks()
        value = world * n_samples * args.steps / (total_ms / 1e3)
        e2e_v = world * n_samples * args.steps / e2e_total
        fam = {"ffma": (prof["conv_ms"], prof["conv_flops"], prof["conv_launches"]),
               "tc": (prof.get("tc_ms", 0.0), prof.get("tc_flops", 0.0), prof.get("tc_launches", 0))}
        dom = "tc" if fam["tc"][0] > fam["ffma"][0] else "ffma"
        d_ms, d_fl, d_n = fam[dom]
        ach = d_fl / (d_ms / 1e3) / 1e12 if d_ms > 0 else 0.0
        kname = {"tc": "conv_tc_kernel<64, cluster split-K> (tcgen05 + TMA conv1d-as-GEMM, split-bf16 x3, fp32 accumulate in TMEM, DSMEM reduce-scatter)",
                 "ffma": "conv_kernel<G> (fp32 FFMA conv1d-as-GEMM, cluster split-K)"}[dom]
        other = "ffma" if dom == "tc" else "tc"
        o_ms, o_fl, o_n = fam[other]
        traffic, traffic_src = ncu_traffic(dom)
        # CPU baseline beside it (bounded sample), N=1 only
        cpu = None
        extra = None
        if world == 1:
            n, times, threads = cpu_reference_run(cfg, wl, args.cpu_steps, 2)
            cpu = {"value": n * len(times) / sum(times), "unit": "samples/s", "cores": threads, "threads": threads, "host_cores": host_cores(),
                   "kind": "port",
                   "sample": "%d runs of the same utterance, one stream, on the host cores (PyTorch-CPU restatement of the reference graph at "
                             "its fastest intra-op thread count; onnxruntime unavailable), %.0f ms each" % (len(times), 1e3 * sum(times) / len(times))}
            if not args.no_extras:
                cpu["throughput_all_cores"] = cpu_throughput_all_cores(threads, steps=2)
                extra = extras(cfg, blob, manifest, eng, dev, pk)
                # fp32-exact mode (precision 0) of the headline workload on a second engine
                try:
                    blob0, man0 = weights.pack(folded, cfg, precision=0)
                    e0_ = Engine(cfg, blob0, man0, device=local, precision=0)
                    es0 = torch.cuda.ExternalStream(e0_.stream(), device=dev)
                    for _ in range(4):
                        e0_.infer_dev(d_ids.data_ptr(), wl["lens"], d_sid.data_ptr(), 1, 128, wl["scales"], d_wav.data_ptr(), (Ty + 64) * hop,
                                      d_eps_dp.data_ptr(), d_eps_z.data_ptr(), Ty)
                    ms0 = []
                    for _ in range(10):
                        flush.fill_(1)
                        torch.cuda.synchronize()
                        a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                        a0.record(es0)
                        e0_.infer_dev(d_ids.data_ptr(), wl["lens"], d_sid.data_ptr(), 1, 128, wl["scales"], d_wav.data_ptr(), (Ty + 64) * hop,
                                      d_eps_dp.data_ptr(), d_eps_z.data_ptr(), Ty)
                        a1.record(es0)
                        a1.synchronize()
                        ms0.append(a0.elapsed_time(a1))
                    extra["value_fp32_exact"] = {"precision_mode": 0, "ms_per_step": sum(ms0) / len(ms0), "value": n_samples / (sum(ms0) / len(ms0) / 1e3),
                                                 "unit": "samples/s", "note": "every conv and attention on the fp32 FFMA pipe (no tensor cores)"}
                    e0_.close()
                except Exception as ex:      # noqa: BLE001
                    extra["value_fp32_exact"] = {"error": repr(ex)}
        line = {"metric": METRIC, "value": value, "unit": "samples/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": total_ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "fp32" if args.precision == 0 else "fp32 (flow/decoder convs + attention: bf16 hi+lo split x3 MMAs on tcgen05, fp32 accumulate; rest fp32 FFMA)",
                "data": "synthetic", "config": conf,
                "engine": {"precision_mode": args.precision, "cuda_graphs": "per length bucket", "speculative_second_phase": eng.speculation_stats(),
                           "ranks_pinned_to_gpu_numa_cores": pinned},
                "rtf": (total_ms / 1e3 / args.steps) / (n_samples / SR),
                "e2e": {"value": e2e_v, "unit": "samples/s", "ms_per_step": 1e3 * e2e_total / args.steps,
                        "h2d_bytes_per_step": int(wl["tok"].nbytes + 16 + 8 + wl["eps_dp"].nbytes + wl["eps_z"][:, :, :Ty].nbytes),
                        "d2h_bytes_per_step": int(n_samples * 4 + 8)},
                "e2e_cold": {"value": cold_n_all / cold_total, "unit": "samples/s", "utterances": N_COLD * world,
                             "ms_per_utterance": 1e3 * cold_total / N_COLD, "ms_median_min_max_rank0": [1e3 * sorted(cold_t)[N_COLD // 2], 1e3 * min(cold_t), 1e3 * max(cold_t)],
                             "value_at_median": (cold_n / N_COLD) / sorted(cold_t)[N_COLD // 2],
                             "phonemes": "100..128 (uniform), the headline speaker (sid 2; with these synthetic weights other speaker vectors push the duration predictor to 10-60 frames per phoneme, i.e. a different workload), engine-drawn noise",
                             "graph_replays_in_timed_region": r2 - r1, "graph_launches_expected": 2 * N_COLD,
                             "speculation_hits_misses": [h2 - h1, m2 - m1],
                             "length_buckets_seen_in_warmup": n_warm_buckets, "first_seen_buckets_in_timed_region_tokens_frames_ms": new_in_timed,
                             "workspace_reserved": "Engine.reserve(128 phonemes, 768 frames) before the warm-up (reached %d frames): no buffer moves afterwards" % reserved_frames,
                             "warmup": "150 OTHER distinct utterances of the same distribution (rank 0: %d graph replays among them); a length "
                                       "bucket's first call runs eagerly and captures its graph (calls 1-3 of a fresh engine: %.2f / %.2f / %.2f ms, "
                                       "incl. lazy kernel loading); such calls inside the timed region are what separates the mean from the median"
                                       % (r1 - r0, 1e3 * first_seen[0], 1e3 * first_seen[1], 1e3 * first_seen[2])},
                "gpu_launches": int(launches),
                "roofline": {"kernel": kname, "bound": "tensor", "achieved": ach,
                             "peak": pk["bf16_sustained"], "unit": "TFLOP/s", "frac": ach / pk["bf16_sustained"],
                             "peak_source": pk["src"] + " cuBLAS bf16 (sustained). achieved = algorithmic FLOPs (2*Cin*k*Cout per output "
                             "position) / summed CUDA-event durations of the launches in the profiled pass; the split-bf16 kernel "
                             "issues 3 MMAs per algorithmic MAC, so its ceiling on this scale is peak/3",
                             "traffic": traffic, "traffic_source": traffic_src, "launches_per_step": d_n / max(args.steps, 1),
                             "share_of_step": d_ms / prof_total_ms if prof_total_ms else None,
                             "flops_per_step": d_fl / max(args.steps, 1),
                             "other_family": {"kernel": other, "ms_per_step": o_ms / max(args.steps, 1),
                                              "tflops": (o_fl / (o_ms / 1e3) / 1e12) if o_ms > 0 else 0.0,
                                              "launches_per_step": o_n / max(args.steps, 1)},
                             "profiled_ms_per_step": prof_total_ms / max(args.steps, 1)},
                "cpu_baseline": cpu, "clocks": clocks, "stage_ms": stage,
                "extra": extra if sharded is None else dict(extra or {}, configs3_sharded=sharded),
                "init": {"seconds": init_s, "weight_broadcast_ms": bcast_ms, "weight_bytes": 4 * nblob,
                         "graph_replays": eng.graph_replays()}}
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
