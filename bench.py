#!/usr/bin/env python
"""bench.py — tokens/s of greedy caption decoding (BASELINE.json metric) on N B200s, plus the other BASELINE configs as blocks.

A "step" is one pass of the hot path over one batch of synthetic clips: prologue (region / frame feature encoding, object
interaction) + the 20-step greedy loop, i.e. one ``forward(..., 'sample')`` of the reference (misc/model.py:492-624) for B=100 clips
of 10x100x2048 fc6 RoIs and T frame rows (BASELINE configs[1]).

  value          tokens/s with the clip tensors already resident in HBM (device-timed: CUDA events, barrier + synchronize both sides,
                 max over ranks)
  e2e            the same through the C-ABI host-buffer entry point gvd_sample_greedy_host (pinned host inputs -> H2D -> prologue ->
                 loop -> D2H of ids / logits / similarity), every step
  loop_only      the 20-step greedy loop alone (gvd_decode_greedy: one CUDA-graph replay), timed directly with events
  roofline       dominant kernel family of the step (tcgen05 GEMMs of the prologue) against the measured dense tensor peak
  roofline_decode  attention kernel / whole decode step against the measured HBM peak (SURVEY.md 8d algorithmic bytes)
  stages_ms_per_step  per-stage CUDA-event times recorded on the launching stream by the library's profiler in a SEPARATE pass (the
                 profiled pass enqueues the loop kernel by kernel instead of replaying the graph)
  t480           the reference-default T=480 frame rows (opts.py:50)
  beam           BASELINE configs[3]: beam_size=3 decode, B=100
  train          BASELINE configs[2] (N=1) / configs[4] (N=8): one optimisation step, 100 clips/GPU, ONE NCCL all-reduce of the flat
                 gradient buffer when N>1 (its time reported separately)
  cpu_baseline   the oracle (CPU restatement of the reference's PyTorch path) on the host cores, bounded sample
  gpu_reference  the same restatement (plain PyTorch, fp32, allow_tf32=False, cudnn.benchmark) on the SAME GPU: the "reference
                 single-GPU PyTorch" figure of BASELINE.json's north_star.  Checker code, never the product path.

`--impl reference` times the reference's CPU algorithm (the oracle port; the reference itself is Python that cannot travel to the GPU
box) on a bounded sample of the same workload.  Multi-GPU: one process per GPU (torchrun), clips sharded, no decode collective.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
for p in (ROOT, os.path.join(ROOT, "oracle")):
    if p not in sys.path:
        sys.path.insert(0, p)

import torch  # noqa: E402

METRIC = "tokens/sec greedy decode seq_len=20 batch=100 10x100x2048 RoIs"
UNIT = "tokens/s"
KEYS = ("segs_feat", "ppls", "num", "ppls_feat", "sample_idx", "pnt_mask")


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--batch", type=int, default=100, help="clips per GPU (BASELINE config: 100)")
    ap.add_argument("--frames", type=int, default=10, help="frame-feature rows T (BASELINE literal: 10x3072; reference default 480)")
    ap.add_argument("--cpu-sample", type=int, default=100, help="clips in the bounded CPU-baseline sample")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--quick", action="store_true", help="profiling aid: 1 warm-up, headline leg only (never a bench number)")
    ap.add_argument("--only", default="", help="comma list of extra blocks to run (t480,beam,train,gpu_reference,transformer); default: all")
    ap.add_argument("--no-gpu-reference-tfm", action="store_true", help="skip the eager-PyTorch timing inside the transformer block")
    ap.add_argument("--train-steps", type=int, default=3)
    ap.add_argument("--dump-outputs", metavar="DIR", default="",
                    help="write the outputs of the headline's last timed step (rank 0) as .npy files under DIR")
    return ap.parse_args()


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        p = json.load(open(path))
        return dict(hbm_gbs=float(p["hbm_gbs"]), bf16_tflops=float(p.get("bf16_tflops_sustained", p["bf16_tflops"])),
                    source="measured (MEASURED_PEAKS.json)")
    return dict(hbm_gbs=6650.0, bf16_tflops=1400.0, source="fallback (B200_PROFILING.md)")


def ncu_traffic():
    """dram bytes per launch of the named kernels from the committed ncu captures of this round (profiles/traffic.json, written by
    tools/ncu_traffic.py from `ncu --set full` reports); {} when no capture has been committed."""
    path = os.path.join(ROOT, "profiles", "traffic.json")
    try:
        return json.load(open(path))
    except (OSError, ValueError):
        return {}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits",
                                          "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            try:
                sm.append(float(r[1])); mx.append(float(r[2]))
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[4:8]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            except (ValueError, IndexError):
                pass
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": sorted(reasons),
                "samples": len(sm)}


def algorithmic_bytes(opt, B, T):
    """SURVEY.md 8(d): fp32, dense masks.  Returns (per-step decode bytes, per-step attention-kernel bytes)."""
    R, A, H, E, V = opt.num_sampled_frm * opt.num_prop_per_frm, opt.att_hid_size, opt.rnn_size, opt.input_encoding_size, opt.vocab_size
    per_clip = R * A * 4 + R * H * 4 + T * A * 4 + T * H * 4 + 2 * R + 8 * H * 4 + H * 4 + R * 4 + E * 4 + 8
    shared = 4 * H * (E + H + H) * 4 + 4 * H * (2 * H + H) * 4 + 2 * 4 * H * 4 * 2 + 2 * (A * H + A) * 4 + 2 * (A + 1) * 4 + (V * H + V) * 4
    attn_kernel = B * ((R + T) * (A + H) * 4 + 2 * R + R * 4 + 2 * A * 4)          # rows streamed + masks + logits out + queries
    return B * per_clip + shared, attn_kernel


def prologue_flops(opt, B, T):
    """Dense-contraction FLOPs of the prologue (SURVEY.md 8d 'Algorithmic FLOPs')."""
    R, A, H, D = opt.num_sampled_frm * opt.num_prop_per_frm, opt.att_hid_size, opt.rnn_size, opt.detect_size
    G = H // 2
    per_clip = 2 * R * (2048 * 2048 + (D + 1) * 2048 + (2048 + 300 + D + 1) * H + A * H)
    if opt.obj_interact:
        per_clip += 2 * (2 * R * (4 * H * H + 2 * H * (H // 2)) + 2 * 2 * R * R * H)
    per_clip += 2 * T * ((2048 + (opt.fc_feat_size - 2048)) * (H // 2) + 2 * (3 * G * H + 3 * G * 2 * G) + 2 * 2 * 3 * G * G + A * H)
    return B * per_clip


def workload_config(B, T, L, world):
    """The `config` object of the JSON line: the same for both arms (the reference arm runs this workload on the host cores)."""
    return {"workload": "greedy decode, B=%d clips/GPU, R=10x100 RoIs x 2048, T=%d frame rows x 3072, L=20, V=4905, obj_interact on, "
                        "prologue + 20-step loop per step" % (B, T),
            "batch_per_gpu": B, "seq_len": L, "frames": T, "parallelism": "dp%d (clips sharded, no collective)" % world,
            "l2": "inputs larger than L2 (fc6 819 MB + region features 614 MB per step), no explicit flush"}


class Ctx:
    """Rank / process-group plumbing shared by every leg."""

    def __init__(self, args):
        self.rank = int(os.environ.get("RANK", 0))
        self.world = int(os.environ.get("WORLD_SIZE", 1))
        self.local = int(os.environ.get("LOCAL_RANK", 0))
        self.dist = None
        torch.cuda.set_device(self.local)
        if self.world > 1:
            # NCCL prints its version banner to STDOUT (NCCL_DEBUG=VERSION, also when it comes from an nccl.conf); rank 0 must print
            # one JSON line only: ask for WARN unless the user wants more, and point fd 1 at stderr while the communicator is created
            if os.environ.get("NCCL_DEBUG", "").upper() in ("", "VERSION"):
                os.environ["NCCL_DEBUG"] = "WARN"
            import torch.distributed as dist
            sys.stdout.flush()
            saved_fd = os.dup(1)
            os.dup2(2, 1)
            try:
                dist.init_process_group("nccl", device_id=torch.device("cuda", self.local))
                dist.barrier()                                  # communicator creation (and its banner) happens on the first collective
                torch.cuda.synchronize()
            finally:
                sys.stdout.flush()
                os.dup2(saved_fd, 1)
                os.close(saved_fd)
            self.dist = dist

    def barrier(self):
        if self.dist is not None:
            self.dist.barrier()
        torch.cuda.synchronize()

    def max_ms(self, ms):
        from gvd_b200.dist import max_over_ranks
        return max_over_ranks(ms, "cuda")

    def timed(self, fn, K):
        """K calls of fn bracketed by barrier + synchronize, CUDA events on the launching stream; max over ranks (ms)."""
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        self.barrier()
        e0.record()
        out = None
        for _ in range(K):
            out = fn()
        e1.record()
        self.barrier()
        return self.max_ms(e0.elapsed_time(e1)), out


def measure_decode(ctx, args, T, full):
    """Headline leg at T frame rows.  full=True adds loop_only, the profiled stage pass and the clock record."""
    from gvd_b200 import capi, synth
    B, K, W = args.batch, args.steps, (1 if args.quick else max(args.warmup, 3))
    opt = synth.make_opt(t_attn_size=T)
    sd = synth.make_state_dict(opt)
    nm = capi.NativeModel(opt)
    nm.load_state_dict(sd)
    inp = synth.make_inputs(opt, B, seed=1234 + ctx.rank, masked=False)      # dense masks for the roofline run (SURVEY.md 8d)
    dev = {k: inp[k].cuda() for k in KEYS}
    pin = {k: inp[k].pin_memory() for k in KEYS}

    def step_dev():
        sim = nm.prologue(*(dev[k] for k in KEYS), want_sim=True)
        return nm.decode_greedy(B, T, dev["pnt_mask"]) + (sim,)

    for _ in range(W):
        step_dev()
    # ---- value: inputs resident in HBM
    sampler = ClockSampler(ctx.local)
    if ctx.rank == 0 and full and not args.quick:
        sampler.start()
    l0 = capi.kernel_launches()
    ms, (seq, logp, att2, sim) = ctx.timed(step_dev, K)
    launches = capi.kernel_launches() - l0
    r = dict(opt=opt, sd=sd, ms=ms, launches=launches, uniq=int(len(torch.unique(seq))), B=B, K=K, W=W, T=T,
             outputs=dict(seq=seq, logp=logp, att2=att2, sim=sim))
    if args.quick:
        r["clocks"] = None
        return r
    # ---- loop only: features resident (prologue outputs in the workspace), gvd_decode_greedy alone
    ms_loop, _ = ctx.timed(lambda: nm.decode_greedy(B, T, dev["pnt_mask"]), K)
    r["ms_loop"] = ms_loop
    r["clocks"] = sampler.stop() if (ctx.rank == 0 and full) else None
    # ---- e2e: host buffers through the C-ABI
    out_host = None
    for _ in range(2):
        out_host = nm.sample_greedy_host(*(pin[k] for k in KEYS), out=out_host)
    ms_e2e, out_host = ctx.timed(lambda: nm.sample_greedy_host(*(pin[k] for k in KEYS), out=out_host), K)
    assert torch.equal(out_host["seq"], seq.cpu()), "host-buffer path and device path disagree"
    r["ms_e2e"] = ms_e2e
    r["h2d"] = sum(pin[k].numel() * pin[k].element_size() for k in KEYS)
    r["d2h"] = sum(out_host[k].numel() * out_host[k].element_size() for k in ("seq", "logp", "att2", "sim"))
    if full:
        # ---- per-stage CUDA-event times: separate pass, kernel-by-kernel enqueue (the library skips the graph while profiling)
        capi.profile_reset()
        capi.profile_enable(True)
        ctx.barrier()
        for _ in range(K):
            seq_p = step_dev()[0]
        ctx.barrier()
        capi.profile_enable(False)
        r["stages"] = capi.profile_read()
        assert torch.equal(seq_p, seq), "graph replay and kernel-by-kernel enqueue disagree"
    return r


def measure_beam(ctx, args, T, beam=3):
    """BASELINE configs[3]: beam decode (CaptionModelBU path, repaired semantics), all clips batched on the device."""
    from gvd_b200 import capi, synth
    B, K = args.batch, args.steps
    opt = synth.make_opt(t_attn_size=T)
    nm = capi.NativeModel(opt)
    nm.load_state_dict(synth.make_state_dict(opt))
    inp = synth.make_inputs(opt, B, seed=1234 + ctx.rank, masked=False)
    dev = {k: inp[k].cuda() for k in KEYS}

    def step():
        nm.prologue(*(dev[k] for k in KEYS), want_sim=True, beam=beam)
        return nm.beam_decode(B, T, beam, dev["pnt_mask"])

    for _ in range(3):
        step()
    ms, _ = ctx.timed(step, K)
    return {"config": "beam_size=%d, B=%d clips/GPU, T=%d, L=20 (prologue + beam loop per step)" % (beam, B, T), "beam_size": beam,
            "value": ctx.world * B * opt.seq_length * K / (ms / 1e3), "unit": UNIT, "ms_per_step": ms / K}


def measure_tfm(ctx, args, T):
    """SURVEY 8(f) row 4: the transformer captioner (att_model='transformer'): prologue + Decoder.greedy, B clips per GPU."""
    from gvd_b200 import capi, synth
    B, K = args.batch, args.steps
    opt = synth.make_opt(t_attn_size=T, att_model="transformer")
    sd = synth.make_state_dict(opt)
    nm = capi.NativeModel(opt)
    nm.load_state_dict(sd)
    H, V, L, R = opt.rnn_size, opt.vocab_size, opt.seq_length, nm.R
    cap = capi.TransformerCaptioner(H, V, L)
    cap.load_state_dict(sd)
    inp = synth.make_inputs(opt, B, seed=1234 + ctx.rank, masked=False)
    dev = {k: inp[k].cuda() for k in KEYS}
    enc = lambda: (nm.workspace_tensor(B, T, "conv_feats", (B, T, H)), nm.workspace_tensor(B, T, "pool_feats", (B, R, H)))

    def step():
        nm.prologue(*(dev[k] for k in KEYS), want_sim=False)
        return cap.decode_greedy(*enc())

    for _ in range(3):
        seq = step()
    l0 = capi.kernel_launches()
    ms, seq = ctx.timed(step, K)
    launches = (capi.kernel_launches() - l0) // K
    e0, e1 = enc()
    ms_loop, _ = ctx.timed(lambda: cap.decode_greedy(e0, e1), K)
    pk = peaks()
    # algorithmic bytes of one decode step: K and V of both encoder outputs once per clip, every decoder weight once per batch
    kv_bytes = B * (T + R) * 2 * H * 4
    w_bytes = (2 * (8 * H * H + 2 * H * (H // 2) + 6 * H + H // 2 + H) + V * H + V) * 4
    step_ms = ms_loop / K / L                                           # (includes 1/L of the once-per-batch K / V projection)
    out = {"config": "att_model='transformer' (misc/model.py:137-143,570-578): prologue + 2-layer Decoder.greedy, B=%d clips/GPU, T=%d, L=%d" % (B, T, L),
           "value": ctx.world * B * L * K / (ms / 1e3), "unit": UNIT, "ms_per_step": ms / K, "loop_only_ms": ms_loop / K,
           "loop_only_tokens_per_s": ctx.world * B * L * K / (ms_loop / 1e3), "gpu_launches": launches, "distinct_tokens": int(len(torch.unique(seq))),
           "roofline_decode": {"bound": "hbm", "algorithmic_bytes_per_step": kv_bytes + w_bytes, "ms_per_decode_step": step_ms,
                               "achieved": (kv_bytes + w_bytes) / (step_ms / 1e3) / 1e9, "peak": pk["hbm_gbs"], "unit": "GB/s",
                               "frac": (kv_bytes + w_bytes) / (step_ms / 1e3) / 1e9 / pk["hbm_gbs"],
                               "how": "(K + V of both encoder outputs per clip + decoder weights per batch) / (timed gvd_tfm_decode_greedy / L)"}}
    if ctx.rank == 0 and ctx.world == 1 and not args.no_gpu_reference_tfm:
        sys.path.insert(0, os.path.join(ROOT, "oracle"))
        import gvd_oracle as O
        Wd = {k: v.cuda() for k, v in sd.items()}
        torch.backends.cuda.matmul.allow_tf32 = False
        torch.backends.cudnn.allow_tf32 = False
        with torch.no_grad():
            encs = [e0.clone(), e1.clone()]
            ref = O.tfm_greedy(Wd, opt, encs, reproject=True)
            torch.cuda.synchronize()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            for _ in range(2):
                O.tfm_greedy(Wd, opt, encs, reproject=True)
            b.record()
            torch.cuda.synchronize()
        rms = a.elapsed_time(b) / 2
        out["gpu_reference"] = {"loop_only_ms": rms, "loop_only_tokens_per_s": B * L / (rms / 1e3), "ids_equal": bool(torch.equal(ref, seq)),
                                "speedup_loop_only": rms / (ms_loop / K),
                                "kind": "eager PyTorch port of Decoder.greedy on cuda:0 (fp32, allow_tf32=False), re-projecting the encoder output with "
                                        "wk / wv at every step as the reference does (transformer.py:117-119,232-236)"}
    return out


def measure_train(ctx, args, T):
    """BASELINE configs[2] / [4]: one optimisation step (train-mode forward, four losses with w_att2 = 0.1 / w_cls = 0.1, explicit backward,
    [N>1: ONE NCCL sum-all-reduce of the flat gradient buffer], global-norm clip, Adam) on 100 clips per GPU."""
    from gvd_b200 import synth
    from gvd_b200.train import Trainer
    from gvd_b200.train_ops import NativeOps
    B, K = args.batch, args.train_steps
    opt = synth.make_opt(t_attn_size=T)
    opt.w_att2, opt.w_grd, opt.w_cls = 0.1, 0.0, 0.1
    sd = synth.make_state_dict(opt)
    inp = synth.make_inputs(opt, B, seed=4321 + ctx.rank, masked=True, train=True)
    dev = {k: v.cuda() for k, v in inp.items()}
    host = {k: inp[k] for k in ("gt_seq", "input_seq", "sample_idx")}
    ar_ms = []

    def all_reduce(flat):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        ctx.dist.all_reduce(flat, op=ctx.dist.ReduceOp.SUM)
        e1.record()
        ar_ms.append((e0, e1))
        return flat

    tr = Trainer(NativeOps(), sd, opt, all_reduce=all_reduce if ctx.world > 1 else None, n_replicas=ctx.world)
    for _ in range(2):
        losses, loss = tr.step(dev, host)
    ar_ms.clear()
    ms, (losses, loss) = ctx.timed(lambda: tr.step(dev, host), K)
    out = {"config": "training step, %d clips/GPU x %d GPU(s), T=%d, w_att2=0.1 w_cls=0.1, obj_interact on, dropout p=0 "
                     "(deterministic parity mode), fp32" % (B, ctx.world, T),
           "ms_per_step": ms / K, "clips_per_s": ctx.world * B * K / (ms / 1e3), "loss": float(loss), "losses": [float(x) for x in losses],
           "grad_norm": float(tr.norm[0]), "grad_bytes": tr.numel * 4, "collective": None}
    if ctx.rank == 0 and ctx.world == 1:
        # the same optimisation step in eager PyTorch on this GPU (oracle restatement + autograd, fp32, TF32 off): context for ms_per_step
        try:
            import gvd_oracle as O
            torch.backends.cuda.matmul.allow_tf32 = False
            torch.backends.cudnn.allow_tf32 = False
            sdc = {k: v.cuda() for k, v in sd.items()}
            ts = []
            for it in range(4):
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                torch.cuda.synchronize()
                e0.record()
                O.train_step(sdc, opt, dev)
                e1.record()
                torch.cuda.synchronize()
                if it >= 1:
                    ts.append(e0.elapsed_time(e1))
            ts.sort()
            out["gpu_reference"] = {"ms_per_step": ts[len(ts) // 2], "kind": "oracle train_step (eager PyTorch autograd, fp32, allow_tf32=False) on cuda:0",
                                    "speedup": ts[len(ts) // 2] / (ms / K)}
            del sdc
        except Exception as e:                                          # noqa: BLE001
            out["gpu_reference"] = {"unavailable": "%s: %s" % (type(e).__name__, str(e)[:200])}
    if ar_ms:
        t = [a.elapsed_time(b) for a, b in ar_ms]
        ar = ctx.max_ms(sum(t) / len(t))                                 # slowest rank's view (a late rank sees a shorter collective)
        out["collective"] = {"op": "ncclAllReduce(sum) of the flat fp32 gradient buffer, one call per step", "bytes": tr.numel * 4,
                             "ms": ar, "calls_per_step": len(t) / K, "share_of_step": ar / (ms / K),
                             "busbw_GBs": tr.numel * 4 * 2 * (ctx.world - 1) / ctx.world / (ar / 1e3) / 1e9}
    return out


def pick_cpu_threads(opt, sd, inp):
    """The host has far more cores than small fp32 GEMMs can use; choose the thread count that makes
    the oracle fastest on a 2-clip probe (the count used is reported as `cores`)."""
    import gvd_oracle as O
    ncpu = os.cpu_count() or 1
    cands = sorted({c for c in (8, 16, 32, 64, ncpu) if c <= ncpu})
    probe = {k: v[:2] for k, v in inp.items()}
    best = None
    with torch.no_grad():
        for c in cands:
            torch.set_num_threads(c)
            O.sample_greedy(sd, opt, probe)
            t0 = time.perf_counter()
            O.sample_greedy(sd, opt, probe)
            dt = time.perf_counter() - t0
            if best is None or dt < best[0]:
                best = (dt, c)
    torch.set_num_threads(best[1])
    return best[1]


def cpu_baseline(opt, sd, n_clips, T, repeats=1):
    """Oracle port of the reference's CPU PyTorch path on a bounded sample of the workload."""
    import gvd_oracle as O
    from gvd_b200 import synth
    inp = synth.make_inputs(opt, n_clips, seed=1234, masked=False)
    pick_cpu_threads(opt, sd, inp)
    with torch.no_grad():
        best = None
        for _ in range(repeats):
            t0 = time.perf_counter()
            O.sample_greedy(sd, opt, inp)
            dt = time.perf_counter() - t0
            best = dt if best is None else min(best, dt)
    return {"value": n_clips * opt.seq_length / best, "unit": UNIT, "cores": torch.get_num_threads(), "kind": "port",
            "sample": "%d clips (of the %d-clip batch), T=%d, same weights/inputs generator, greedy L=%d; %.1f s of CPU work"
                      % (n_clips, 100, T, opt.seq_length, best)}


def gpu_reference(opt, sd, B, T):
    """The reference's PyTorch algorithm (oracle restatement: plain torch ops, no nn.Module) on THIS GPU in fp32 with TF32 off and
    cudnn.benchmark on (main.py:532) — BASELINE.md row R-GPU, the 'reference single-GPU PyTorch' of the north_star.  3 warm-ups,
    median of 5, CUDA events; loop-only and end-to-end 'sample' like SURVEY.md 8(d)."""
    import gvd_oracle as O
    from gvd_b200 import synth
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cudnn.benchmark = True
    sdc = {k: v.cuda() for k, v in sd.items()}
    inp = {k: v.cuda() for k, v in synth.make_inputs(opt, B, seed=1234, masked=False).items()}
    times, loops = [], []
    with torch.no_grad():
        for it in range(8):
            e0, e1, e2 = (torch.cuda.Event(enable_timing=True) for _ in range(3))
            torch.cuda.synchronize()
            e0.record()
            feats = O.prologue(sdc, opt, inp["segs_feat"], inp["ppls"], inp["num"], inp["ppls_feat"], inp["sample_idx"], inp["pnt_mask"])
            e1.record()
            O.sample_greedy(sdc, opt, inp, feats=feats)
            e2.record()
            torch.cuda.synchronize()
            if it >= 3:
                times.append(e0.elapsed_time(e2)); loops.append(e1.elapsed_time(e2))
    times.sort(); loops.sort()
    ms, ms_loop = times[len(times) // 2], loops[len(loops) // 2]
    return {"value": B * opt.seq_length / (ms / 1e3), "unit": UNIT, "ms_per_step": ms, "loop_only_ms": ms_loop,
            "loop_only_tokens_per_s": B * opt.seq_length / (ms_loop / 1e3), "kind": "port of the reference's PyTorch path on cuda:0 "
            "(fp32, allow_tf32=False, cudnn.benchmark=True), eager", "torch": torch.__version__}


DUMP_BYTES = 63_000_000                     # array bytes of --dump-outputs; the .npy headers stay within the rest of 64 MB


def dump_outputs(path, seq, logp, att2, sim):
    """--dump-outputs: what one headline step hands its caller, as .npy files, so that two builds run with the same arguments (hence the
    same seeded inputs) can be compared output for output.  seq (token ids, as exact float64) and logp are written whole; att2 and sim
    (1.8 MB per clip at the default sizes) on a fixed, seeded sample of clips, listed in clips.npy, that keeps the directory under 64 MB."""
    import numpy as np
    os.makedirs(path, exist_ok=True)
    B = seq.shape[0]
    out = {"seq": seq.double(), "logp": logp.float()}
    room = DUMP_BYTES - sum(t.numel() * t.element_size() for t in out.values()) - B * 8
    n = min(B, room // ((att2[0].numel() + sim[0].numel()) * 4))
    clips = torch.randperm(B, generator=torch.Generator().manual_seed(0))[:n].sort().values
    out.update(clips=clips.double(), att2=att2[clips.to(att2.device)], sim=sim[clips.to(sim.device)])
    for name, t in out.items():
        np.save(os.path.join(path, name + ".npy"), t.cpu().numpy())


def run_ours(args):
    ctx = Ctx(args)
    only = set(x for x in args.only.split(",") if x) or {"t480", "beam", "train", "gpu_reference", "transformer"}
    T = args.frames
    r = measure_decode(ctx, args, T, True)
    outputs = r.pop("outputs")
    if args.dump_outputs and ctx.rank == 0:
        dump_outputs(args.dump_outputs, **outputs)
    del outputs
    opt, B, K, W = r["opt"], r["B"], r["K"], r["W"]
    world = ctx.world
    tokens = world * B * opt.seq_length * K
    pk = peaks()
    traffic = ncu_traffic()
    dec_bytes, attn_bytes = algorithmic_bytes(opt, B, T)
    line = {
        "metric": METRIC, "value": tokens / (r["ms"] / 1e3), "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W,
        "ms_per_step": r["ms"] / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic (seeded |N(0,1)| fc6 10x100x2048, N(0,1) frame feats, random-init weights of the reference architecture)",
        "config": workload_config(B, T, opt.seq_length, world),
        "gpu_launches": r["launches"], "clocks": r["clocks"], "distinct_tokens": r["uniq"],
    }
    if args.quick:
        if ctx.rank == 0:
            print(json.dumps(line))
        return
    line["e2e"] = {"value": tokens / (r["ms_e2e"] / 1e3), "unit": UNIT, "h2d_bytes_per_step": r["h2d"], "d2h_bytes_per_step": r["d2h"],
                   "ms_per_step": r["ms_e2e"] / K, "api": "gvd_sample_greedy_host (C-ABI, pinned host buffers)"}
    st = r["stages"]
    stage_ms = {k: v[0] / K for k, v in st.items()}
    loop_ms = r["ms_loop"] / K                                          # timed directly (events around gvd_decode_greedy)
    line["loop_only"] = {"ms_per_step": loop_ms, "tokens_per_s": world * B * opt.seq_length / (loop_ms / 1e3),
                         "how": "CUDA events around gvd_decode_greedy alone (one graph replay of 20 steps), features resident"}
    a = st.get("decode.attn_partial")
    if a and a[1]:
        a_ms = a[0] / a[1]
        ach = attn_bytes / (a_ms / 1e3) / 1e9
        step_ms = loop_ms / opt.seq_length
        tr_attn = traffic.get("attn_partial_kernel", {})
        line["roofline_decode"] = {
            "kernel": "attn_partial_kernel (TMA-fed region+temporal attention, one launch per decode step)", "bound": "hbm",
            "achieved": ach, "peak": pk["hbm_gbs"], "unit": "GB/s", "frac": ach / pk["hbm_gbs"],
            "traffic": tr_attn.get("dram_bytes") if (B == 100 and T == 10) else None, "traffic_source": tr_attn.get("source"),
            "algorithmic_bytes_per_launch": attn_bytes, "avg_launch_ms": a_ms, "peak_source": pk["source"],
            "whole_step": {"algorithmic_bytes_per_step": dec_bytes, "ms_per_decode_step": step_ms,
                           "achieved": dec_bytes / (step_ms / 1e3) / 1e9, "frac": dec_bytes / (step_ms / 1e3) / 1e9 / pk["hbm_gbs"],
                           "how": "SURVEY 8(d) bytes per step / (directly timed loop / 20)"},
        }
    gemm_stages = [k for k in stage_ms if k.split(".")[0] in ("region", "interact", "frame", "clip") and
                   k not in ("region.sim_softmax", "region.sim_transpose", "region.pool_in", "interact.softmax", "interact.add_ln",
                             "interact.k_split", "interact.v_transpose", "frame.gru_pointwise", "clip.frame_mean", "clip.vector")]
    gemm_ms = sum(stage_ms[k] for k in gemm_stages)
    note = ("algorithmic fp32 FLOPs; each product is 3 tensor-core MMAs on an 11+11-bit hi/lo split (fp16x3; token ids must be bit-exact vs an "
            "fp32 oracle), so the fp32-faithful ceiling is 1/3 of the dense fp16/bf16 peak used as the denominator")
    kg = st.get("kernel.f16ss_gemm")
    if kg and kg[1]:
        # the dominant kernel: the conversion-free persistent GEMM; every launch of it in the step, live CUDA-event times
        H, A_, R_, NC = opt.rnn_size, opt.att_hid_size, opt.num_sampled_frm * opt.num_prop_per_frm, opt.detect_size + 1
        per_row = 2048 * 2048 + NC * 2048 + H * (2048 + 300 + NC) + A_ * H           # unpadded (algorithmic) sizes
        if opt.obj_interact:
            per_row += 2 * (3 * H * H + H * H + 2 * (H // 2) * H)
        fl_k = 2.0 * B * R_ * per_row
        n_launch = kg[1] / K
        k_ms = kg[0] / K
        tr_k = traffic.get("f16ss_persistent_kernel", {})
        ach = fl_k / (k_ms / 1e3) / 1e12
        line["roofline"] = {
            "kernel": "f16ss_persistent_kernel<256> (conversion-free persistent tcgen05 GEMM, both operands fp16x3 images; %d launches per step: fc7, "
                      "similarity, region embedding, Q|K|V, Wo, FFN x2 per encoder layer, ctx2pool; %.0f%% of the step)" % (round(n_launch), 100 * k_ms / (r["ms"] / K)),
            "bound": "tensor", "achieved": ach, "peak": pk["bf16_tflops"], "unit": "TFLOP/s", "frac": ach / pk["bf16_tflops"],
            "frac_of_3pass_ceiling": ach / (pk["bf16_tflops"] / 3),
            "algorithmic_flops_per_launch": fl_k / n_launch, "avg_launch_ms": k_ms / n_launch, "launches_per_step": n_launch,
            "traffic": tr_k.get("dram_bytes"), "traffic_launch": "fc7 (M=100000, N=2048, K=2048): algorithmic 2.47 GB (A image 819 MB + W image 17 MB read; fp32 C 819 MB + "
                                                                   "output image 819 MB written)" if tr_k else None,
            "traffic_source": tr_k.get("source"), "tensor_pipe_active_pct_ncu": tr_k.get("tensor_pipe_active_pct"),
            "peak_source": pk["source"], "note": note,
        }
    if gemm_ms:
        fl = prologue_flops(opt, B, T)
        ach = fl / (gemm_ms / 1e3) / 1e12
        line["roofline_prologue_family"] = {
            "kernels": "every dense contraction of the prologue: f16ss_persistent_kernel, tc2_gemm_kernel (frame branch, clip vector), tc_astat_kernel + "
                       "tc_pv_kernel (self-attention pair), gru_step_f16_kernel, and the remaining activation packing passes",
            "achieved": ach, "peak": pk["bf16_tflops"], "unit": "TFLOP/s", "frac": ach / pk["bf16_tflops"], "algorithmic_flops_per_step": fl,
            "ms_per_step": gemm_ms, "share_of_step": gemm_ms / (r["ms"] / K), "note": note,
        }
        if "roofline" not in line:
            line["roofline"] = dict(line["roofline_prologue_family"], bound="tensor", kernel=line["roofline_prologue_family"]["kernels"], traffic=None)
    line["stages_ms_per_step"] = {k: round(v, 4) for k, v in sorted(stage_ms.items(), key=lambda kv: -kv[1])}
    own = {k: v for k, v in stage_ms.items() if not k.startswith("kernel.")}           # (kernel.* entries are nested inside the stages)
    line["dominant_stage"] = max(own, key=own.get) if own else None
    def block(name, fn):
        """Extra blocks never take the headline line down with them (all ranks take the same branch: failures here are deterministic)."""
        try:
            line[name] = fn()
        except Exception as e:                                          # noqa: BLE001
            import traceback
            traceback.print_exc(file=sys.stderr)
            line[name] = {"unavailable": "%s: %s" % (type(e).__name__, str(e)[:300])}

    def t480():
        r2 = measure_decode(ctx, args, 480, False)
        return {"value": world * B * opt.seq_length * K / (r2["ms"] / 1e3), "ms_per_step": r2["ms"] / K,
                "e2e": world * B * opt.seq_length * K / (r2["ms_e2e"] / 1e3), "loop_only_ms": r2["ms_loop"] / K,
                "config": "as the headline with T=480 frame rows (reference default, opts.py:50)"}

    def gpu_ref():
        g = gpu_reference(r["opt"], r["sd"], B, T)
        g["speedup_value"] = line["value"] / g["value"]
        g["speedup_loop_only"] = line["loop_only"]["tokens_per_s"] / g["loop_only_tokens_per_s"]
        return g

    if "t480" in only:
        block("t480", t480)
    if "beam" in only:
        block("beam", lambda: measure_beam(ctx, args, T))
    if "train" in only:
        block("train", lambda: measure_train(ctx, args, T))
    if "transformer" in only:
        block("transformer", lambda: measure_tfm(ctx, args, T))
    if ctx.rank == 0 and world == 1:
        if not args.no_cpu_baseline:
            line["cpu_baseline"] = cpu_baseline(r["opt"], r["sd"], args.cpu_sample, T)
        if "gpu_reference" in only:
            block("gpu_reference", gpu_ref)
    if ctx.rank == 0:
        print(json.dumps(line))
    if ctx.dist is not None:
        ctx.dist.destroy_process_group()


def run_reference(args):
    """Reference arm: the reference's CPU algorithm (oracle port) on the host cores.  Each step is a bounded sample of the workload
    (--cpu-sample clips of the 100-clip batch); `--warmup` untimed steps run first (capped at 2 to bound the run).  Under torchrun rank 0
    alone runs it; `n_gpus` reports the launch, the value is ONE host's CPU throughput whatever N is."""
    rank = int(os.environ.get("RANK", 0))
    if rank != 0:
        return
    from gvd_b200 import synth
    import gvd_oracle as O
    T, n = args.frames, args.cpu_sample
    opt = synth.make_opt(t_attn_size=T)
    sd = synth.make_state_dict(opt)
    inp = synth.make_inputs(opt, n, seed=1234, masked=False)
    pick_cpu_threads(opt, sd, inp)
    K, W = args.steps, max(0, min(args.warmup, 2))
    with torch.no_grad():
        for _ in range(W):
            O.sample_greedy(sd, opt, inp)
        t0 = time.perf_counter()
        for _ in range(K):
            O.sample_greedy(sd, opt, inp)
        dt = time.perf_counter() - t0
    v = n * opt.seq_length * K / dt
    # the same workload object as our arm; the arm-specific facts (CPU algorithm, bounded sample, one host process) sit next to it
    cfg = workload_config(args.batch, T, opt.seq_length, max(1, int(os.environ.get("WORLD_SIZE", args.gpus))))
    arm = ("reference CPU algorithm (oracle port) on the host cores: %d clips of the %d-clip batch per step; one host process whatever --gpus is"
           % (n, args.batch))
    line = {"impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": K, "warmup": W,
            "ms_per_step": dt / K * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": cfg, "reference_arm": arm,
            "cpu_baseline": {"value": v, "unit": UNIT, "cores": torch.get_num_threads(), "kind": "port",
                             "sample": "%d clips per step x %d steps (+%d warm-up)" % (n, K, W)},
            "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0}
    print(json.dumps(line))


if __name__ == "__main__":
    a = parse()
    if a.impl == "reference":
        run_reference(a)
    else:
        run_ours(a)
