#!/usr/bin/env python
"""Benchmark of the community-1 diarization hot path (BASELINE.json metric: audio-hours/sec).

A "step" = one pass of the whole pipeline (segmentation -> embeddings -> clustering -> reconstruction -> annotations)
over a batch of synthetic 10-minute files (12 per GPU by default = BASELINE.json configs[4], 100 x 10 min over
8 GPUs, scaled to one GPU).  Weak scaling.  For N > 1 the default data path is the north star's: the chunks of all
files form one global pool (each rank computes its share), ONE in-place NCCL all-gather replicates embeddings +
powerset classes, and file g is clustered / reconstructed on rank g mod N (`--parallelism pool`);
`--parallelism files` keeps plain file sharding without any data-path collective.

  value : audio-hours/sec, waveforms already resident in HBM (CUDA events, max over ranks)
  e2e   : the same through the public batch API with HOST waveforms (H2D + D2H inside the timed region)
  roofline     : ResNet34 trunk conv kernels (~98 % of the FLOPs) measured live with CUDA events; `traffic` from the
                 latest ncu capture of the same kernels (profiles/*_trunk_traffic.json)
  cpu_baseline : the CPU oracle (reference-equivalent: 3 trunk passes per chunk) on a bounded sample, rank 0, N=1
  eager_cuda_baseline : the same oracle networks in PyTorch-eager CUDA fp32 with TF32 off (what the reference itself
                 would run on this GPU, utils/reproducibility.py:68-83), batch 32, CUDA events

`--impl reference` times the CPU oracle arm (the reference package itself cannot be imported in this image:
lightning / pyannote.core / asteroid_filterbanks are absent, see DESIGN.md).  Its sample is one short file per step,
end to end, normalised to the chunk density of the 10-minute workload (stated in cpu_baseline.sample).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "audio-hours/sec (RTF) community-1 diarization, 16kHz mono, 1/2/4/8 B200"
TRUNK_FLOP_PER_SEGMENT = 45.18e9   # 33 conv3x3 + 3 conv1x1 of ResNet34 at (80 x 998), SURVEY.md section 8(d)


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--files-per-gpu", type=int, default=12)
    ap.add_argument("--minutes", type=float, default=10.0)
    ap.add_argument("--cpu-sample-seconds", type=float, default=24.0)
    ap.add_argument("--parallelism", default="auto", choices=["auto", "pool", "files"],
                    help="N>1 data path: global chunk pool + one all-gather (default) or collective-free file sharding")
    ap.add_argument("--collective", default="p2p", choices=["p2p", "nccl"],
                    help="pool mode: embeddings pushed to peers from the GEMM epilogue over symmetric memory (p2p, "
                         "falls back to nccl when unavailable) or one ncclAllGather")
    ap.add_argument("--no-eager-baseline", action="store_true", help="skip the PyTorch-eager CUDA fp32 leg")
    ap.add_argument("--min-warmup", type=int, default=3, help="lower only when profiling under ncu")
    ap.add_argument("--no-cpu-baseline", action="store_true", help="skip the CPU oracle leg (profiling runs)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step returned for each file to DIR/<uri>_<output>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of the b200 arm")
    return args


def peaks():
    try:
        return json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        return {}


class ClockSampler:
    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits",
                                          "-i", str(self.index), "-lms", "200"], stdout=subprocess.PIPE, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        sm, mx, pw, reasons = [], [], [], set()
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx.append(float(r[1]))
            except Exception:
                continue
            try:
                pw.append(float(r[2]))
            except Exception:
                pass
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm),
                "power_w": float(np.median(pw)) if pw else None, "power_max_w": max(pw) if pw else None}


def oracle_models():
    from oracle import nets, pipeline as P
    from pyannote_audio_b200 import synthetic as syn

    seg, emb = nets.PyanNet(), nets.WeSpeakerResNet34()
    seg.load_state_dict(syn.make_segmentation_state_dict(0))
    emb.load_state_dict(syn.make_embedding_state_dict(1))
    return seg.eval(), emb.eval(), P.PLDA(**syn.make_plda(2))


def workload_config(args, world):
    """The `config` object of the JSON line: identical for the GPU arm and the CPU reference arm."""
    step_chunks = int(round(args.minutes * 60.0)) - 10 + 1
    par = "single GPU" if world == 1 else (
        f"global chunk pool x{world}, embeddings + classes exchanged once ({args.collective}: "
        + ("pushed to the peers from the embedding GEMM's epilogue over NVLink" if args.collective == "p2p"
           else "one ncclAllGather") + f"), per-file stage on rank g mod {world}"
        if pool_mode(args, world) else f"file-sharded x{world}, no data-path collective")
    return {"workload": f"community-1 diarization pipeline end-to-end, {args.files_per_gpu} x {args.minutes:g} min "
                        f"synthetic 16 kHz mono files per GPU (BASELINE.json configs[4] scaled per GPU)",
            "files_per_gpu": args.files_per_gpu, "chunks_per_gpu": args.files_per_gpu * step_chunks,
            "audio_hours_per_step_per_gpu": args.files_per_gpu * args.minutes / 60.0, "parallelism": par,
            "l2": f"inputs larger than L2: {args.files_per_gpu * args.minutes * 60 * 16000 * 4 / 1e6:.0f} MB of "
                  f"waveform per step"}


def pool_mode(args, world):
    return world > 1 and args.parallelism in ("auto", "pool")


def dump_outputs(outdir, outputs):
    """Writes the (file, DiarizeOutput) pairs of one step: per file, the speaker turns of both diarizations as
    (start s, end s, speaker index) rows and the speaker embeddings (one row per speaker, in label order)."""
    os.makedirs(outdir, exist_ok=True)
    for file, out in outputs:
        for name, ann in (("diarization", out.speaker_diarization),
                          ("exclusive_diarization", out.exclusive_speaker_diarization)):
            rows = [(s.start, s.end, int(lab.rsplit("_", 1)[1])) for s, _, lab in ann.itertracks(yield_label=True)]
            np.save(os.path.join(outdir, f"{file['uri']}_{name}.npy"), np.array(rows, dtype=np.float64).reshape(-1, 3))
        np.save(os.path.join(outdir, f"{file['uri']}_speaker_embeddings.npy"),
                np.asarray(out.speaker_embeddings, dtype=np.float64))


def cpu_pass(seconds, models, seed=4242):
    """One reference-equivalent CPU pass (3 trunk forwards per chunk like the reference) -> (wall seconds, chunks)."""
    from oracle import pipeline as P
    from pyannote_audio_b200 import synthetic as syn

    seg, emb, plda = models
    wav = syn.make_conversation(seconds, seed=seed)
    t0 = time.perf_counter()
    out = P.apply(seg, emb, plda, wav, seg_batch=32, emb_batch=8, share_trunk=False)
    return time.perf_counter() - t0, int(out.segmentations.data.shape[0])


def cpu_value(args, t, chunks):
    """audio-hours/sec of the CPU arm on the bench workload: the sample's chunks per second, divided by the chunk
    density of the workload's files (591 chunks per 600 s: a 10 s window every 1 s) -- per-chunk cost dominates (the
    three ResNet passes per chunk are > 99 % of the CPU time), so the short sample extrapolates linearly."""
    file_s = args.minutes * 60.0
    density = (int(round(file_s)) - 10 + 1) / file_s           # chunks per audio-second of the workload
    return (chunks / t) / density / 3600.0


def cpu_sample_text(args, t, chunks):
    return (f"CPU oracle (PyTorch CPU fp32, 3 trunk passes per chunk as the reference), one {args.cpu_sample_seconds:g} s "
            f"synthetic file end-to-end = {chunks} chunks in {t:.1f} s wall, extrapolated linearly to the workload's "
            f"{int(round(args.minutes * 60)) - 9} chunks per {args.minutes:g}-min file (per-chunk cost)")


def run_reference(args, rank, world):
    if rank != 0:
        return
    torch.set_num_threads(min(32, os.cpu_count() or 1))   # conv on >32 threads oversubscribes and gets slower
    models = oracle_models()
    secs = args.cpu_sample_seconds
    for _ in range(min(args.warmup, 1)):
        cpu_pass(12.0, models)
    runs = [cpu_pass(secs, models, seed=4242 + i) for i in range(max(1, args.steps))]
    t = float(np.mean([r[0] for r in runs]))
    chunks = runs[0][1]
    value = cpu_value(args, t, chunks)
    line = {"metric": METRIC, "value": value, "unit": "audio-hours/sec", "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": t * 1e3, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic", "impl": "reference",
            "config": workload_config(args, world),
            "rtf": 1.0 / (value * 3600.0),
            "cpu_baseline": {"value": value, "unit": "audio-hours/sec", "cores": torch.get_num_threads(),
                             "kind": "port", "sample": cpu_sample_text(args, t, chunks)},
            "e2e": {"value": value, "unit": "audio-hours/sec", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


def eager_cuda_baseline(args, dev, chunks=64):
    """The oracle networks (= the reference's modules) in PyTorch-eager CUDA fp32 with TF32 off, batch 32, timed with
    CUDA events: PyanNet on `chunks` chunks + WeSpeaker on 3 x `chunks` (waveform, mask) pairs, i.e. the reference's
    GPU work per chunk without its host loops, numpy round trips and clustering (which only flatters this leg)."""
    from oracle import nets
    from pyannote_audio_b200 import synthetic as syn

    torch.backends.cuda.matmul.allow_tf32 = False            # utils/reproducibility.py:68-83
    torch.backends.cudnn.allow_tf32 = False
    seg, emb = nets.PyanNet(), nets.WeSpeakerResNet34()
    seg.load_state_dict(syn.make_segmentation_state_dict(0))
    emb.load_state_dict(syn.make_embedding_state_dict(1))
    seg, emb = seg.eval().to(dev), emb.eval().to(dev)
    wav = syn.make_conversation(10.0 + chunks - 1, seed=77)
    x = wav.unfold(1, 160000, 16000).permute(1, 0, 2).contiguous().to(dev)[:chunks]      # (chunks,1,160000)
    masks = (torch.rand(chunks, 589, device=dev) < 0.5).float()

    def run():
        with torch.inference_mode():
            for c in range(0, chunks, 32):
                seg(x[c:c + 32])
            for _ in range(3):                                  # one forward per local speaker, like the reference
                for c in range(0, chunks, 32):
                    emb(x[c:c + 32], weights=masks[c:c + 32])

    run()
    torch.cuda.synchronize(dev)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    run()
    e1.record()
    torch.cuda.synchronize(dev)
    t = e0.elapsed_time(e1) / 1e3
    del seg, emb, x
    torch.cuda.empty_cache()
    return {"value": cpu_value(args, t, chunks), "unit": "audio-hours/sec", "kind": "oracle modules, PyTorch eager "
            "CUDA fp32, TF32 off (cuDNN / cuBLAS), batch 32", "sample": f"{chunks} chunks: PyanNet + 3 x WeSpeaker "
            f"ResNet34 forwards in {t * 1e3:.0f} ms (networks only: no host loops, no clustering), extrapolated per "
            f"chunk like cpu_baseline"}


def trunk_traffic():
    """(DRAM bytes, segments, file) of one trunk pass over an embedding sub-batch from the newest committed ncu
    capture (profiles/*_trunk_traffic.json, produced by scripts/ncu_trunk_traffic.py from an
    `ncu --metrics dram__bytes_*` launch list)."""
    import glob

    files = sorted(glob.glob(os.path.join(ROOT, "profiles", "r*_trunk_traffic.json")))
    if not files:
        return None, None, None
    d = json.load(open(files[-1]))
    return (d.get("dram_bytes_per_pass", d.get("dram_bytes_per_256_segments")), int(d.get("segments", 256)),
            os.path.basename(files[-1]))


def main():
    args = parse()
    rank = int(os.environ.get("RANK", 0))
    local_rank = int(os.environ.get("LOCAL_RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    import torch.distributed as dist

    from pyannote_audio_b200 import synthetic as syn
    from pyannote_audio_b200.models import PyanNet, WeSpeakerResNet34, get_context
    from pyannote_audio_b200.parallel import ChunkPool
    from pyannote_audio_b200.pipeline import SpeakerDiarization

    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    seg, emb = PyanNet(), WeSpeakerResNet34()
    seg.load_state_dict(syn.make_segmentation_state_dict(0), strict=False)
    emb.load_state_dict(syn.make_embedding_state_dict(1), strict=False)
    pipe = SpeakerDiarization(segmentation=seg, embedding=emb, plda=syn.make_plda(2), device=dev)
    ctx = get_context(dev)
    nfiles = args.files_per_gpu
    files = []
    for i in range(nfiles):
        wav = syn.make_conversation(args.minutes * 60.0, seed=1000 + rank * 1000 + i)
        files.append({"waveform": wav.pin_memory(), "sample_rate": 16000, "uri": f"r{rank}_f{i}"})
    audio_hours = nfiles * args.minutes / 60.0
    h2d = sum(f["waveform"].numel() * 4 for f in files)
    use_pool = pool_mode(args, world)
    pool = ChunkPool(pipe, collective=args.collective) if use_pool else None

    def sync():
        torch.cuda.synchronize(dev)
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize(dev)

    def timed(fn, steps):
        sync()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        sync()
        ms = e0.elapsed_time(e1)
        if world > 1:
            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms / steps

    resident = pool.upload(files) if use_pool else pipe.upload(files)
    done = [0]
    coll_ms = []
    last_outputs = []

    def step_resident():
        last_outputs[:] = pool.run_resident(resident) if use_pool else pipe.run_resident(resident)
        done[0] = len(last_outputs)
        if use_pool:
            coll_ms.append(pool._events)

    d2h = [0]

    def step_e2e():
        n = 0
        for _ in (pool.apply_batch(files) if use_pool else pipe.apply_batch(files)):
            n += 1
        done[0] = n
        d2h[0] = pipe.d2h_bytes

    for _ in range(max(args.min_warmup, args.warmup)):
        step_resident()
    step_e2e()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    ctx.set_option("profile", 1)
    ctx.timer("trunk"); ctx.timer("seg")
    l0 = ctx.launch_count
    coll_ms.clear()
    ms_resident = timed(step_resident, args.steps)
    launches = (ctx.launch_count - l0) // max(1, args.steps)
    trunk_ms, trunk_segments = ctx.timer("trunk")
    seg_ms, seg_chunks = ctx.timer("seg")
    ctx.set_option("profile", 0)
    clocks = sampler.stop() if rank == 0 else None
    collective = None
    if use_pool:
        per_step = [ev[0].elapsed_time(ev[1]) for ev in coll_ms if ev is not None]
        t = torch.tensor([float(np.mean(per_step)) if per_step else 0.0], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        collective = {"op": ("fused: embedding GEMM epilogue pushes its tiles to every peer (P2P stores over NVLink, "
                             "symmetric memory) + P2P copy of the powerset classes + symmetric-memory barrier; "
                             "timed part = class copy + barrier (the embedding pushes are inside the GEMM)")
                      if pool.collective == "p2p" else
                      "ncclAllGather (in place, one packed buffer: embeddings f32 | powerset classes u8)",
                      "bytes_sent_per_rank": pool.last_collective["bytes_sent"],
                      "bytes_received_per_rank": pool.last_collective["bytes_received"],
                      "ms_per_step_max_over_ranks": float(t.item()),
                      "note": "event-timed on the launching stream: includes waiting for the slowest rank's compute"}
    files_done = torch.tensor([done[0]], device=dev)
    if world > 1:
        dist.all_reduce(files_done)
    assert int(files_done.item()) == world * nfiles, "every file must come out of the per-file stage exactly once"
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, last_outputs)
    ms_e2e = timed(step_e2e, max(1, args.steps))
    value = world * audio_hours / (ms_resident / 1e3)
    e2e = world * audio_hours / (ms_e2e / 1e3)
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    pk = peaks()
    peak = pk.get("bf16_tflops_sustained", 1400.0)
    achieved = trunk_segments * TRUNK_FLOP_PER_SEGMENT / (trunk_ms / 1e3) / 1e12 if trunk_ms > 0 else 0.0
    traffic, traffic_segments, traffic_src = trunk_traffic()
    sub_batch = traffic_segments or 296                    # segments of the launch unit (one embedding sub-batch)
    roofline = {"bound": "tensor",
                "kernel": "ResNet34 trunk = stem + tcgen05 conv kernels, one dependent chain per embedding sub-batch "
                          "(296 segments in the library, the launch unit below is the captured one)",
                "achieved": achieved, "peak": peak, "unit": "TFLOP/s", "frac": achieved / peak if peak else None,
                "traffic": traffic, "traffic_unit": f"bytes per {sub_batch}-segment trunk pass (ncu dram read+write)",
                "traffic_source": traffic_src,
                "algorithmic_flop_per_launch_unit": sub_batch * TRUNK_FLOP_PER_SEGMENT,
                "peak_source": "MEASURED_PEAKS.json bf16_tflops_sustained (fp16 = same tensor rate)"
                if pk else "fallback 1.4 PFLOP/s sustained",
                "trunk_ms_per_step": trunk_ms / args.steps, "seg_ms_per_step": seg_ms / args.steps}
    cpu = eager = None
    if world == 1 and not args.no_eager_baseline:
        eager = eager_cuda_baseline(args, dev)
    if args.gpus == 1 and not args.no_cpu_baseline:
        torch.set_num_threads(min(32, os.cpu_count() or 1))
        models = oracle_models()
        t, chunks = cpu_pass(args.cpu_sample_seconds, models)
        cpu = {"value": cpu_value(args, t, chunks), "unit": "audio-hours/sec", "cores": torch.get_num_threads(),
               "kind": "port", "sample": cpu_sample_text(args, t, chunks)}
    line = {"metric": METRIC, "value": value, "unit": "audio-hours/sec", "n_gpus": world, "steps": args.steps,
            "warmup": max(args.min_warmup, args.warmup), "ms_per_step": ms_resident, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f16 tensor-core trunk (f32 accumulate) + split-f16x3 tensor-core segmentation (f32-level accuracy) + f64 clustering",
            "data": "synthetic", "config": workload_config(args, world),
            "rtf": (ms_resident / 1e3) / (audio_hours * 3600.0) / world,
            "e2e": {"value": e2e, "unit": "audio-hours/sec", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h[0],
                    "ms_per_step": ms_e2e},
            "gpu_launches": int(launches), "clocks": clocks, "roofline": roofline, "cpu_baseline": cpu,
            "eager_cuda_baseline": eager, "collective": collective}
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
