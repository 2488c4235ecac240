#!/usr/bin/env python
"""Builds profiles/README.md and profiles/ncu_traffic.json from the measurement files of the current round
(profiles/r02_*; gathered on the B200 box by tools/gpu_measure_r02.sh and the bench.py runs named below).
Round-1 files stay in profiles/ under their r01_ names."""
import csv
import json
import re
from pathlib import Path

P = Path(__file__).resolve().parent.parent / "profiles"
R = "r02"


def load_json(name):
    f = P / name
    if not f.exists():
        return None
    lines = [l for l in f.read_text().splitlines() if l.strip().startswith("{")]
    return json.loads(lines[-1]) if lines else None


def ncu_rows(name):
    f = P / name
    if not f.exists():
        return None, None
    rows = list(csv.reader(f.open()))
    return rows[0], rows[1:]


def col(hdr, prefix):
    return [i for i, n in enumerate(hdr) if n.startswith(prefix)][0]


_SCALE = {"ns": 1e-3, "us": 1.0, "ms": 1e3, "s": 1e6,                      # -> microseconds
          "byte": 1e-6, "Kbyte": 1e-3, "Mbyte": 1.0, "Gbyte": 1e3}          # -> megabytes


def val(hdr, row, i):
    """Cell i of an ncu raw-page row in canonical units (us / MB): ncu picks the unit per report, e.g. [ms] or [us]."""
    m = re.search(r"\[(\w+)\]", hdr[i])
    return float(row[i]) * _SCALE.get(m.group(1), 1.0) if m else float(row[i])


def kernel_name(s):
    m = re.search(r"(\w+_kernel(?:<[^>]*>)?)", s)
    return m.group(1) if m else s[:60]


def main():
    out = []
    w = out.append
    bench = load_json(f"{R}_bench.json")
    prof = json.loads((P / f"{R}_launch_profile.json").read_text())
    w("# profiles — round 2 (B200, sm_100a)\n")
    w("All numbers were produced on the pool's B200 boxes through `gpurun`. Timed numbers come from CUDA events "
      "(bench.py / tools/*.py); ncu numbers are cold-cache, serialised replays and are used for SHARES, tensor-pipe "
      "activity and DRAM traffic only. Round-1 files keep their `r01_` names.\n")
    rf, e2e, cpu, ck = bench["roofline"], bench["e2e"], bench["cpu_baseline"], bench["clocks"]
    w(f"## Headline (`{R}_bench.json` = `python bench.py --steps 20 --warmup 3`)\n")
    w("| quantity | value |\n|---|---|")
    w(f"| workload | {bench['config']['workload']}, {bench['config']['pairs_per_step']} pairs per step |")
    w(f"| `value` (device-timed, inputs in HBM, profiling off) | **{bench['value']:.1f} frames/s** ({bench['ms_per_step']:.2f} ms per step) |")
    w(f"| `e2e` (`FrameInterpolator(...).interpolate_clip`: 600 host u8 frames -> 599 host u8 midpoints) | **{e2e['value']:.1f} frames/s** ({e2e['seconds']:.3f} s) |")
    w(f"| per-rank clip call (round-1 e2e definition) | {e2e['per_rank_clip_call_weak']['value']:.1f} frames/s |")
    w(f"| whole-step arithmetic rate | {rf['whole_step_tflops']:.0f} TFLOP/s |")
    w(f"| tcgen05 conv launches ({rf['share_of_step']*100:.1f} % of the step, separate profiled pass) | {rf['achieved']:.0f} TFLOP/s = "
      f"**{rf['frac']*100:.1f} %** of the measured burst bf16 peak ({rf['peak']:.0f}), {rf['frac_sustained']*100:.1f} % of the sustained one ({rf['peak_sustained']:.0f}) |")
    w(f"| DRAM traffic / algorithmic bytes per conv launch | {rf['traffic']/1e6:.0f} MB / {rf['algorithmic_bytes']/1e6:.0f} MB |")
    w(f"| clocks during the timed region | {ck['sm_mhz']:.0f} MHz median of {ck['sm_max_mhz']:.0f}, reasons {ck['reasons']} |")
    if cpu:
        w(f"| CPU baseline ({cpu['kind']}: unmodified reference module, {cpu['cores']} host cores) | {cpu['value']:.3f} frames/s |")
    ref = load_json(f"{R}_ref.json")
    if ref:
        w(f"| `bench.py --impl reference` ({ref['cpu_baseline']['kind']}, {ref['cpu_baseline']['cores']} cores, same config) | {ref['value']:.3f} frames/s |")
    w("")
    sc = P / f"{R}_scaling.jsonl"
    if sc.exists():
        rows = [json.loads(l) for l in sc.read_text().splitlines() if l.strip().startswith("{")]
        w(f"## Scaling (`{R}_scaling.jsonl`: `torchrun --nproc-per-node N bench.py --gpus N --steps 20 --warmup 3`)\n")
        w("`value`: one process per GPU, each on its shard of the clip (weak). `e2e`: rank 0 drives all N GPUs through "
          "`FrameInterpolator(gpus=N).interpolate_clip` on the fixed 600-frame host clip (strong).\n")
        w("| GPUs | value frames/s | x of 1 GPU | e2e frames/s (599 pairs) | seconds | x of 1 GPU |\n|---|---|---|---|---|---|")
        for r in rows:
            w(f"| {r['n_gpus']} | {r['value']:.0f} | {r['value']/rows[0]['value']:.2f} | {r['e2e']['value']:.0f} | "
              f"{r['e2e']['seconds']:.3f} | {r['e2e']['value']/rows[0]['e2e']['value']:.2f} |")
        w("")
    w(f"## Per-launch table (`{R}_launch_profile.json`, CUDA events around every launch in a separate profiled pass, "
      f"{bench['config']['pairs_per_step']} pairs per launch)\n")
    w("| launch | kernel | ms | TFLOP/s | algorithmic GB/s | share |\n|---|---|---|---|---|---|")
    tot = sum(p["ms_total"] for p in prof)
    for p in prof:
        ms = p["ms_total"] / p["calls"]
        kind = {0: "stem_mma", 1: "tcgen05 conv", 2: "upsample"}[p["kind"]]
        w(f"| {p['name']} | {kind} | {ms:.3f} | {p['flops']/ms/1e9:.0f} | {p['bytes']/ms/1e6:.0f} | {p['ms_total']/tot*100:.1f} % |")
    w(f"| **total** | | **{tot/prof[0]['calls']:.2f}** | | | |")
    w("")
    h, rows = ncu_rows(f"{R}_kernels_ncu_full.csv")
    if h:
        w(f"## ncu, one forward at 1 pair (`{R}_kernels_ncu_full.csv`: `--set full`; `{R}_launches_ncu.csv`: launch list of "
          "`bench.py --steps 2 --warmup 1`)\n")
        ik, it, ir, iw = col(h, "Kernel Name"), col(h, "gpu__time_duration"), col(h, "dram__bytes_read"), col(h, "dram__bytes_write")
        itn = col(h, "sm__pipe_tensor_cycles_active.avg.pct_of_peak_sustained_active")
        il2, idr = col(h, "lts__t_sector_hit_rate"), col(h, "gpu__dram_throughput")
        w("| # | kernel | us | DRAM read MB | DRAM write MB | DRAM % of peak | tensor pipe active % | L2 hit % |\n|---|---|---|---|---|---|---|---|")
        dram, n_conv = 0.0, 0
        for i, r in enumerate(rows):
            name = kernel_name(r[ik])
            w(f"| {i} | `{name}` | {val(h, r, it):.1f} | {val(h, r, ir):.1f} | {val(h, r, iw):.1f} | {float(r[idr]):.0f} | {float(r[itn]):.1f} | {float(r[il2]):.1f} |")
            if "stem" not in name:
                dram += (val(h, r, ir) + val(h, r, iw)) * 1e6
                n_conv += 1
        algo = sum(p["bytes"] for p in prof if p["kind"] == 1) / bench["config"]["pairs_per_step"]
        w("")
        w(f"DRAM traffic of the {n_conv} tcgen05 conv launches of one forward (1 pair): **{dram/1e9:.2f} GB** measured vs "
          f"{algo/1e9:.2f} GB algorithmic (every activation/weight touched once).\n")
        (P / "ncu_traffic.json").write_text(json.dumps({"source": f"{R}_kernels_ncu_full.csv", "pairs": 1,
                                                        "conv_launches": n_conv, "dram_bytes": dram,
                                                        "algorithmic_bytes": algo}, indent=1))
    aux_f = P / f"{R}_aux_kernels.jsonl"
    if aux_f.exists():
        aux = [json.loads(l) for l in aux_f.read_text().splitlines() if l.strip()]
        w(f"## Non-GEMM kernels (`{R}_aux_kernels.jsonl` = `python tools/bench_aux.py`, CUDA events)\n")
        w("A write-only stream reaches 3.9 TB/s on this GPU against 6.45 TB/s for a 1:1 copy (`r01_bw_probe.txt`), so a "
          "kernel reading R and writing W bytes is bounded by max((R+W)/copy peak, W/3.9 TB/s); the last column is the "
          "measured time against that bound.\n")
        w("| kernel | ms | achieved GB/s | of HBM copy peak | write share | of the read/write-mix bound | note |\n|---|---|---|---|---|---|---|")
        write_share = {"pack_pair_u8": 8 / 10, "head_post_u8": 1 / 5, "upsample2x_bilinear": 4 / 5,
                       "stem_conv (tcgen05, hi/lo split)": 128 / 130}
        for a in aux:
            ws = write_share.get(a["kernel"], 0.0)
            total = a["algorithmic_bytes"]
            bound_ms = max(total / (a["hbm_peak_gbs"] * 1e6), ws * total / (3900.0 * 1e6))
            w(f"| {a['kernel']} | {a['ms']} | {a['achieved_gbs']} | {a['frac_of_hbm_peak']*100:.1f} % | {ws*100:.0f} % | "
              f"{bound_ms / a['ms'] * 100:.0f} % | {a['note']} |")
        w("")
    for title, name in (("Non-GEMM kernels under ncu", f"{R}_aux_ncu_full.csv"),
                        ("Training kernels under ncu, forward BatchNorm (one eager step, batch 16 x 256²)",
                         f"{R}_train_ncu_full.csv"),
                        ("Training kernels under ncu, weight gradient and BatchNorm backward (same step)",
                         f"{R}_train_bwd_ncu_full.csv")):
        h, rows = ncu_rows(name)
        if not h:
            continue
        w(f"## {title} (`{name}`, `--set full`, one launch each)\n")
        ik, it, ir, iw = col(h, "Kernel Name"), col(h, "gpu__time_duration"), col(h, "dram__bytes_read"), col(h, "dram__bytes_write")
        idr, itn = col(h, "gpu__dram_throughput"), col(h, "sm__pipe_tensor_cycles_active.avg.pct_of_peak_sustained_active")
        ism = col(h, "sm__throughput")
        w("| kernel | us | DRAM read MB | DRAM write MB | DRAM GB/s | DRAM % of peak | SM % | tensor pipe % |\n|---|---|---|---|---|---|---|---|")
        seen = {}
        for r in rows:
            name_k = kernel_name(r[ik])
            us = val(h, r, it)
            key = (name_k, round(us, -1))
            if "train" in name:   # keep the largest launch of every kernel
                if name_k in seen and seen[name_k][0] >= us:
                    continue
                seen[name_k] = (us, r)
                continue
            gbs = (val(h, r, ir) + val(h, r, iw)) * 1e6 / (us * 1e-6) / 1e9
            w(f"| `{name_k}` | {us:.1f} | {val(h, r, ir):.1f} | {val(h, r, iw):.1f} | {gbs:.0f} | {float(r[idr]):.0f} | {float(r[ism]):.0f} | {float(r[itn]):.1f} |")
        for name_k, (us, r) in seen.items():
            gbs = (val(h, r, ir) + val(h, r, iw)) * 1e6 / (us * 1e-6) / 1e9
            w(f"| `{name_k}` (largest launch) | {us:.1f} | {val(h, r, ir):.1f} | {val(h, r, iw):.1f} | {gbs:.0f} | {float(r[idr]):.0f} | {float(r[ism]):.0f} | {float(r[itn]):.1f} |")
        w("")
    for name, title in ((f"{R}_small_profile.json", "ConvTranspose2d decoder"), (f"{R}_small_profile_bilinear.json", "bilinear decoder")):
        f = P / name
        if f.exists():
            d = json.loads(f.read_text())
            w(f"## One {d['shape'][1]}x{d['shape'][2]} pair, {title} (`{name}` = `python tools/profile_small.py`)\n")
            w(f"Forward, back to back with programmatic dependent launch: **{d['forward_ms_back_to_back']} ms**; sum of the "
              f"serialised per-launch times: {d['sum_of_serialised_launches_ms']} ms.\n")
            w("| launch | us | TFLOP/s |\n|---|---|---|")
            for r in d["launches"]:
                w(f"| {r['launch']} | {r['us']} | {r['tflops']} |")
            w("")
    w("## Other workloads (same JSON schema as the headline line)\n")
    for name, cmd in ((f"{R}_api256.json", "python bench.py --workload api256"),
                      (f"{R}_4k_eval.json", "python bench.py --workload 4k_eval --steps 10"),
                      (f"{R}_train1.json", "python bench.py --workload train"),
                      (f"{R}_train2.json", "torchrun --nproc-per-node 2 bench.py --gpus 2 --workload train"),
                      (f"{R}_train_8gpu.json", "torchrun --nproc-per-node 8 bench.py --gpus 8 --workload train"),
                      (f"{R}_4k_eval_2gpu.json", "torchrun --nproc-per-node 2 bench.py --gpus 2 --workload 4k_eval --steps 10"),
                      (f"{R}_4k_eval_8gpu.json", "torchrun --nproc-per-node 8 bench.py --gpus 8 --workload 4k_eval --steps 10")):
        d = load_json(name)
        if d:
            e = d.get("e2e") or {}
            w(f"* `{name}` = `{cmd}`: **{d['value']:.1f} {d['unit']}** ({d['ms_per_step']:.3f} ms per step, {d['n_gpus']} GPU(s)); "
              f"e2e {e.get('value', float('nan')):.1f} {e.get('unit', '')}; whole-step {d['roofline']['achieved']:.0f} TFLOP/s "
              f"= {d['roofline']['frac']*100:.0f} % of the burst peak. {d['config']['workload']}.")
    w("")
    vid = load_json(f"{R}_video_path.json")
    if vid:
        w(f"File-to-file video path (`{R}_video_path.json` = `python tools/bench_video.py`, {vid['clip']}, {vid['host_cores']} host "
          f"cores): cv2 decode {vid['decode_frames_per_s']} frames/s, cv2 `mp4v` encode {vid['encode_frames_per_s']} frames/s, GPU "
          f"stage on decoded BGR frames (grey model: 3 forwards per new frame, planes split / merged on the host) "
          f"{vid['gpu_stage_new_bgr_frames_per_s']} new frames/s; `interpolate_video` end to end "
          f"{vid['interpolate_video_output_frames_per_s']} output frames/s — bound by the software encoder, which the three "
          "pipelined stages hide everything else behind.\n")
    pp = [(k, load_json(f"{R}_bench_p{k}.json")) for k in (4, 6, 8)]
    if all(d for _, d in pp):
        w("Pairs per forward (`bench.py --pairs K`): " + ", ".join(f"K={k}: {d['value']:.1f} frames/s" for k, d in pp) + ".\n")
    notes = [(f"{R}_fused_inc.md", "fused `inc` kernel: ncu source-page reading (per-role wait shares, shared-memory port)"),
             (f"{R}_rows.md", "row-stacked conv kernel (removed kernel, commit c63f920): parity-green, measured slower than the halo kernels, why"),
             ("sass_summary.txt", "opcode counts per kernel from `cuobjdump -sass` (tcgen05 MMA, TMA, TMEM, PDL; no legacy HMMA)"),
             ("ncu_traffic.json", "DRAM bytes per conv launch from the `--set full` capture (the `roofline.traffic` source of bench.py)")]
    notes = [(f, t) for f, t in notes if (P / f).exists()]
    if notes:
        w("## Kernel write-ups and evidence files\n")
        for f, t in notes:
            w(f"* `{f}` — {t}")
        w("")
    (P / "README.md").write_text("\n".join(out) + "\n")
    print("\n".join(out)[:2500])


if __name__ == "__main__":
    main()
