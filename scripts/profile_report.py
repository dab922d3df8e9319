"""Turns the two ncu captures of `bench.py --no-graph` into the committed summaries under profiles/ (development aid).

  python scripts/profile_report.py launches gpurun_out/launches.csv            -> markdown table of one step (kernel, launches, us, share)
  python scripts/profile_report.py metrics  gpurun_out/full.ncu-rep out.json   -> per-kernel DRAM bytes / time / pipe utilisation (+ per-call traffic)

The launch list comes from `ncu --metrics gpu__time_duration.sum --clock-control none --csv --log-file ...`, the metrics from one
`ncu --set full --clock-control none` capture; both are cold-cache and serialised, so only SHARES and per-launch bytes are comparable
with the graph-replayed step.
"""
import collections
import csv
import io
import json
import re
import subprocess
import sys


def short(name):
    name = re.sub(r"\(.*$", "", name)                       # drop the argument list
    name = name.replace("void ", "").replace("crf::", "").replace("(int)", "")
    return name.strip()


def launches(path):
    rows = [r for r in csv.reader(l for l in open(path) if l.startswith('"'))]
    hdr, rows = rows[0], rows[1:]
    iK, iV = hdr.index("Kernel Name"), hdr.index("Metric Value")
    seq = [(short(r[iK]), float(r[iV].replace(",", "")) / 1e3) for r in rows]
    # one step = the span between two consecutive occurrences of the first kernel of the forward pass (two steps are captured)
    names = [n for n, _ in seq]
    # find the period: smallest p such that the last 2p launches repeat
    period = None
    for p in range(20, len(seq) // 2 + 1):
        if names[-p:] == names[-2 * p:-p]:
            period = p
            break
    step = seq[-period:] if period else seq
    agg = collections.OrderedDict()
    for n, us in step:
        a = agg.setdefault(n, [0, 0.0])
        a[0] += 1
        a[1] += us
    tot = sum(v[1] for v in agg.values())
    print(f"kernels per step: {len(step)}; summed device time (cold-cache, serialised): {tot:.1f} us\n")
    print("| kernel | launches/step | us/step | share |\n|---|---|---|---|")
    for n, (c, us) in sorted(agg.items(), key=lambda kv: -kv[1][1]):
        print(f"| `{n[:80]}` | {c} | {us:.1f} | {100 * us / tot:.1f}% |")


KEYS = {
    "time_us": "gpu__time_duration.sum",
    "dram_read_mb": "dram__bytes_read.sum",
    "dram_write_mb": "dram__bytes_write.sum",
    "issue_active_pct": "smsp__issue_active.avg.pct_of_peak_sustained_active",
    "tensor_pipe_pct": "sm__pipe_tensor_cycles_active.avg.pct_of_peak_sustained_active",
    "l1tex_pct": "l1tex__throughput.avg.pct_of_peak_sustained_active",
    "lts_pct": "lts__throughput.avg.pct_of_peak_sustained_elapsed",
    "dram_pct": "dram__cycles_active.avg.pct_of_peak_sustained_elapsed",
    "regs": "launch__registers_per_thread",
    "warps_active_pct": "sm__warps_active.avg.pct_of_peak_sustained_active",
}


def metrics(rep, out):
    txt = subprocess.run(["ncu", "-i", rep, "--page", "raw", "--csv"], capture_output=True, text=True).stdout
    rows = list(csv.reader(io.StringIO(txt)))
    hdr, units, rows = rows[0], rows[1], rows[2:]
    ks = collections.OrderedDict()
    order = []
    seen = {}
    for r in rows:
        d = dict(zip(hdr, r))
        n = short(d["Kernel Name"]) + " grid=" + d.get("Grid Size", "").replace(" ", "")
        m = {}
        for k, col in KEYS.items():
            if col in d and d[col] not in ("", "n/a"):
                v = float(d[col].replace(",", ""))
                u = units[hdr.index(col)]
                if k == "time_us":
                    v = v / 1e3 if u in ("ns", "nsecond") else (v * 1e3 if u in ("ms", "msecond") else v)
                if k in ("dram_read_mb", "dram_write_mb"):
                    v = {"byte": v / 1e6, "Kbyte": v / 1e3, "Mbyte": v, "Gbyte": v * 1e3}.get(u, v)
                m[k] = round(v, 3)
        order.append((n, m))
        seen[n] = seen.get(n, 0) + 1
        ks[n + f" #{seen[n]}"] = m                           # every captured launch, numbered per (kernel, grid)
    calls = {}

    def first(sub):
        for n, m in order:
            if sub in n:
                return m
        return None
    # linear_bwd[64<-128] (fusion layer, first Linear backward of the step) = its dgrad + its wgrad launch
    dg, wg = first("dgrad2_kernel<128"), first("wgrad3_kernel<64") or first("wgrad2_kernel<64, 128")
    if dg and wg:
        calls["linear_bwd[64<-128]"] = {"traffic_bytes": round((dg["dram_read_mb"] + dg["dram_write_mb"] + wg["dram_read_mb"] + wg["dram_write_mb"]) * 1e6)}
    sb = first("step_bwd_reg_kernel")
    if sb:
        calls["crf_step_bwd[16]"] = {"traffic_bytes": round((sb["dram_read_mb"] + sb["dram_write_mb"]) * 1e6)}
    fw = first("fwd3_kernel<64")
    if fw:
        calls["linear_fwd[16->64]"] = {"traffic_bytes": round((fw["dram_read_mb"] + fw["dram_write_mb"]) * 1e6)}
    json.dump({"source": "ncu --set full --clock-control none, profiles/README_r01.md (scripts/profile_report.py)", "kernels": ks, "calls": calls},
              open(out, "w"), indent=1)
    print("| kernel (grid) | us | DRAM rd MB | DRAM wr MB | DRAM % | L2 % | L1TEX % | issue % | tensor % | regs |\n|---|---|---|---|---|---|---|---|---|---|")
    for n, m in ks.items():
        print(f"| `{n[:70]}` | {m.get('time_us', 0):.1f} | {m.get('dram_read_mb', 0):.1f} | {m.get('dram_write_mb', 0):.1f} | {m.get('dram_pct', 0):.0f} | "
              f"{m.get('lts_pct', 0):.0f} | {m.get('l1tex_pct', 0):.0f} | {m.get('issue_active_pct', 0):.0f} | {m.get('tensor_pipe_pct', 0):.0f} | {int(m.get('regs', 0))} |")


# ---- `ncu --set full --csv --page raw --log-file x.csv` (no .ncu-rep: they exceed gpurun's 64 MiB return limit)
CSV_KEYS = [("us", ["gpu__time_duration.sum"]), ("rd_MB", ["dram__bytes_read.sum"]), ("wr_MB", ["dram__bytes_write.sum"]),
            ("dram%", ["gpu__dram_throughput.avg.pct_of_peak_sustained_elapsed"]),
            ("L2%", ["lts__throughput.avg.pct_of_peak_sustained_elapsed"]),
            ("L1TEX%", ["l1tex__throughput.avg.pct_of_peak_sustained_elapsed"]),
            ("lsu_wavefronts%", ["l1tex__data_pipe_lsu_wavefronts.avg.pct_of_peak_sustained_elapsed"]),
            ("issue%", ["smsp__issue_active.avg.pct_of_peak_sustained_active", "sm__inst_executed_realtime.avg.pct_of_peak_sustained_elapsed"]),
            ("tensor%", ["sm__pipe_tensor_cycles_active_realtime.avg.pct_of_peak_sustained_elapsed"]),
            ("regs", ["launch__registers_per_thread"]), ("grid", ["launch__grid_size"]),
            ("L1 hit%", ["l1tex__t_sector_hit_rate.pct"]), ("L2 hit%", ["lts__t_sector_hit_rate.pct"])]


def metrics_csv(path, out_json=None, skip_prefixes=("at::", "knn::")):
    rows = [r for r in csv.reader(l for l in open(path) if l.startswith('"'))]
    hdr, units, rows = rows[0], rows[1], rows[2:]

    def col(names):
        for n in names:
            for i, h in enumerate(hdr):
                if h == n or h.endswith("." + n):
                    return i
        return None
    cols = [(k, col(v)) for k, v in CSV_KEYS]
    iK = hdr.index("Kernel Name")
    table, total_dram = [], 0.0
    for r in rows:
        name = short(r[iK])
        rec = {"kernel": name}
        for k, i in cols:
            if i is None or r[i] in ("", "n/a", "no data"):
                continue
            try:
                v = float(r[i].replace(",", ""))
            except ValueError:
                continue
            u = units[i]
            if k == "us":
                v = v / 1e3 if u in ("ns", "nsecond") else (v * 1e3 if u in ("ms", "msecond") else v)
            if k in ("rd_MB", "wr_MB"):
                v = {"byte": v / 1e6, "Kbyte": v / 1e3, "Mbyte": v, "Gbyte": v * 1e3}.get(u, v)
            rec[k] = round(v, 2)
        table.append(rec)
    keep = [t for t in table if not t["kernel"].startswith(skip_prefixes)]
    print("| kernel | " + " | ".join(k for k, _ in CSV_KEYS) + " |\n|---|" + "---|" * len(CSV_KEYS))
    for t in keep:
        print(f"| `{t['kernel'][:60]}` | " + " | ".join(str(t.get(k, "")) for k, _ in CSV_KEYS) + " |")
    step = [t for t in table if not t["kernel"].startswith("knn::")]
    tot_us = sum(t.get("us", 0) for t in keep)
    tot_mb = sum(t.get("rd_MB", 0) + t.get("wr_MB", 0) for t in keep)
    print(f"\nlayer kernels: {len(keep)}; summed time {tot_us:.1f} us; DRAM traffic {tot_mb:.1f} MB (read + write)")
    if out_json:
        # bench.py's call labels → DRAM bytes (read + write) of the kernel(s) behind them, per launch
        call_of = {"cl::step_bwd_kernel": "crf_step_bwd_fused", "mf::step_fwd_kernel<16>": "crf_step_fwd[16]", "cl::out_bwd_kernel": "out16_bwd",
                   "lin3::fwd3_kernel<64>": "linear_fwd_bn[128->64]", "cl::up16_fwd_kernel<64>": "up16_fwd[64]",
                   "lin::bn_bwd_reduce_kernel": "bn_bwd_reduce_fin[64]", "lin3d::dgrad3_kernel<128>": "linear_bwd[64<-128]:dgrad",
                   "lin3w::wgrad3_kernel<64>": "linear_bwd[64<-128]:wgrad", "lin3b::bwd3_kernel": "linear_bwd[64<-128]",
                   "lin::bn_act_fwd_kernel": "bn_act_fwd[64]"}
        calls = {}
        for t in keep:
            for kname, label in call_of.items():
                if t["kernel"].startswith(kname) and label not in calls:
                    calls[label] = round((t.get("rd_MB", 0) + t.get("wr_MB", 0)) * 1e6)
        json.dump({"source": f"ncu --set full --clock-control none --csv --page raw ({path})", "kernels": keep,
                   "step_dram_bytes": round(tot_mb * 1e6), "step_sum_us": round(tot_us, 1), **calls}, open(out_json, "w"), indent=1)



if __name__ == "__main__":
    if sys.argv[1] == "launches":
        launches(sys.argv[2])
    elif sys.argv[1] == "csv":
        metrics_csv(sys.argv[2], sys.argv[3] if len(sys.argv) > 3 else None)
    else:
        metrics(sys.argv[2], sys.argv[3])
