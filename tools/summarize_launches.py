#!/usr/bin/env python
"""Summarise an ncu launch list (tools/ncu_frame.sh) into profiles/<tag>_launch_summary.md + igemm_traffic.json.

usage: python tools/summarize_launches.py gpurun_out/launches_<tag>.csv <tag>
One frame = the launches from one `lcm_step_kernel`... boundary: we take the window between two consecutive
`post_u8_kernel` launches (post_u8 is the last kernel of a frame).
"""
import csv, json, re, sys, collections

src, tag = sys.argv[1], sys.argv[2]
rows = collections.OrderedDict()
with open(src) as f:
    lines = [l for l in f if l.startswith('"')]
for r in csv.DictReader(lines):
    d = rows.setdefault(int(r["ID"]), {"name": r["Kernel Name"], "grid": r["Grid Size"]})
    d[r["Metric Name"]] = float(r["Metric Value"].replace(",", ""))
ids = sorted(rows)
ends = [i for i in ids if rows[i]["name"].startswith("post_u8_kernel")]
assert len(ends) >= 2, "need two frame boundaries in the capture"
frame = [rows[i] for i in ids if ends[-2] < i <= ends[-1]]


def short(n):
    return re.sub(r"\(.*", "", n)


agg = collections.OrderedDict()
for k in frame:
    a = agg.setdefault(short(k["name"]), dict(n=0, ns=0.0, rd=0.0, wr=0.0, tp=0.0))
    t = k["gpu__time_duration.sum"]
    a["n"] += 1; a["ns"] += t
    a["rd"] += k["dram__bytes_read.sum"]; a["wr"] += k["dram__bytes_write.sum"]
    a["tp"] += t * k.get("sm__pipe_tensor_cycles_active.avg.pct_of_peak_sustained_active", 0.0)
tot = sum(a["ns"] for a in agg.values())
out = [f"# ncu launch list summary -- one frame of `python bench.py --steps 2 --warmup 1` (SD-Turbo 512x512, T=1), {tag}", "",
       "`ncu --metrics gpu__time_duration.sum,dram__bytes_read.sum,dram__bytes_write.sum,sm__pipe_tensor_cycles_active... --clock-control none`;",
       f"per-launch times are cold-cache and serialised: compare SHARES, not absolutes.  Raw list: `{tag}_launches.csv`.", "",
       f"launches in the frame: {len(frame)}; sum of kernel durations: {tot/1e6:.3f} ms", "",
       "| kernel | launches | total us | share | DRAM read MB | DRAM write MB | avg tensor-pipe active % (time-weighted) |",
       "|---|---|---|---|---|---|---|"]
for n, a in sorted(agg.items(), key=lambda kv: -kv[1]["ns"]):
    out.append(f"| `{n}` | {a['n']} | {a['ns']/1e3:.1f} | {100*a['ns']/tot:.1f}% | {a['rd']/1e6:.1f} | {a['wr']/1e6:.1f} | {a['tp']/max(a['ns'],1):.1f} |")
fam = [agg[k] for k in ("igemm_kernel", "igemm_pair_kernel") if k in agg]   # one source (igemm_body<PAIR>): single CTAs / CTA pairs
ig = {k: sum(a[k] for a in fam) for k in ("n", "ns", "rd", "wr")}

per = (ig["rd"] + ig["wr"]) / ig["n"]
out += ["", f"igemm_kernel + igemm_pair_kernel: {ig['n']} launches/frame ({100*ig['ns']/tot:.1f}% of the summed kernel time), DRAM traffic "
        f"{(ig['rd']+ig['wr'])/1e6:.1f} MB/frame = {per/1e6:.2f} MB per launch (algorithmic minimum ~ weights once 1.73 GB + activations)."]
if "tconv_kernel" in agg:
    a = agg["tconv_kernel"]
    out += ["", f"tconv_kernel: {a['n']} launches/frame, DRAM traffic {(a['rd']+a['wr'])/1e6:.1f} MB/frame = {(a['rd']+a['wr'])/a['n']/1e6:.2f} MB per launch."]
open(f"profiles/{tag}_launch_summary.md", "w").write("\n".join(out) + "\n")
# the stored list ends with the summarised frame: the launches after it (the frame the capture stopped in) are dropped, which
# keeps the file under 1 MB
with open(src) as fi, open(f"profiles/{tag}_launches.csv", "w") as fo:
    fo.writelines(l for l in fi if not l.startswith('"') or l.startswith('"ID"') or int(next(csv.reader([l]))[0]) <= ends[-1])
json.dump({"dram_bytes_per_launch": per, "dram_bytes_per_frame": ig["rd"] + ig["wr"], "launches_per_frame": ig["n"],
           "note": f"igemm_kernel + igemm_pair_kernel, ncu dram__bytes_read.sum + dram__bytes_write.sum averaged over the launches of one SD-Turbo "
                   f"512x512 frame (profiles/{tag}_launches.csv)"}, open("profiles/igemm_traffic.json", "w"), indent=1)
print("\n".join(out))
