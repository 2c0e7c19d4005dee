"""Turn gpurun_out/ captures into the tracked summaries under profiles/.
usage: make_profiles.py TAG launches.csv step.ncu-rep"""
import csv, json, re, subprocess, sys
tag, launches, rep = sys.argv[1], sys.argv[2], sys.argv[3]
# ---- 1. launch list of one bench step (from one zero-fill of the accumulator block to the next)
rows = list(csv.reader(open(launches)))
hdr = [i for i, r in enumerate(rows) if r and r[0] == 'ID'][0]
H = rows[hdr]; ki = H.index('Kernel Name'); vi = H.index('Metric Value')
L = [(r[ki], float(r[vi]) / 1e3) for r in rows[hdr + 1:] if len(r) > vi]
fin = [i for i, (k, v) in enumerate(L) if 'FillFunctor<float>' in k]
a, b = fin[-2], fin[-1]
tot = sum(v for k, v in L[a:b])
open(f'profiles/{tag}_launch_list.csv', 'w').write("us,kernel\n" + "\n".join(f"{v:.1f},\"{k}\"" for k, v in L[a:b]) + "\n")
md = [f"# {tag}: every launch of ONE bench step (cfg2 G-A, B=16, C=150), `ncu --metrics gpu__time_duration.sum --clock-control none`", "",
      "command: `python bench.py --steps 3 --warmup 3 --no-e2e --no-cpu-baseline` (per-launch times are cold-cache and serialised: compare shares;",
      "in-situ section times of the same step are in the bench line's `section_us` with `--kernel-times`)", "",
      "| us | share | kernel |", "|---:|---:|---|"]
md += [f"| {v:.1f} | {v / tot * 100:.1f}% | `{k[:110]}` |" for k, v in L[a:b]]
md += ["", f"sum = {tot:.1f} us over {b - a} launches"]
open(f'profiles/{tag}_launch_list.md', 'w').write("\n".join(md) + "\n")
# ---- 2. ncu --set full summaries
out = subprocess.run(["ncu", "-i", rep, "--page", "raw", "--csv"], capture_output=True, text=True).stdout
rr = list(csv.reader(out.splitlines())); h, units = rr[0], rr[1]
mul = {"byte": 1, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}
traffic = {}
for r in rr[2:]:
    nm = r[h.index("Kernel Name")].split("(")[0].replace("void ", "").strip()
    ir, iw = h.index("dram__bytes_read.sum"), h.index("dram__bytes_write.sum")
    traffic[nm] = int(float(r[ir]) * mul[units[ir]] + float(r[iw]) * mul[units[iw]])
summ = subprocess.run([sys.executable, "tools/ncu_summary.py", rep], capture_output=True, text=True).stdout
src = subprocess.run(["ncu", "-i", rep, "--page", "source", "--csv"], capture_output=True, text=True).stdout
kern = None; h2 = None; data = {}; hdrs = {}
for r in csv.reader(src.splitlines()):
    if r and r[0] == "Kernel Name": kern = r[1]; data[kern] = []; continue
    if r and r[0] == "Address": h2 = r; hdrs[kern] = r; continue
    if h2 and len(r) == len(h2) and kern: data[kern].append(r)
def opmix(d, h2):
    ix = {k: i for i, k in enumerate(h2)}          # (the column set differs from kernel to kernel)
    ti = sum(int(r[ix["Instructions Executed"]]) for r in d); o = {}
    for r in d:
        t = r[ix["Source"]].split(); op = t[1] if t and t[0].startswith("@") else (t[0] if t else "?")
        o[op] = o.get(op, 0) + int(r[ix["Instructions Executed"]])
    lines = [f"total {ti}"] + [f"{n / ti * 100:5.1f}% {n:11d}  {op}" for op, n in sorted(o.items(), key=lambda kv: -kv[1])[:18]]
    st = {}
    for s_ in [c for c in h2 if c.startswith("stall_") and "Not" not in c]:
        st[s_[6:]] = sum(int(r[ix[s_]]) for r in d)
    t = sum(st.values()) or 1
    return "\n".join(lines + ["", "warp-state samples: " + ", ".join(f"{k} {v / t * 100:.1f}%" for k, v in sorted(st.items(), key=lambda kv: -kv[1])[:8])])
names = {"k23_rc": "k23rc", "k1_logits": "k1", "k1b_dv": "k1bdv", "k1b_dt_kernel": "k1bdt", "k2_strip": "k2", "k3_strip": "k3strip", "prepass": "prepass", "prep_f32": "k1bprep", "pack_labels": "packlabels"}
for blk in summ.split("-" * 60):
    m = re.search(r"Kernel Name = (.*)", blk)
    if not m: continue
    kn = m.group(1); key = [v for k, v in names.items() if k in kn]
    if not key: continue
    dk = [k for k in data if k.split("(")[0].split("::")[-1].split("<")[0] in kn][0]
    open(f"profiles/{tag}_{key[0]}_ncu_full.txt", "w").write(
        f"# {tag} {key[0]}: ncu --set full --clock-control none --import-source on (one launch inside the step: "
        f"`python tools/run_one.py step A 16`, cfg2 G-A B=16 C=150)\n\n## metrics\n{blk.strip()}\n\n## executed SASS opcodes\n{opmix(data[dk], hdrs[dk])}\n")
try: tj = json.load(open("profiles/traffic.json"))
except Exception: tj = {}
tj["note"] = "dram__bytes_read.sum + dram__bytes_write.sum per launch, ncu --set full, cfg2 G-A B=16 C=150 (profiles/*_ncu_full.txt)"
for k, v in traffic.items():
    if "k23_rc" in k: tj["k23_rc_kernel<16>"] = v
    elif "pack_labels" in k: tj["k2_pack_labels_kernel"] = v
    elif "prep_f32" in k: tj["k1b_prep_f32_kernel"] = v
json.dump(tj, open("profiles/traffic.json", "w"), indent=1)
print(open(f'profiles/{tag}_launch_list.md').read()); print(tj)
