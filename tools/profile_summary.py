#!/usr/bin/env python
"""Turn the gpurun_out/<tag>_* artefacts of tools/prof_bench.sh into the tracked summaries under profiles/:
traffic.json (dram bytes per launch), the launch-list CSV and the ncu details text."""
import collections, csv, io, json, subprocess, sys
tag = sys.argv[1]
rep = f"gpurun_out/{tag}_full.ncu-rep"
raw = subprocess.run(["ncu", "-i", rep, "--page", "raw", "--csv"], capture_output=True, text=True).stdout
rows = list(csv.reader(io.StringIO(raw))); h, u = rows[0], rows[1]
f = {'Gbyte': 1e9, 'Mbyte': 1e6, 'Kbyte': 1e3, 'byte': 1}
t = {}
for v in rows[2:]:
    d = dict(zip(h, zip(u, v)))
    name = v[4].split('(')[0].replace('void ', '').strip()
    t[name] = int(float(d['dram__bytes_read.sum'][1]) * f[d['dram__bytes_read.sum'][0]] + float(d['dram__bytes_write.sum'][1]) * f[d['dram__bytes_write.sum'][0]])
    print(name, t[name], d['gpu__time_duration.sum'], 'issue %', d['smsp__issue_active.avg.pct_of_peak_sustained_active'][1],
          'dram %', d.get('gpu__dram_throughput.avg.pct_of_peak_sustained_elapsed', ('', ''))[1])
ev = next(v for k, v in t.items() if 'event_kernel' in k)
parts = {k: v for k, v in t.items() if 'event_kernel' not in k}
json.dump({"_source": f"ncu --set full, dram__bytes_read.sum + dram__bytes_write.sum per launch at the bench size (tools/prof_bench.sh, report {tag}_full, timed region); bytes",
           "c5": {"feature_kernel": sum(parts.values()), "statistics_pass": parts, "event_kernel": ev}}, open('profiles/traffic.json', 'w'), indent=1)
rows = list(csv.reader(open(f'gpurun_out/{tag}_launches.csv')))
i = next(k for k, r in enumerate(rows) if r and r[0] == 'ID')
hh = rows[i]; kn = hh.index('Kernel Name'); mv = hh.index('Metric Value')
seq = [(r[0], r[kn].split('(')[0].strip(), float(r[mv].replace(',', ''))) for r in rows[i + 1:] if len(r) > mv]
mlb = [x for x in seq if 'mlb::' in x[1]]
agg = collections.OrderedDict()
for _, n, tm in seq: agg.setdefault(n, []).append(tm)
timed = mlb[3 * 259:3 * 279]   # three launches per bench-size step
per = collections.OrderedDict()
for _, n, tm in timed: per.setdefault(n, []).append(tm)
tot = sum(sum(v) for v in per.values())
with open('profiles/r01_launches_four_kernel_step.csv', 'w') as fo:
    fo.write("# ncu --metrics gpu__time_duration.sum --clock-control none; python bench.py --steps 20 --warmup 3 --no-cpu --e2e-steps 2 (256 burn-in steps)\n")
    fo.write("# per-launch times are cold-cache and serialised: shares matter, not absolutes. A step = event_kernel + pair_kernel<.,2> (both statistics classes) + feature_kernel.\n")
    fo.write("# whole run (burn-in included: in the first steps after reset every touched reservoir is re-sorted by feature_kernel)\n")
    fo.write("kernel,launches,total_ms,mean_us\n")
    for k, v in agg.items(): fo.write(f"\"{k[:80]}\",{len(v)},{sum(v)/1e6:.3f},{sum(v)/len(v)/1e3:.1f}\n")
    fo.write("# timed region only (20 steps after 256 burn-in + 3 warm-up): kernel,mean_us,share_of_step\n")
    for k, v in per.items(): fo.write(f"\"{k}\",{sum(v)/len(v)/1e3:.1f},{sum(v)/tot:.3f}\n")
    fo.write("# per-launch rows of the timed region: id,kernel,duration_ns\n")
    for i_, k, tm in timed: fo.write(f"{i_},{k},{tm:.0f}\n")
det = subprocess.run(["ncu", "-i", rep, "--page", "details"], capture_output=True, text=True).stdout
keep = [l for l in det.splitlines() if l.strip() and not l.lstrip().startswith(("INF", "OPT", "---"))]
open('profiles/r01_four_kernel_step_ncu_full_details.txt', 'w').write("\n".join(keep[:300]) + "\n")
print(''.join(open('profiles/r01_launches_four_kernel_step.csv').readlines()[12:18]))
