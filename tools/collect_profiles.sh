#!/bin/bash
# Copies the round-end measurement set (tools/final_runs.sh output) into profiles/ under a round tag and writes
# the derived summaries.  Usage: bash tools/collect_profiles.sh gpurun_out/final2 r02
set -eu
src=$1; tag=$2
for f in default exact profile_train scannet scannet448 kitti376x4 reference_arm short; do
  [ -s $src/bench_$f.json ] && cp $src/bench_$f.json profiles/${tag}_bench_$f.json
done
[ -s $src/bench_ops.json ] && cp $src/bench_ops.json profiles/${tag}_bench_ops_b24_192x640.json
cp $src/pytest_gpu.txt profiles/${tag}_pytest_gpu.txt
cp $src/smoke.txt profiles/${tag}_smoke.txt
for a in fast exact; do
  cp $src/launches_$a.csv profiles/${tag}_ncu_launches_$a.csv
  python tools/ncu_summary.py $src/prof_${a}_raw.csv > profiles/${tag}_ncu_pair_kernels_summary_$a.txt
  python tools/ncu_source_hot.py $src/prof_${a}_src.csv 30 > profiles/${tag}_ncu_pair_kernels_hot_lines_$a.txt
done
cp $src/launches_bench.csv profiles/${tag}_ncu_launches_bench_py.csv
cp $src/launches_pft_hotpath.csv profiles/${tag}_ncu_launches_pft_hotpath.csv
python - $src $tag <<'PY'
import collections, csv, json, sys
src, tag = sys.argv[1], sys.argv[2]

def launches(path):
    rows = list(csv.reader(open(path)))
    h = next(i for i, r in enumerate(rows) if "Kernel Name" in r)
    idx = {k: i for i, k in enumerate(rows[h])}
    return [(r[idx["Kernel Name"]], float(r[idx["Metric Value"]].replace(",", ""))) for r in rows[h + 1:] if len(r) >= len(rows[h])]

def summary(path, out, title):
    seq = launches(path)
    agg, tot = collections.OrderedDict(), 0.0
    for k, v in seq:
        a = agg.setdefault(k[:90], [0, 0.0]); a[0] += 1; a[1] += v; tot += v
    with open(out, "w") as f:
        f.write("%s\n%d launches, %.3f ms of kernel time (ncu gpu__time_duration.sum, cold cache, serialised)\n\n" % (title, len(seq), tot / 1e6))
        for k, (n, v) in sorted(agg.items(), key=lambda kv: -kv[1][1]):
            f.write("%6.2f%%  %5d x %9.2f us  %s\n" % (100 * v / tot, n, v / n / 1e3, k))

for a in ("fast", "exact"):
    summary("%s/launches_%s.csv" % (src, a), "profiles/%s_ncu_launch_list_summary_%s.txt" % (tag, a),
            "tools/profile_step.py 3 2 (config 2, arithmetic %s): 5 eager steps" % a)
summary("%s/launches_bench.csv" % src, "profiles/%s_ncu_launch_list_summary_bench_py.txt" % tag,
        "python bench.py --only loss --no-cpu-baseline --steps 3 --warmup 3")
summary("%s/launches_pft_hotpath.csv" % src, "profiles/%s_ncu_launch_list_summary_pft_hotpath.txt" % tag,
        "tools/profile_pft_hotpath.py 3: three PFT epochs (B=6 window, 2 sources, 4 egomotion iterations) without the depth network")

traffic = {}
for a in ("fast", "exact"):
    rows = list(csv.reader(open("%s/prof_%s_raw.csv" % (src, a))))
    idx = {k: i for i, k in enumerate(rows[0])}
    units = rows[1]
    t = {}
    for r in rows[2:]:
        name = r[idx["Kernel Name"]]
        key = "pair_loss_bwd" if "bwd" in name else "pair_loss_fwd"
        tot = 0.0
        for m in ("dram__bytes_read.sum", "dram__bytes_write.sum"):
            scale = {"Mbyte": 1e6, "Gbyte": 1e9, "Kbyte": 1e3, "byte": 1.0}[units[idx[m]]]
            tot += float(r[idx[m]].replace(",", "")) * scale
        t.setdefault(key, int(tot))
    traffic[a] = t
traffic["source"] = "profiles/%s_ncu_pair_kernels_summary_{fast,exact}.txt (ncu --set full, config 2, one launch each)" % tag
json.dump(traffic, open("profiles/ncu_traffic.json", "w"), indent=1)
print(json.dumps(traffic))
PY
cuobjdump -sass -fun '_ZN5tcsfm15pair_bwd_kernelILi0ELb1EEEvNS_10PairLaunchE' tightly-coupled-sfm_b200/libtcsfm_b200.so > /tmp/sass_bwd.txt 2>/dev/null || true
python - $tag <<'PY'
import collections, re, subprocess, sys
tag = sys.argv[1]
out = subprocess.run(["cuobjdump", "-sass", "tightly-coupled-sfm_b200/libtcsfm_b200.so"], capture_output=True, text=True).stdout
fn, hist = None, collections.OrderedDict()
keep = []
for line in out.splitlines():
    m = re.search(r"Function : (\S+)", line)
    if m:
        fn = m.group(1); hist[fn] = collections.Counter(); continue
    m = re.search(r"/\*[0-9a-f]{4}\*/\s+(?:@!?U?P\d+\s+)?([A-Z0-9_.]+)", line)
    if m and fn:
        op = m.group(1).split(".")[0]
        hist[fn][op] += 1
        if op in ("UTMALDG", "UTMASTG", "SYNCS", "UBLKCP", "LDGSTS", "FFMA2", "FADD2", "FMUL2", "REDG", "RED", "ATOMG"):
            if op in ("UTMALDG", "SYNCS"):
                keep.append("%s: %s" % (fn[:60], line.strip()[:150]))
with open("profiles/%s_sass_pair_kernels.txt" % tag, "w") as f:
    f.write("cuobjdump -sass libtcsfm_b200.so (sm_100a): instruction mnemonics per kernel (pair / warp kernels, flavour 0)\n\n")
    for fn, c in hist.items():
        if "pair_" in fn and "ILi0" in fn:
            tot = sum(c.values())
            pick = ["UTMALDG", "SYNCS", "LDGSTS", "LDG", "STG", "LDS", "STS", "FFMA", "FFMA2", "FADD", "FADD2", "FMUL", "FMUL2", "MUFU", "RED", "REDG", "ATOMG", "SHFL", "BAR", "IMAD", "LDL", "STL"]
            f.write("%s\n  %d SASS instructions; %s\n\n" % (fn, tot, ", ".join("%s %d" % (k, c[k]) for k in pick if c[k])))
    f.write("TMA / mbarrier instructions (the backward's coefficient staging):\n")
    for k in keep:
        f.write("  " + k + "\n")
print(open("profiles/%s_sass_pair_kernels.txt" % tag).read()[:3000])
PY
