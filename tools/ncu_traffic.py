"""DRAM bytes per kernel family from an `ncu --metrics dram__bytes_read.sum,dram__bytes_write.sum,gpu__time_duration.sum --csv` log:
   python tools/ncu_traffic.py gpurun_out/traffic_b64.csv > profiles/rN_dram_traffic_b64.json"""
import collections, csv, json, sys
rows = list(csv.reader(open(sys.argv[1])))
h = [i for i, r in enumerate(rows) if r and r[0] == "ID"][0]
H = rows[h]
ki, mi, ui, vi = H.index("Kernel Name"), H.index("Metric Name"), H.index("Metric Unit"), H.index("Metric Value")
fam = {"tc_conv_kernel": "tc_conv", "tc_conv2_kernel": "tc_conv", "snake_aa": "snake", "attention_tc5": "attention"}
agg = collections.defaultdict(lambda: {"launches": 0, "dram_read_bytes": 0.0, "dram_write_bytes": 0.0, "ncu_ms": 0.0})
scale = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9, "ns": 1e-6, "us": 1e-3, "ms": 1.0, "s": 1e3}
for r in rows[h + 1:]:
    if len(r) <= vi:
        continue
    name = next((v for k, v in fam.items() if k in r[ki]), None)
    if name is None:
        continue
    v = float(r[vi].replace(",", "")) * scale.get(r[ui], 1.0)
    d = agg[name]
    if r[mi] == "dram__bytes_read.sum":
        d["dram_read_bytes"] += v
        d["launches"] += 1
    elif r[mi] == "dram__bytes_write.sum":
        d["dram_write_bytes"] += v
    elif r[mi] == "gpu__time_duration.sum":
        d["ncu_ms"] += v
out = dict(agg)
out["note"] = ("ncu --metrics dram__bytes_read.sum,dram__bytes_write.sum,gpu__time_duration.sum at B=64 (one step, "
               "tools/profile_step.py --batch 64), summed over all launches of the kernel family")
print(json.dumps(out, indent=1))
