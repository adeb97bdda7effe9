#!/usr/bin/env python
"""profiles/{spmv,update,c3_spmv}_traffic.json (read by bench.py for the streaming roofline) from the captures of
profiles/run_ncu.sh:  python profiles/make_stream_traffic.py <tag>
  <tag>_stream_ncu_raw.csv  ncu --set full of k_pcg_spmv / k_pcg_update (streaming comparison solve of bench.py)
  <tag>_c3_traffic.csv      ncu --metrics dram bytes / time of the same kernels on config 3 (cantilever L4)"""
import csv, json, os, re, sys
here = os.path.dirname(os.path.abspath(__file__))
tag = sys.argv[1]
rows = list(csv.reader(open(os.path.join(here, "%s_stream_ncu_raw.csv" % tag))))
hdr, units = rows[0], rows[1]
col = lambda name: hdr.index(name)
scale = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9, "ns": 1e-3, "us": 1.0, "ms": 1e3}
def val(r, name):
    return float(r[col(name)]) * scale.get(units[col(name)], 1.0)
per = {}
for r in rows[2:]:
    per.setdefault(re.sub(r"^void\s+|\(.*", "", r[col("Kernel Name")]), []).append(r)
for k, rs in per.items():
    n = len(rs)
    rd = sum(val(r, "dram__bytes_read.sum") for r in rs) / n
    wr = sum(val(r, "dram__bytes_write.sum") for r in rs) / n
    us = sum(val(r, "gpu__time_duration.sum") for r in rs) / n
    out = {"kernel": k, "source": "profiles/%s_stream_ncu_raw.csv (ncu --set full, %d launches, iterations 20-22 of the streaming "
                                  "comparison solve of bench.py, all 400 systems active)" % (tag, n),
           "workload": "100 plates x 4 conditions, mesh_size 1e-2", "nnz": 49452160, "n_active_dofs": 3664196,
           "dram_bytes_read_per_launch": rd, "dram_bytes_write_per_launch": wr, "dram_bytes_per_launch": rd + wr,
           "gpu_time_us_under_ncu": us, "dram_GBs_under_ncu": (rd + wr) / us / 1e3,
           "registers_per_thread": int(rs[0][col("launch__registers_per_thread")]),
           "l2_hit_rate_pct": float(rs[0][col("lts__t_sector_hit_rate.pct")])}
    name = "spmv_traffic.json" if "spmv" in k else "update_traffic.json"
    json.dump(out, open(os.path.join(here, name), "w"), indent=1)
    print(name, round(out["dram_bytes_per_launch"] / 1e6, 1), "MB", round(us, 1), "us", round(out["dram_GBs_under_ncu"]), "GB/s")
c3 = {}
for r in csv.reader(open(os.path.join(here, "%s_c3_traffic.csv" % tag))):
    if len(r) > 14 and r[0].isdigit():
        c3.setdefault(re.sub(r"^void\s+|\(.*", "", r[4]), {}).setdefault(r[12], []).append(float(r[14]))
out = {"source": "profiles/%s_c3_traffic.csv (ncu --metrics dram bytes / time, 4 iterations of tools/tune_spmv_c3.py cantilever 4)" % tag}
for k, m in c3.items():
    mean = lambda name: sum(m[name]) / len(m[name])
    us = mean("gpu__time_duration.sum") * 1e-3
    by = mean("dram__bytes_read.sum") + mean("dram__bytes_write.sum")
    out[k] = {"us_under_ncu": us, "dram_bytes_per_launch": by, "dram_GBs": by / us / 1e3,
              "l2_bytes_per_launch": 32.0 * mean("lts__t_sectors.sum")}
    if "spmv" in k:
        out["cantilever_L4"] = out[k]["dram_GBs"]
json.dump(out, open(os.path.join(here, "c3_spmv_traffic.json"), "w"), indent=1)
print("c3", {k: round(v["dram_GBs"]) for k, v in out.items() if isinstance(v, dict)})
