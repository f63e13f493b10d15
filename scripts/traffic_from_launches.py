"""Per-stage time and DRAM traffic of the LAST bench step in an ncu launch list (gpu__time_duration.sum,
dram__bytes_read.sum, dram__bytes_write.sum), and -- with --update -- the `profiles/traffic.json` entry bench.py reads for
`roofline.traffic`.   python scripts/traffic_from_launches.py launches.csv <workload> [--update] [--source "text"]"""
import collections, csv, json, os, re, sys

STAGES = [   # (stage, regex over kernel names); first match wins
    ("project_fwd", r"in_wproj_image_kernel|in_proj_gemm<\(bool\)1>|in_proj_gemm<true>|in_proj_gemm<1>|build_b_images|gemm_tc_ws2|gemm_simt|wabsmax|in_w_absmax"),
    ("gat_fwd", r"gat_fwd_"),
    ("gat_bwd_dst_src", r"gat_bwd_dst|gat_bwd_src|gat_hub_chunk_sum"),
    ("project_bwd", r"dw_tc|dax_partial|colsum_partial|reduce_slices|datt_from_g|dw_reduce|gemm_tc_ws\b|transpose"),
    ("in_logits", r"in_u_kernel|in_logits_kernel|in_scales_kernel|in_wout_image|in_wgd_image"),
    ("in_fwd_edges", r"in_alpha_|gat_in_fwd_"),
    ("in_out_gemm", r"in_out_gemm"),
    ("in_bwd_gd_edges", r"in_ximg_kernel|in_proj_gemm|gat_in_bwd_"),
    ("in_bwd_dasrc", r"in_dasrc_kernel"),
    ("in_bwd_params", r"in_absmax|in_dw_gemm|in_dw_finalize"),
]
FIRST = r"in_wproj_image_kernel|build_b_images|in_u_kernel"     # the first kernel of a step (either formulation)

def main():
    path, workload = sys.argv[1], sys.argv[2]
    rows = list(csv.reader(open(path)))
    start = next(i for i, r in enumerate(rows) if "Kernel Name" in r)
    hdr = rows[start]
    ki, mi, vi, idi = hdr.index("Kernel Name"), hdr.index("Metric Name"), hdr.index("Metric Value"), hdr.index("ID")
    data = collections.OrderedDict()
    for r in rows[start + 1:]:
        if len(r) <= vi or not r[idi].isdigit():
            continue
        d = data.setdefault(r[idi], {"name": r[ki]})
        try:
            d[r[mi]] = float(r[vi].replace(",", ""))
        except ValueError:
            pass
    items = list(data.values())
    firsts = [i for i, d in enumerate(items) if re.search(FIRST, d["name"])]
    last = items[firsts[-1]:]
    stages = STAGES
    if any("in_u_kernel" in d["name"] for d in last):      # an input-space step: the shared helper kernels belong to its stages
        stages = [("in_bwd_gd_edges", r"gat_hub_chunk_sum|gat_in_bwd_"),
                  ("in_bwd_params", r"dax_partial|colsum_partial|reduce_slices|datt_from_g")] + STAGES[4:]
    agg = collections.OrderedDict()
    per_kernel = collections.OrderedDict()
    for d in last:
        nm = d["name"].split("(")[0].replace("void ", "").replace("gnnfd::", "")[:60]
        if nm.startswith("at::") or "elementwise" in nm:
            continue
        stage = next((s for s, rx in stages if re.search(rx, d["name"])), "other")
        a = agg.setdefault(stage, [0.0, 0.0, 0.0])
        k = per_kernel.setdefault(nm, [0, 0.0, 0.0, 0.0, stage])
        ms, rd, wr = d.get("gpu__time_duration.sum", 0) / 1e6, d.get("dram__bytes_read.sum", 0), d.get("dram__bytes_write.sum", 0)
        a[0] += ms; a[1] += rd; a[2] += wr
        k[0] += 1; k[1] += ms; k[2] += rd; k[3] += wr
    tot = sum(a[0] for a in agg.values())
    print(f"last step: {len(last)} launches, {tot:.2f} ms (ncu: cold cache, serialised -- compare shares, not absolutes)")
    print(f"{'ms':>9} {'share':>6} {'rd GB':>8} {'wr GB':>8} {'GB/s':>7}  stage")
    for s, a in agg.items():
        print(f"{a[0]:9.3f} {100 * a[0] / tot:5.1f}% {a[1] / 1e9:8.2f} {a[2] / 1e9:8.2f} {(a[1] + a[2]) / 1e6 / max(a[0], 1e-9):7.0f}  {s}")
    print(f"{'ms':>9} {'share':>6} {'n':>3} {'rd GB':>8} {'wr GB':>8} {'GB/s':>7}  kernel (stage)")
    for nm, k in per_kernel.items():
        print(f"{k[1]:9.3f} {100 * k[1] / tot:5.1f}% {k[0]:3d} {k[2] / 1e9:8.2f} {k[3] / 1e9:8.2f} {(k[2] + k[3]) / 1e6 / max(k[1], 1e-9):7.0f}  {nm} ({k[4]})")
    if "--update" in sys.argv:
        src = sys.argv[sys.argv.index("--source") + 1] if "--source" in sys.argv else os.path.basename(path)
        tf = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "profiles", "traffic.json")
        cur = json.load(open(tf)) if os.path.exists(tf) else {}
        e = cur.setdefault(workload, {})
        for s, a in agg.items():
            if s != "other":
                e[s] = int(a[1] + a[2])
        e["what"] = "dram__bytes_read.sum + dram__bytes_write.sum per step, summed over the kernels of each bench stage (ncu launch list)"
        e["source"] = src
        json.dump(cur, open(tf, "w"), indent=1)
        print("updated", tf)

main()
