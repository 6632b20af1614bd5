"""Turn the files of scratch/r2_evidence.sh (gpurun_out/r02ev/*) into the committed summaries under profiles/ (r02_*)."""
import collections, csv, gzip, json, os, shutil, sys
src = sys.argv[1] if len(sys.argv) > 1 else "gpurun_out/r02ev"
rnd = sys.argv[2] if len(sys.argv) > 2 else "r02"
os.chdir(os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
def f(x):
    try: return float(x.replace(',', ''))
    except Exception: return 0.0
KEYS = ["gpu__time_duration.sum", "launch__grid_size", "launch__block_size", "launch__registers_per_thread", "dram__bytes_read.sum", "dram__bytes_write.sum",
        "sm__throughput.avg.pct_of_peak_sustained_elapsed", "sm__pipe_tensor_subpipe_hmma_cycles_active.avg.pct_of_peak_sustained_active",
        "sm__inst_executed_pipe_xu.avg.pct_of_peak_sustained_active", "smsp__issue_active.avg.pct_of_peak_sustained_active",
        "l1tex__throughput.avg.pct_of_peak_sustained_elapsed", "lts__throughput.avg.pct_of_peak_sustained_elapsed",
        "sm__warps_active.avg.pct_of_peak_sustained_active", "l1tex__data_bank_conflicts_pipe_lsu_mem_shared.sum",
        "l1tex__data_pipe_lsu_wavefronts_mem_shared.sum", "smsp__inst_executed.sum", "sm__cycles_elapsed.max"]
names = ["score_incr", "score_late", "score_small", "score_step0", "alpha_incr", "alpha_late", "alpha_small", "alpha_step0", "colblock", "rowqkv", "rowqk", "rowpv", "ffn", "softmax", "merge", "merge_late", "derive", "rowqk_bf16", "rowpv_bf16"]
out, tr = [], {}
def gb(v, u): return f(v) * {"Gbyte": 1e9, "Mbyte": 1e6, "Kbyte": 1e3, "byte": 1}[u]
for name in names:
    p = f"{src}/{name}.raw.csv"
    if not os.path.exists(p): continue
    rows = list(csv.reader(open(p)))
    if len(rows) < 3: continue
    hdr, units, r = rows[0], rows[1], rows[2]
    d = {k: (r[hdr.index(k)], units[hdr.index(k)]) for k in KEYS if k in hdr}
    out.append(f"== {name}: {r[hdr.index('Kernel Name')][:80]}")
    for k in KEYS:
        if k in d: out.append(f"   {k:85s} {d[k][0]:>16s} {d[k][1]}")
    tu = d["gpu__time_duration.sum"]; t_us = f(tu[0]) * {"ms": 1e3, "us": 1.0, "usecond": 1.0, "msecond": 1e3, "ns": 1e-3, "nsecond": 1e-3, "s": 1e6, "second": 1e6}.get(tu[1], 1.0)
    by = gb(*d["dram__bytes_read.sum"]) + gb(*d["dram__bytes_write.sum"])
    tr[name] = {"dram_bytes": by, "time_us": t_us}
    out.append(f"   -> DRAM {by / 1e9:.2f} GB in {t_us:.0f} us = {by / t_us / 1e6:.2f} TB/s")
    rs = list(csv.reader(open(f"{src}/{name}.source.csv")))
    h2 = rs[1]; si = h2.index("# Samples")
    st = [i for i, h in enumerate(h2) if h.startswith("stall_") and "Not Issued" not in h]
    data = [x for x in rs[2:] if len(x) == len(h2)]
    T = sum(f(x[si]) for x in data) or 1
    out.append("   warp-state samples: " + "  ".join(f"{h2[i][6:]}={100 * sum(f(x[i]) for x in data) / T:.1f}%" for i in st if sum(f(x[i]) for x in data) / T > 0.02))
head = ("round 2 (" + rnd + "): ncu --set full --import-source on --clock-control none, python scratch/prof_rollout.py 128 1 (one 128-alignment chunk, 50 x 1024, bf16x3); one launch per kernel\n"
        "score_incr = k_score_inc launch #15 (NJ step 16, 33 pairs per tree); score_late = k_score_inc launch #30 (19 pairs: narrow mode); score_small = k_score_small launch #4 (12 pairs);\n"
        "alpha_incr = k_alpha_v3 launch #20 (step 16); alpha_late = k_alpha_v3 launch #36 (4-way site split, ~18 pairs); alpha_small = k_alpha_small launch #4; step0 = first launch, 256 pairs per tree;\n"
        "rowqk = k_tc_gemm2s launch #2 (Q K^T + softmax on CTA pairs), rowpv = k_tc_gemm2w launch #1 (one-pass P V on CTA pairs); merge = k_merge launch #20 (30 live nodes), merge_late = launch #40 (10 live nodes); derive = k_node_derive; *_bf16 = the same GEMM launches with precision=\"bf16\" (one product)\n")
open(f"profiles/{rnd}_ncu_full_summary_b128.txt", "w").write(head + "\n".join(out) + "\n")
json.dump(tr, open(f"profiles/{rnd}_traffic_b128.json", "w"), indent=1)
# launch list
rows = [r for r in csv.reader(open(f"{src}/launches.csv")) if len(r) > 5]
hdr = rows[0]; ki = hdr.index("Kernel Name"); vi = hdr.index("Metric Value")
agg = collections.OrderedDict()
for r in rows[1:]:
    k = r[ki].split("(")[0].replace("void ", "").replace("nnj::", "")
    a = agg.setdefault(k, [0, 0.0]); a[0] += 1; a[1] += f(r[vi])
tot = sum(a[1] for a in agg.values())
cls = {"k_enc_colblock_tc<2, 7>": "col_attn", "k_score_tc": "pair_score", "k_score_inc": "pair_score", "k_score<0>": "pair_score", "k_alpha_v3": "alpha", "k_enc_colblock_tc": "col_attn", "k_tc_gemm<256, 0>": "row_qk_gemm",
       "k_tc_gemm<256, 1>": "row_pv_gemm", "k_tc_gemm<128, 1>": "row_pv_gemm", "k_tc_gemm<128, 0>": "row_qk_gemm", "k_softmax_rows_split": "row_softmax", "k_softmax_rows_split_reg<4>": "row_softmax", "k_softmax_rows_split_reg<2>": "row_softmax", "k_enc_ffn_tc": "ffn",
       "k_enc_rowqkv_tc": "ln_qkv", "k_alpha1": "merge", "k_merge<1>": "merge", "k_merge<0>": "merge", "k_node_derive": "node_derive",
       "k_alpha_softmax": "alpha_softmax", "k_select": "select", "k_embed": "embed"}
lines = ["ncu --metrics gpu__time_duration.sum --clock-control none python scratch/prof_rollout.py 128 1   (one chunk of 128 alignments, 50 x 1024, bf16x3)",
         "per-launch times under ncu are cold-cache and serialised: compare SHARES with bench.py's live CUDA-event classes (profiles/" + rnd + "_bench_final.json)",
         f"{'kernel':34s} {'launches':>8s} {'total ms':>10s} {'share':>7s} {'avg us':>10s}"]
for k, a in sorted(agg.items(), key=lambda kv: -kv[1][1]):
    lines.append(f"{k[:34]:34s} {a[0]:8d} {a[1] / 1e6:10.3f} {100 * a[1] / tot:6.2f}% {a[1] / a[0] / 1e3:10.1f}")
lines.append(f"{'total':34s} {sum(a[0] for a in agg.values()):8d} {tot / 1e6:10.3f}")
byc = collections.defaultdict(float)
def klass(k):
    if k in cls: return cls[k]
    if k.startswith("k_tc_gemm2w"): return "row_pv_gemm"
    if k.startswith("k_tc_gemm2s"): return "row_qk_gemm"
    if k.startswith("k_tc_gemm2<"): return "row_pv_gemm" if k.startswith("k_tc_gemm2<1") else "row_qk_gemm"
    if k.startswith("k_tc_gemm<"):      # <BN, BMN, ONE>: MN-major B = the P V GEMM
        return "row_pv_gemm" if k.split(",")[1].strip().startswith("1") else "row_qk_gemm"
    for pre, c in (("k_merge<", "merge"), ("k_node_derive", "node_derive"), ("k_score_small", "pair_score"), ("k_alpha_small", "alpha"), ("k_enc_colblock_tc", "col_attn"), ("k_score_big", "pair_score"), ("k_blend_planes", "pair_blend")):
        if k.startswith(pre): return c
    return "misc"
for k, a in agg.items(): byc[klass(k)] += a[1]
b = json.loads(open(f"{src}/bench.json").read().strip().splitlines()[-1])
lines += ["", f"share by bench.py class (ncu)  vs  live CUDA events (bench line of the same run, profiles/{rnd}_bench_final.json)"]
for c, v in sorted(byc.items(), key=lambda kv: -kv[1]):
    live = b["kernels"].get(c, {}).get("share")
    lines.append(f"  {c:16s} ncu {100 * v / tot:6.2f}%" + (f"   live {100 * live:6.2f}%" if live is not None else ""))
open(f"profiles/{rnd}_ncu_launch_summary_bf16x3_b128.txt", "w").write("\n".join(lines) + "\n")
with open(f"{src}/launches.csv", "rb") as fi, gzip.open(f"profiles/{rnd}_ncu_launches_bf16x3_b128.csv.gz", "wb") as fo: shutil.copyfileobj(fi, fo)
shutil.copy(f"{src}/bench.json", f"profiles/{rnd}_bench_final.json")
for a, bname in (("bench_config4.json", "bench_config4.json"), ("search.json", "search_mode.json"), ("col_trace.txt", "col_trace.txt"), ("hmma_bench.txt", "hmma_bench.txt")):
    if os.path.exists(f"{src}/{a}"): shutil.copy(f"{src}/{a}", f"profiles/{rnd}_{bname}")
if os.path.exists(f"{src}/chunk_sweep.jsonl"):
    sweep = []
    for l in open(f"{src}/chunk_sweep.jsonl"):
        d = json.loads(l); c = d["classes"]
        nj = sum(c[k][0] for k in ("alpha", "alpha_softmax", "pair_score", "select", "merge", "node_derive", "misc") if k in c)
        enc = sum(c[k][0] for k in ("embed", "ln_qkv", "row_qk_gemm", "row_softmax", "row_pv_gemm", "col_attn", "ffn") if k in c)
        sweep.append({"trees_per_chunk": int(d["chunk_max"]), "trees_per_s": d["trees_per_s"], "encoder_ms_per_tree": round(enc / d["B"], 3), "nj_loop_ms_per_tree": round(nj / d["B"], 3),
                      "launches": sum(v[1] for v in c.values())})
    json.dump({"what": "128 alignments of 50 x 1024 in chunks of NNJ_CHUNK_MAX trees (scratch/r2_explore.py): an L2-resident NJ loop would get FASTER per tree as the chunk's live node pool (n x 1.5 MB per tree) drops under the 126 MB L2; it gets slower - fewer work items per launch, same bytes",
               "sweep": sweep}, open(f"profiles/{rnd}_chunk_sweep.json", "w"), indent=1)
print("\n".join(out)); print("\n".join(lines[-18:])); print(b["value"], b["e2e"]["value"], b["clocks"])
