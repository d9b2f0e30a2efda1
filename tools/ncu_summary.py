"""Turns an `ncu --page raw --csv` export of one bench step (tools/profile_round.sh) into the tracked
summary profiles/<tag>_ncu_full_one_step.csv and refreshes profiles/roofline_traffic.json.

    python tools/ncu_summary.py gpurun_out/r01d_full_raw.csv r01d
"""
import csv, json, os, re, sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
COLS = ["gpu__time_duration.sum", "dram__bytes_read.sum", "dram__bytes_write.sum",
        "sm__throughput.avg.pct_of_peak_sustained_elapsed",
        "gpu__dram_throughput.avg.pct_of_peak_sustained_elapsed",
        "sm__pipe_fma_cycles_active.avg.pct_of_peak_sustained_active",
        "sm__pipe_tensor_cycles_active.avg.pct_of_peak_sustained_active",
        "sm__inst_executed_pipe_tensor.sum",
        "smsp__issue_active.avg.pct_of_peak_sustained_active",
        "sm__warps_active.avg.pct_of_peak_sustained_active",
        "launch__registers_per_thread", "launch__occupancy_limit_shared_mem", "launch__occupancy_limit_registers",
        "l1tex__data_pipe_lsu_wavefronts_mem_shared.sum", "l1tex__data_bank_conflicts_pipe_lsu_mem_shared.sum",
        "smsp__inst_executed.sum", "sm__cycles_elapsed.max",
        "lts__t_sector_hit_rate.pct", "l1tex__t_sector_hit_rate.pct"]
STALLS = "smsp__average_warps_issue_stalled_%s_per_issue_active.ratio"
STALL_NAMES = ["long_scoreboard", "short_scoreboard", "barrier", "math_pipe_throttle", "mio_throttle",
               "lg_throttle", "wait", "not_selected", "no_instruction", "sleeping", "membar", "dispatch_stall",
               "branch_resolving", "tex_throttle", "drain", "imc_miss", "selected"]


def short(name, seen):
    table = [("conv12", "conv12"), ("frontend", "frontend"), ("seg_table", "seg_table"), ("conv1_pool1", "pool1_dump"),
             ("linear_rows_kernel<64", "lin_ln"), ("linear_rows_kernel<20", "fc_out"), ("qkv", "qkv"),
             ("sa_layer", "sa_layer"), ("pool_logits", "pool_logits"), ("pool_final", "pool_final"),
             ("lstm", "lstm"), ("lastbi", "lastbi")]
    name = name.replace("(int)", "").replace("(bool)", "")
    m = re.search(r"conv_pipe_kernel<nisqa::SpCfg<[^>]*>, (\d+)>", name)
    if m:
        return "conv%s" % m.group(1)
    for k, v in table:
        if k in name:
            return v
    return name.split("(")[0][:24]


def main():
    raw, tag = sys.argv[1], sys.argv[2]
    rows = list(csv.reader(open(raw)))
    hdr, units, data = rows[0], rows[1], rows[2:]
    idx = {}
    for i, h in enumerate(hdr):
        idx.setdefault(h, i)
        idx.setdefault(h.split(".", 2)[-1] if h.count(".") > 2 else h, i)   # strip "SM_A.TriageCompute." prefixes
    def col(name):
        return idx.get(name)
    out_cols = [c for c in COLS if col(c) is not None]
    stall_cols = [(s, col(STALLS % s)) for s in STALL_NAMES if col(STALLS % s) is not None]
    out = [["short", "Kernel Name", "Grid Size", "Block Size"] + out_cols + ["top_stalls(cycles per issue)"],
           ["", "", "", ""] + [units[col(c)] for c in out_cols] + [""]]
    traffic, seen = {}, []
    for r in data:
        nm = r[col("Kernel Name")]
        sh = short(nm, seen)
        seen.append(sh)
        vals = [r[col(c)] for c in out_cols]
        st = []
        for s, i in stall_cols:
            try:
                st.append((float(r[i].replace(",", "")), s))
            except ValueError:
                pass
        st.sort(reverse=True)
        out.append([sh, nm, r[col("Grid Size")], r[col("Block Size")]] + vals +
                   [" ".join("%s=%.2f" % (s, v) for v, s in st[:4])])
        def tobytes(c):
            v, u = float(r[col(c)].replace(",", "")), units[col(c)].lower()
            return v * {"byte": 1, "kbyte": 1e3, "mbyte": 1e6, "gbyte": 1e9}.get(u, 1)
        b = tobytes("dram__bytes_read.sum") + tobytes("dram__bytes_write.sum")
        traffic[sh] = traffic.get(sh, 0) + b
    cnt = {}
    for s in seen:
        cnt[s] = cnt.get(s, 0) + 1
    traffic = dict((k, int(v / cnt[k])) for k, v in traffic.items())      # per launch
    if "pool_logits" in traffic and "pool_final" in traffic:
        traffic["pool"] = traffic["pool_logits"] + traffic["pool_final"]
    dst = os.path.join(ROOT, "profiles", "%s_ncu_full_one_step.csv" % tag)
    csv.writer(open(dst, "w")).writerows(out)
    traffic["_note"] = ("dram__bytes_read.sum + dram__bytes_write.sum per launch, ncu --set full --clock-control none, "
                        "bench.py 64 x 10 s clips (profiles/%s_ncu_full_one_step.csv)" % tag)
    sys.path.insert(0, ROOT)
    from nisqa_b200 import build as nb_build
    traffic["_source_digest"] = nb_build.kernel_digest()      # bench.py refuses the table on any other kernel sources
    json.dump(traffic, open(os.path.join(ROOT, "profiles", "roofline_traffic.json"), "w"), indent=1)
    print("wrote", dst)
    for r in out[2:]:
        print(r[0].ljust(12), " ".join(str(x)[:9].rjust(9) for x in r[4:-1]), "|", r[-1])


if __name__ == "__main__":
    main()
