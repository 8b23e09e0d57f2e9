"""profiles/r02_traffic.json from an `ncu --set full` capture: per C-ABI entry, DRAM bytes
(dram__bytes_read.sum + dram__bytes_write.sum) of ONE launch of each kernel behind the entry.

    ncu -i gpurun_out/prof.ncu-rep --page raw --csv > raw.csv
    python tools/ncu_traffic.py raw.csv profiles/r02_traffic.json
"""
import csv
import json
import sys

ENTRY_OF = [
    ("preprocess_kernel", "arl_preprocess_push"),
    ("Conv1Fwd", "arl_conv1_forward"),
    ("Conv2Fwd", "arl_conv2_forward"),
    ("FcFwdCluster", "arl_fc_heads_forward"),            # (int)/(bool) casts are stripped below
    ("heads_fwd_kernel", "arl_fc_heads_forward"),
    ("heads_bwd_kernel", "arl_heads_backward"),
    ("returns_lossgrad_kernel", "arl_returns_lossgrad"),
    ("sumsq_kernel", "arl_clip_rmsprop"),
    ("rmsprop_kernel", "arl_clip_rmsprop"),
    ("BulkGemm<128, 32, 0, 0, 2", "arl_fc_backward"),    # fc dgrad
    ("BulkGemm<128, 64, 1, 1, 0", "arl_fc_backward"),    # fc wgrad (earlier form)
    ("BulkGemm<256, 32, 1, 0, 0", "arl_fc_backward"),    # fc wgrad
    ("Conv2Bwd", "arl_conv2_backward"),
    ("Conv2Wgrad", "arl_conv2_backward"),                # (earlier form: two kernels)
    ("Conv2Dgrad", "arl_conv2_backward"),
    ("Conv1Wgrad", "arl_conv1_backward"),
]
UNIT = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}


def main(src, dst):
    rows = list(csv.reader(open(src)))
    hdr, units = rows[0], rows[1]
    name_i = hdr.index("Kernel Name")
    rd_i, wr_i = hdr.index("dram__bytes_read.sum"), hdr.index("dram__bytes_write.sum")
    t_i = hdr.index("gpu__time_duration.sum")
    seen, out = set(), {}
    for r in rows[2:]:
        kname = r[name_i].replace("(int)", "").replace("(bool)", "")
        for pat, entry in ENTRY_OF:
            if pat in kname and pat not in seen:
                seen.add(pat)
                b = float(r[rd_i]) * UNIT[units[rd_i]] + float(r[wr_i]) * UNIT[units[wr_i]]
                e = out.setdefault(entry, {"dram_bytes_per_launch": 0.0, "kernels": []})
                e["dram_bytes_per_launch"] += b
                e["kernels"].append({"kernel": pat, "dram_bytes": b,
                                     "ncu_duration_us": float(r[t_i]) * (1e-3 if units[t_i] == "ns" else 1.0)})
    json.dump(out, open(dst, "w"), indent=1)
    for k, v in out.items():
        print("%-24s %8.1f MB" % (k, v["dram_bytes_per_launch"] / 1e6))


if __name__ == "__main__":
    main(sys.argv[1], sys.argv[2])
