"""Turn an ncu capture of one bench step (raw-page CSV with dram__bytes_read.sum / dram__bytes_write.sum, as written
by tools/ncu_export.py) into profiles/ncu_traffic.json: DRAM bytes (read + write) per launch under the kernel names
bench.py reports.  bench.py copies the figure of its dominant kernel into `roofline.traffic`.

    ncu --metrics dram__bytes_read.sum,dram__bytes_write.sum,gpu__time_duration.sum --clock-control none \
        -k regex:... --launch-skip <n> --launch-count <n> -o x python tools/prof_step.py 2
    python tools/ncu_export.py x.ncu-rep ; python tools/ncu_traffic.py x.raw.csv.gz profiles/ncu_traffic.json
"""
import csv
import gzip
import json
import re
import sys
from collections import defaultdict

SRC = {"ZoneTokSrc": "hist2image", "WindowRows": "lsa", "SrTokSrc": "gsa", "InsideSrc": "dapm",
       "ZonePatchRows": "hist2image", "FrameRows": "gsa", "OutsideRows": "dapm"}


def to_bytes(value, unit):
    scale = {"byte": 1, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}
    return float(value) * scale.get(unit, 1)


def main(path, out):
    rows = list(csv.reader(gzip.open(path, "rt")))
    h, units = rows[0], rows[1]
    ci = {n: (h.index(n) if n in h else None) for n in ("Kernel Name", "dram__bytes_read.sum", "dram__bytes_write.sum", "gpu__time_duration.sum")}
    def cell(r, n):
        return (r[ci[n]], units[ci[n]]) if ci[n] is not None else ("0", "byte")
    acc = defaultdict(lambda: [0, 0.0, 0.0, 0.0])
    conv_parity, level_c = 0, None
    for r in rows[2:]:
        full = r[ci["Kernel Name"]]
        base = re.sub(r"^void ", "", full).replace("cfp::", "")
        fn = re.match(r"(\w+)", base).group(1)
        targs = re.search(r"<(.*)>\(", base)
        t = [x.strip() for x in re.sub(r"\((int|bool)\)", "", targs.group(1)).split(",")] if targs else []
        kind = next((v for k, v in SRC.items() if k in base), None)
        if fn == "kv_state_tc_kernel":
            name = f"kv_state_tc<{kind},{t[0]}>"
        elif fn in ("loftr_query_tc_kernel", "loftr_query_mono_kernel"):
            name = (f"attn_query_tc<{kind},{t[0]}>" if t[2] == "1" else f"loftr_query_tc<{kind},{t[0]}>")
        elif fn == "conv3x3_tc_kernel":
            level_c = t[0]
            name = f"conv3x3_tc<{'2C->C' if conv_parity == 0 else 'C->C'},{t[0]}>"
            conv_parity ^= 1
        elif fn == "dwconv_tc_kernel":
            name = f"dwconv_tc<{ {'32': 31, '64': 15, '128': 7}.get(level_c, '?') }>"
        elif fn == "dwconv_bn_relu_kernel":
            name = f"dwconv<{t[0]}>"
        elif fn in ("lkpm_mlp_tc_kernel", "sr_conv_tc_kernel"):
            name = fn.replace("_kernel", "") + f"<{t[0]}>"
        elif fn.startswith("layout"):
            name = "layout_kernel"
        elif fn == "sr_bias_ln_kernel":
            name = "sr_bias_ln"
        elif fn == "dw_plane_pack_kernel":
            name = "dw_plane_pack"
        elif fn == "hist_encoder_tc_kernel":
            name = "hist_encoder_tc"
        else:
            name = fn
        a = acc[name]
        a[0] += 1
        a[1] += to_bytes(*cell(r, "dram__bytes_read.sum"))
        a[2] += to_bytes(*cell(r, "dram__bytes_write.sum"))
        a[3] += float(r[ci["gpu__time_duration.sum"]])
    doc = {"source": path, "note": "ncu dram__bytes_read.sum + dram__bytes_write.sum per launch (cold-cache, serialised replay)",
           "bytes_per_launch": {k: (v[1] + v[2]) / v[0] for k, v in acc.items()},
           "detail": {k: {"launches": v[0], "read_MB": v[1] / v[0] / 1e6, "write_MB": v[2] / v[0] / 1e6, "us": v[3] / v[0]}
                      for k, v in acc.items()}}
    with open(out, "w") as fh:
        json.dump(doc, fh, indent=1)
    for k, v in sorted(doc["detail"].items(), key=lambda kv: -kv[1]["us"] * acc[kv[0]][0]):
        print(f"{k:34s} x{v['launches']:2d} {v['us']:7.1f} us  rd {v['read_MB']:7.1f} MB  wr {v['write_MB']:7.1f} MB")


if __name__ == "__main__":
    main(sys.argv[1], sys.argv[2])
