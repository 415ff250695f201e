"""A/B of library variants (build_native.py --variant NAME): runs bench.py once per variant with SSDGEOM_LIB set and
prints value / step / kernel times side by side.  usage: python tools/ab_bench.py [--args "bench args"] [--jsonl FILE]
NAME [NAME ...]  (NAME "base" = the default build; list names repeatedly, e.g. "old base old base", to alternate them;
--jsonl appends every run's bench result line, tagged with its variant, to FILE)."""
import json, os, subprocess, sys

root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
libdir = os.path.join(root, "ssd-object-detection_b200", "ssdgeom", "_lib")
argv = sys.argv[1:]
extra = []
jsonl = None
while argv and argv[0] in ("--args", "--jsonl"):
    if argv[0] == "--args":
        extra = argv[1].split()
    else:
        jsonl = argv[1]
    argv = argv[2:]
for name in argv:
    env = dict(os.environ)
    if name != "base":
        env["SSDGEOM_LIB"] = os.path.join(libdir, "libssdgeom_%s.so" % name)
    p = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--no-cpu-baseline", "--no-e2e"] + extra,
                       env=env, capture_output=True, text=True)
    try:
        d = json.loads(p.stdout.strip().splitlines()[-1])
        k = d["detail"]["kernels_ms"]
        print("%-10s %9.0f img/s  step %.4f ms  closed %.4f ms  frac %.3f  filter %.4f nms %.4f match %.4f  detect %.4f "
              "assign %.4f" % (
            name, d["value"], d["ms_per_step"], d["detail"]["steps_in_flight"]["closed_step_ms"], d["roofline"]["frac"],
            k["filter_kernel_with_row_stats"], k["nms_kernel"], k["match_kernel"],
            d["detail"]["stages_ms"]["detect_with_row_stats_ms"], d["detail"]["stages_ms"]["assign_ms"]), flush=True)
        if jsonl:
            with open(jsonl, "a") as f:
                f.write(json.dumps({"variant": name, "result": d}) + "\n")
    except Exception as e:   # noqa: BLE001
        print(name, "FAILED", e, p.stderr[-400:], flush=True)
