"""Full SASS listings of the hot kernels (north_star: "each kernel's choice is evidenced by a committed SASS listing").
    python scripts/dump_sass.py [tag]     -> profiles/sass_<tag>/<kernel>.sass + profiles/sass_<tag>/README.md
Instruction encodings are stripped (address + instruction text are kept)."""
import os
import re
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
tag = sys.argv[1] if len(sys.argv) > 1 else "r02"
out = os.path.join(ROOT, "profiles", f"sass_{tag}")
os.makedirs(out, exist_ok=True)
lib = os.path.join(ROOT, "generalized-icp_b200", "libgicp_b200.so")
txt = subprocess.run(["cuobjdump", "-sass", lib], capture_output=True, text=True, check=True).stdout
want = {
    "knn_hist_kernel_3_float": "_ZN4gicp15knn_hist_kernelILi3EfEEvNS_7KnnArgsIT0_EE",
    "correspond_kernel_3_float": "_ZN4gicp17correspond_kernelILi3EfEEvNS_7ObjArgsIT0_EE",
    "accumulate_kernel_3_float": "_ZN4gicp17accumulate_kernelILi3EfLb0EEEvNS_7ObjArgsIT0_EE",
    "solve_kernel_3": "_ZN4gicp12solve_kernelILi3EEEvNS_9SolveArgsE",
    "register_loop_kernel_2_double": "_ZN4gicp20register_loop_kernelILi2EdLb0ELb0EEEvNS_7ObjArgsIT0_EENS_9SolveArgsEPKd",
}
rows = []
for part in re.split(r"(?=\n\s+Function : )", txt):
    for name, sym in want.items():
        if f"Function : {sym}\n" not in part:
            continue
        lines = []
        for ln in part.strip("\n").splitlines():
            if re.match(r"\s+/\* 0x[0-9a-f]+ \*/\s*$", ln):
                continue                                   # second half of an instruction's encoding
            lines.append(re.sub(r"\s+/\* 0x[0-9a-f]+ \*/\s*$", "", ln).rstrip())
        open(os.path.join(out, name + ".sass"), "w").write("\n".join(lines) + "\n")
        body = "\n".join(lines)
        n = len(re.findall(r"^\s+/\*[0-9a-f]{4,5}\*/", body, re.M))
        cnt = {m: len(re.findall(r"\b" + m, body)) for m in ("UBLKCP", "SYNCS", "LDS", "STS", "LDG", "STG", "DFMA", "FFMA", "SHFL", "BAR")}
        rows.append((name, n, cnt))
with open(os.path.join(out, "README.md"), "w") as f:
    f.write(f"# SASS listings ({tag}) - `cuobjdump -sass generalized-icp_b200/libgicp_b200.so`, sm_100a\n\n"
            "One file per hot kernel (encodings stripped).  `UBLKCP` = TMA bulk copy (`cp.async.bulk`), `SYNCS` = mbarrier "
            "operations; no tensor-core instruction appears (the contractions have K = 2-3).\n\n"
            "| kernel | instructions | UBLKCP | SYNCS | LDS | STS | LDG | STG | FFMA | DFMA | SHFL |\n|---|---:|---:|---:|---:|---:|---:|---:|---:|---:|---:|\n")
    for name, n, c in rows:
        f.write(f"| `{name}` | {n} | {c['UBLKCP']} | {c['SYNCS']} | {c['LDS']} | {c['STS']} | {c['LDG']} | {c['STG']} | {c['FFMA']} | {c['DFMA']} | {c['SHFL']} |\n")
print(rows)
