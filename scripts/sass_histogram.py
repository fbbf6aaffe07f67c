"""profiles/r2_sass_opcodes.md: per-kernel SASS opcode histogram of the in-tree libb200nuts.so (cuobjdump -sass), the
mnemonics that prove which hardware path a kernel uses (B200_PROFILING.md): DMMA (fp64 tensor path), UTCHMMA (tcgen05.mma
kind::f16), UTMALDG (TMA tensor-map loads), UBLKCP (bulk TMA), LDTM/STTM (tcgen05.ld/st), UTCBAR (tcgen05.commit),
LDGSTS (cp.async), SYNCS (mbarrier), DFMA/DADD/DMUL."""
import collections, os, re, subprocess, sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
lib = os.path.join(ROOT, "pymc_b200", "libb200nuts.so")
out = subprocess.run(["cuobjdump", "-sass", lib], capture_output=True, text=True).stdout
KEYS = ["UTCHMMA", "UTMALDG", "UBLKCP", "LDTM", "STTM", "UTCBAR", "UTCATOMSWS", "DMMA", "LDGSTS", "SYNCS", "DFMA", "DADD", "DMUL",
        "MUFU", "SHFL", "LDS", "STS", "LDG", "STG", "ATOMG", "BAR"]
kern, cur = collections.OrderedDict(), None
for line in out.splitlines():
    m = re.match(r"\s*Function : (\S+)", line)
    if m:
        cur = m.group(1)
        kern[cur] = collections.Counter()
        continue
    m = re.match(r"\s+/\*[0-9a-f]{4,}\*/\s+(?:@!?U?P\d+\s+)?([A-Z0-9_]+)", line)
    if m and cur:
        kern[cur][m.group(1)] += 1
        kern[cur]["_total"] += 1
demangle = subprocess.run(["c++filt"], input="\n".join(kern), capture_output=True, text=True).stdout.splitlines()
commit = subprocess.run(["git", "-C", ROOT, "rev-parse", "--short", "HEAD"], capture_output=True, text=True).stdout.strip()
rows = []
for (name, c), dn in zip(kern.items(), demangle):
    short = re.sub(r"\(.*", "", dn).replace("void ", "").replace("b200::", "")
    rows.append((short, c))
want = sys.argv[1:] or ["nuts_warp_kernel<RadonModel, 6", "nuts_warp_kernel<StochVolModel, 12", "nuts_warp_kernel<IrModel, 6, 1", "logistic_fused_kernel<16",
                        "gemm_nt_dmma_kernel<8, 17", "gemm_tc_kernel", "ls_advance_kernel<16", "ls_advance_kernel<1",
                        "logp_grad_warp_kernel<RadonModel, 6", "ir_pointwise_kernel"]
with open(os.path.join(ROOT, "profiles", "r2_sass_opcodes.md"), "w") as f:
    f.write(f"# SASS opcode counts per kernel (static, `cuobjdump -sass pymc_b200/libb200nuts.so`), built from commit `{commit}` + working tree\n\n")
    f.write("| kernel | instructions | " + " | ".join(KEYS) + " |\n|---|---|" + "---|" * len(KEYS) + "\n")
    for short, c in rows:
        if any(short.startswith(w) for w in want):
            f.write(f"| `{short}` | {c['_total']} | " + " | ".join(str(c.get(k, 0)) for k in KEYS) + " |\n")
    f.write("\nReading: `UTCHMMA` = `tcgen05.mma.kind::f16` (only the two performance-mode kernels), `UTMALDG` = TMA tensor-map loads, "
            "`LDTM`/`STTM` = `tcgen05.ld`/`st`, `UTCBAR` = `tcgen05.commit`; `DMMA` = the fp64 tensor path of the parity-mode dense "
            "kernels; `UBLKCP` = bulk TMA staging of the observed data; `LDGSTS` = `cp.async` of the DMMA GEMM pipeline.\n")
print(open(os.path.join(ROOT, "profiles", "r2_sass_opcodes.md")).read()[:3000])
