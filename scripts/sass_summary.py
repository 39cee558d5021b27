"""SASS evidence per kernel of libcaffedistri_b200.so (run here, no GPU needed):
   python scripts/sass_summary.py [path/to/lib.so] > summary.txt
Run it on two builds and diff the outputs to compare them kernel by kernel."""
import collections, re, subprocess, sys
so = sys.argv[1] if len(sys.argv) > 1 else "caffeonspark_b200/libcaffedistri_b200.so"
txt = subprocess.run(["cuobjdump", "-sass", so], capture_output=True, text=True).stdout
res = subprocess.run(["cuobjdump", "-res-usage", so], capture_output=True, text=True).stdout
demangle = lambda n: subprocess.run(["c++filt", n], capture_output=True, text=True).stdout.strip()
PREFIX = ("LDGMC", "UBLKCP.S.G", "UBLKCP.G.S", "SYNCS", "MEMBAR.SC.SYS", "MEMBAR.ALL.SYS", "MEMBAR.ALL.GPU", "FFMA",
          "FMUL", "FADD", "BAR.SYNC", "LDG.E.NA.128", "STG.E.128", "LDG.E.128.STRONG.SYS", "STG.E.128.STRONG.SYS",
          "LDG.E.STRONG.SYS", "STG.E.STRONG.SYS", "LDG.E.64.STRONG.SYS", "STG.E.64.STRONG.SYS", "REDG", "CCTL")
BASE = ("LDG", "STG", "LDS", "STS", "LDL", "STL", "ATOMG", "F2F", "F2FP")  # every variant of the opcode


def name(mangled):
    n = re.sub(r"cosb::\(anonymous namespace\)::", "", demangle(mangled))
    return re.sub(r"\(cosb::SyncParams.*", "", n).replace("void ", "")


kernels, cur = collections.OrderedDict(), None
for line in txt.splitlines():
    m = re.search(r"Function : (\S+)", line)
    if m:
        cur = name(m.group(1))
        kernels[cur] = collections.Counter()
        continue
    m = re.search(r"/\*[0-9a-f]{4,}\*/\s+(?:@!?U?P\d+\s+)?([A-Z][A-Z0-9_.]+)", line)
    if m and cur:
        kernels[cur]["total"] += 1
        op = m.group(1)
        for key in PREFIX:
            if op.startswith(key) and not (key == "STG.E.128" and "STRONG" in op):
                kernels[cur][key] += 1
        if op.split(".")[0] in BASE:
            kernels[cur][op.split(".")[0]] += 1
for fn, usage in re.findall(r"Function (\S+):\s*\n\s*(REG:.*)", res):
    if name(fn) in kernels:
        for key in ("REG", "STACK"):
            kernels[name(fn)][key] = int(re.search(key + r":(\d+)", usage).group(1))
print("SASS evidence per kernel (cuobjdump -sass / -res-usage %s, sm_100a, nvcc 12.9)" % so)
print("""  REG / STACK = registers and stack-frame bytes per thread; LDL / STL = local-memory (spill) loads / stores
  LDG STG LDS STS ATOMG F2F F2FP = every variant of that opcode (the dotted columns count one variant each)
  LDG.E.NA.128 = ld.global.L1::no_allocate.v4.f32 (streaming 128-bit loads, local and peer)
  UBLKCP.S.G / UBLKCP.G.S = cp.async.bulk global->shared / shared->global (TMA); SYNCS.* = mbarrier
  LDGMC = multimem.ld_reduce (NVLS in-switch reduction); STG.E.128.STRONG.SYS in the nvls kernel = multimem.st
  LDG/STG.E.128.STRONG.SYS in the ll kernel = ld/st.relaxed.sys.v2.u64: two single-copy-atomic {payload, flag} words
  MEMBAR.ALL.SYS = fence.acq_rel.sys of the cross-GPU flag barrier (release before the flag store, acquire after
  the poll); the ll kernel has NONE (flag-in-data, fence-free)
  FFMA = 0 everywhere in the fused kernels: explicit __fmul_rn/__fadd_rn, nothing contracted -> bit-exact parity
""")
for k, c in kernels.items():
    cols = ("REG", "STACK", "total") + PREFIX + BASE
    print("%-58s %s" % (k[:58], "  ".join("%s=%d" % (a, c[a]) for a in cols if a in c)))
