"""Per-kernel counts of the SASS instructions that matter for the roofline discussion + the bulk-copy excerpt.
cuobjdump -sass tce_rl_b200/libtce_b200.so | python scripts/sass_evidence.py > profiles/r02_sass_evidence.txt"""
import collections, re, sys
txt = sys.stdin.read()
funcs = re.split(r'\n\s*Function : ', txt)
out = ["# SASS evidence (cuobjdump -sass tce_rl_b200/libtce_b200.so, sm_100a); scripts/sass_evidence.py",
       "# per-kernel counts (kernels with bulk copies, cp.async, MMA, or > 300 FMAs):",
       "#   UBLKCP.S.G = cp.async.bulk global -> shared (TMA, non-tensor form); SYNCS.* = mbarrier (ARRIVE.TRANS64 = expect_tx,",
       "#   PHASECHK.TRANS64.TRYWAIT = try_wait.parity); LDGSTS = cp.async (Ampere form); DFMA/FFMA = fp64 / fp32 FMA; FFMA2 = packed fp32x2 FMA (sm_100);",
       "#   MMA = DMMA.8x8x4 (fp64 tensor cores: the projection kernels' shared-memory matrix products, la_gemm); no HMMA /",
       "#   UTC*MMA / LDTM / STTM anywhere: nothing runs on the fp16 / tf32 tensor-core paths (profiles/r02_precision.txt says why)",
       f"{'kernel':58s} {'UBLKCP':>7s} {'SYNCS':>6s} {'LDGSTS':>7s} {'DFMA':>6s} {'FFMA':>6s} {'FFMA2':>6s} {'SHFL':>6s} {'BAR':>5s} {'MMA':>4s}"]
KEYS = ("UBLKCP", "SYNCS", "LDGSTS", "DFMA", "FFMA2", "SHFL", "BAR")
fmt = lambda n, c: f"{n[:58]:58s} {c['UBLKCP']:7d} {c['SYNCS']:6d} {c['LDGSTS']:7d} {c['DFMA']:6d} {c['FFMA']:6d} {c['FFMA2']:6d} {c['SHFL']:6d} {c['BAR']:5d} {c['MMA']:4d}"
tot = collections.Counter()
for f in funcs[1:]:
    name = f.split('\n', 1)[0].strip()
    c = collections.Counter()
    for line in f.split('\n'):
        mm = re.search(r'/\*[0-9a-f]{4}\*/\s+(?:@!?U?P\d+\s+)?([A-Z0-9_.]+)', line)
        if not mm:
            continue
        op = mm.group(1)
        for k in KEYS:
            if op.startswith(k):
                c[k] += 1
        if op == "FFMA" or op.startswith("FFMA."):
            c["FFMA"] += 1
        if "MMA" in op:
            c["MMA"] += 1
    tot.update(c)
    short = re.sub(r'^_ZN\d+_GLOBAL__N__[0-9a-f]+_\d+_', '', name)
    short = re.sub(r'^(tce_\w+?_cu)_[0-9a-f]{8}\d+', '', short)
    if c["UBLKCP"] or c["DFMA"] > 300 or c["FFMA"] > 300 or c["LDGSTS"] or c["FFMA2"] or c["MMA"]:
        out.append(fmt(short, c))
out.append(fmt(f"TOTAL (all {len(funcs) - 1} kernels)", tot))
for f in funcs[1:]:
    if 'rsample_bulk_kernel' in f.split('\n', 1)[0]:
        lines = [l for l in f.split('\n') if re.search(r'/\*[0-9a-f]{4}\*/', l)]
        strip = lambda l: re.sub(r'\s+/\* 0x[0-9a-f]+ \*/', '', l).rstrip()
        idx = [i for i, l in enumerate(lines) if 'UBLKCP' in l][0]
        out += ["", "# rsample_bulk_kernel, around the copy request (elected thread: arrive.expect_tx, then the bulk copy) and the wait:"]
        out += [strip(l) for l in lines[max(0, idx - 8):idx + 3]]
        widx = [i for i, l in enumerate(lines) if 'PHASECHK' in l][0]
        out += ["        ..."] + [strip(l) for l in lines[max(0, widx - 2):widx + 4]]
print("\n".join(out))
