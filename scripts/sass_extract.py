"""SASS extracts of the hot kernels for profiles/: static opcode histogram, the mnemonics that prove TMA / packed fp32 /
mbarrier use, register + shared-memory footprint, and (for the refine kernel) the unrolled main loop.
usage: python scripts/sass_extract.py [lib.so] [out_dir]"""
import collections, os, re, subprocess, sys
lib = sys.argv[1] if len(sys.argv) > 1 else "unmore_b200/libunmore_b200.so"
out_dir = sys.argv[2] if len(sys.argv) > 2 else "profiles"
sass = subprocess.run(["cuobjdump", "-sass", lib], capture_output=True, text=True).stdout
res = subprocess.run(["cuobjdump", "-res-usage", lib], capture_output=True, text=True).stdout
funcs = {}
cur = None
for line in sass.splitlines():
    m = re.search(r"Function : (\S+)", line)
    if m:
        cur = m.group(1); funcs[cur] = []; continue
    m = re.match(r"\s+/\*([0-9a-f]{4,5})\*/\s+(.*?);\s+/\*", line)
    if m and cur:
        funcs[cur].append((m.group(1), m.group(2).strip()))
usage = {}
name = None
for line in res.splitlines():
    m = re.search(r"Function (\S+):", line)
    if m: name = m.group(1); continue
    if name and "REG:" in line: usage[name] = line.strip(); name = None
want = [("refine_kernelILi640", "refine_kernel_640", True), ("center_kernelILb0ELi307200ELb1", "center_kernel_spec", False), ("center_kernelILb0ELi307200ELb0", "center_kernel_spec_second_pass", False),
        ("rle_counts_kernelILb1", "rle_counts_kernel", False),
        ("16existence_kernelE", "existence_kernel", False), ("sat_kernel_tmaILi5", "sat_kernel_tma_5", False),
        ("pack_kernel_vec", "pack_kernel_vec", False), ("score_kernel", "score_kernel", False)]
KEY = ["UBLKCP", "UTMALDG", "SYNCS", "FFMA2", "FMUL2", "FADD2", "LDGSTS", "MUFU", "LDG", "LDS", "STS", "SHFL", "VOTE", "POPC", "IMAD", "BAR", "WARPSYNC"]
for pat, tag, want_loop in want:
    fn = next((f for f in funcs if pat in f), None)
    if fn is None: continue
    ins = funcs[fn]
    hist = collections.Counter()
    for _, t in ins:
        toks = t.split()
        op = toks[1] if toks[0].startswith("@") else toks[0]
        hist[op.split(".")[0]] += 1
    with open(os.path.join(out_dir, f"r02_sass_{tag}.txt"), "w") as f:
        f.write(f"# {fn}\n# {usage.get(fn, '')}\n# {len(ins)} SASS instructions (static); cuobjdump -sass of {os.path.basename(lib)}, sm_100a\n")
        f.write("# key mnemonics: " + ", ".join(f"{k} {hist[k]}" for k in KEY if hist[k]) + "\n# static opcode histogram:\n")
        for k, v in hist.most_common():
            f.write(f"#   {k:12s} {v}\n")
        if want_loop:
            # the main loop = the span between the first and the last MUFU.SQRT of the largest backward branch body
            idx = [i for i, (_, t) in enumerate(ins) if "MUFU.SQRT" in t]
            back = [(i, int(re.search(r"0x([0-9a-f]+)", t).group(1), 16)) for i, (a, t) in enumerate(ins) if re.search(r"BRA 0x", t) and int(re.search(r"0x([0-9a-f]+)", t).group(1), 16) < int(a, 16)]
            best = None
            for i, tgt in back:
                j = next((k for k, (a, _) in enumerate(ins) if int(a, 16) == tgt), None)
                if j is not None and any(j <= q <= i for q in idx) and (best is None or i - j > best[1] - best[0]) and i - j < 900:
                    best = (j, i)
            if best:
                f.write(f"\n# main loop (two output rows per iteration), {best[1] - best[0] + 1} instructions:\n")
                for a, t in ins[best[0]:best[1] + 1]:
                    f.write(f"/*{a}*/ {t} ;\n")
        else:
            f.write("\n# lines with TMA / mbarrier / packed-fp32 mnemonics:\n")
            shown = 0
            for a, t in ins:
                if any(k in t for k in ("UBLKCP", "SYNCS", "FFMA2", "UTMALDG")) and shown < 40:
                    f.write(f"/*{a}*/ {t} ;\n"); shown += 1
    print(tag, len(ins), {k: hist[k] for k in KEY if hist[k]})
