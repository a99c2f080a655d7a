#!/usr/bin/env python
"""SASS instruction-mix summary of the solve kernel for profiles/ (CPU box, from what gpurun brought back).

usage: sass_mix.py <report.ncu-rep> <object file with the kernel> <PANOC iterations of the captured launch> <out.txt> "<note>"

Joins the ncu source page (executed count and stall samples per SASS instruction) with `nvdisasm -g` of the
SAME build (function boundaries, needs -lineinfo): per function the static size and the executed instructions
per PANOC iteration, the opcode mix of what is executed, the share of register moves, the hot-code footprint
in 128-byte instruction-cache lines, and where the `no_instruction` stall samples fall."""
import collections, csv, os, re, subprocess, sys, tempfile

rep, obj, iters, out_path, note = sys.argv[1], sys.argv[2], float(sys.argv[3]), sys.argv[4], sys.argv[5]
src = subprocess.run(["ncu", "-i", rep, "--page", "source", "--csv", "--print-source", "sass"], capture_output=True, text=True).stdout
rows = list(csv.reader(src.splitlines()))
kernel = rows[0][1]
hdr = rows[1]
i_no = hdr.index("stall_no_inst"); i_smp = hdr.index("# Samples"); i_thr = hdr.index("Avg. Threads Executed")
ex = []
for r in rows[2:]:
    try: ex.append((int(r[0], 16), int(r[5]), r[1].strip(), int(r[i_no]), int(r[i_smp]), float(r[i_thr])))
    except Exception: pass
base = ex[0][0]
d = tempfile.mkdtemp()
subprocess.run(["cuobjdump", "-xelf", "all", os.path.abspath(obj)], cwd=d, capture_output=True)
cub = [f for f in os.listdir(d) if f.endswith(".cubin")][0]
dis = subprocess.run(["nvdisasm", "-g", "-c", os.path.join(d, cub)], capture_output=True, text=True).stdout.split("\n")
key = re.sub(r"[^0-9]", " ", kernel.split("Dims<")[1].split(">")[0]).split()          # template arguments of the captured kernel
name = re.findall(r"\w+", kernel.split("<")[0])[-1]                                       # solve_kernel or solve_kernel_small
sec = "%d%sINS_4Dims" % (len(name), name) + "".join("ILi%sE" % key[0] if i == 0 else "Li%sE" % k for i, k in enumerate(key))
start = [i for i, l in enumerate(dis) if l.startswith(".text.") and sec in l][0]
func = "kernel body"; fn_of = {}
for l in dis[start + 1:]:
    if l.startswith("\t.section"): break
    m = re.match(r"\s*\.type\s+(\S+),@function", l)
    if m:
        n = m.group(1)
        func = ("eval_psi" if "eval_psi" in n else "wsum4v" if "wsum4v" in n else "wsum" if "4wsumEd" in n else
                "tt_div" if "tt_div" in n else "tt_sqrt" if "tt_sqrt" in n else "icm_miss" if "icm_miss" in n else
                n.split("$")[-1] if n.startswith("$__") else "kernel body")
        continue
    m = re.match(r"\s*/\*([0-9a-f]{4,})\*/\s+(.*?);", l)
    if m: fn_of[int(m.group(1), 16)] = func
assert len(fn_of) == len(ex), (len(fn_of), len(ex), "the object file is not the build that was profiled")

o = open(out_path, "w")
def P(*a): print(*a, file=o)
P("# " + note)
P("# kernel: " + kernel)
P("# source: %s joined with nvdisasm -g of %s; per PANOC iteration = executed count / %d iterations of the launch" % (rep, obj, iters))
tot = sum(e for _, e, *_ in ex)
P("\nexecuted warp instructions: %.3f G = %.0f per PANOC iteration; avg active threads %.1f" % (tot / 1e9, tot / iters, sum(e * t for _, e, _, _, _, t in ex) / tot))
P("\n## per function: static instructions, executed per PANOC iteration, share")
f = collections.OrderedDict()
for a, e, s, *_ in ex:
    k = fn_of[a - base]; v = f.setdefault(k, [0, 0]); v[0] += 1; v[1] += e
for k, v in f.items(): P("%-44s %6d static  %8.1f per iteration  %5.1f %%" % (k, v[0], v[1] / iters, 100.0 * v[1] / tot))
P("\n## opcode mix of the executed instructions (per PANOC iteration; a 64-bit select is 2 FSEL, a 64-bit shuffle 2 SHFL)")
h = collections.Counter()
for a, e, s, *_ in ex:
    t = s.split(); op = t[1] if t[0].startswith("@") else t[0]
    op = "MOV (IMAD.MOV / MOV / CS2R)" if op.startswith("IMAD.MOV") or op == "MOV" or op.startswith("CS2R") else op.split(".")[0]
    h[op] += e
for k, v in h.most_common(24): P("%-30s %8.1f  %5.1f %%" % (k, v / iters, 100.0 * v / tot))
fp64 = sum(v for k, v in h.items() if k in ("DFMA", "DMUL", "DADD", "DSETP"))
P("FP64 pipe (DFMA + DMUL + DADD + DSETP) %.1f %% of the executed instructions; register moves %.1f %%" % (100.0 * fp64 / tot, 100.0 * h["MOV (IMAD.MOV / MOV / CS2R)"] / tot))
P("\n## hot-code footprint: 128-byte lines with an instruction executed at least x times per PANOC iteration")
lines = collections.defaultdict(float)
for a, e, *_ in ex: lines[(a - base) // 128] = max(lines[(a - base) // 128], e / iters)
for thr in (2.0, 1.0, 0.3, 0.1, 0.03):
    P(">= %-5g per iteration: %5.1f KB" % (thr, sum(1 for v in lines.values() if v >= thr) / 8.0))
P("(the launch runs alone: its tail -- owners with a helper, helper polling -- is in these counts; a bulk batch touches ~1 KB less)")
P("\n## no_instruction stall samples: %d of %d samples" % (sum(x[3] for x in ex), sum(x[4] for x in ex)))
slot = collections.Counter()
for a, e, s, n, *_ in ex: slot[((a - base) % 128) // 16] += n
P("by position of the stalled instruction in its 128-byte line (0 = first): " + " ".join(str(slot[i]) for i in range(8)))
byf = collections.Counter()
for a, e, s, n, *_ in ex: byf[fn_of[a - base]] += n
P("by function: " + ", ".join("%s %d" % kv for kv in byf.most_common(8)))
o.close()
print(open(out_path).read())
