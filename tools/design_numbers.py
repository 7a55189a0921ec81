"""Regenerates the measured tables of DESIGN.md (the blocks between <!-- BEGIN:x --> / <!-- END:x --> markers) from the
committed evidence files, so that the document always quotes the files it names.

    python tools/design_numbers.py [<tag> [--bench-tag <tag2>] [--kbench-tag <tag3>]] [--check]   (no tag: profiles/CURRENT.json)

reads profiles/bench_<tag>.json, profiles/launches_<tag>_summary.txt, profiles/traffic.json,
profiles/kbench_1440x720_<tag>.txt, profiles/kbench_4320x2160_<tag>.txt; --check only reports whether DESIGN.md is current.
The bench line and the kbench files may come from a later checkpoint than the ncu captures (--bench-tag, --kbench-tag)."""
import json, os, re, sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
P = lambda *a: os.path.join(ROOT, "profiles", *a)
pos = [a for i, a in enumerate(sys.argv[1:], 1) if not a.startswith("--") and sys.argv[i - 1] not in ("--bench-tag", "--kbench-tag")]
if pos:
    tag = pos[0]
    btag = sys.argv[sys.argv.index("--bench-tag") + 1] if "--bench-tag" in sys.argv else tag   # bench line of a later checkpoint
    ktag = sys.argv[sys.argv.index("--kbench-tag") + 1] if "--kbench-tag" in sys.argv else tag
else:                                    # the checkpoint DESIGN.md currently quotes
    cur = json.load(open(P("CURRENT.json")))
    tag, btag, ktag = cur["tag"], cur["bench_tag"], cur.get("kbench_tag", cur["tag"])
bench = json.loads(open(P(f"bench_{btag}.json")).read().strip().splitlines()[-1])
traffic = json.load(open(P("traffic.json")))
NAMES = {"ncar": "NCAR", "andreas": "ANDREAS", "coare3p0": "COARE 3.0", "coare3p6": "COARE 3.6", "ecmwf": "ECMWF",
         "coare3p0+skin": "COARE 3.0 + skin", "coare3p6+skin": "COARE 3.6 + skin", "ecmwf+skin": "ECMWF + skin"}
ALG_BYTES = {False: 88, "coare": 176, "ecmwf": 128}


def block(name, text, s):
    a, b = f"<!-- BEGIN:{name} -->\n", f"<!-- END:{name} -->"
    i, j = s.index(a) + len(a), s.index(b)
    return s[:i] + text.rstrip("\n") + "\n" + s[j:]


# ---- ncu table (1440x720 captures behind traffic.json)
rows = ["| kernel | µs | FP64 pipe active | issue slots | lanes / instr | FP64 thread-instr / pt | registers | spill instr / pt | DRAM B/pt (algorithmic) |",
        "|---|---|---|---|---|---|---|---|---|"]
for k in ("ncar", "andreas", "coare3p0", "coare3p6", "ecmwf", "coare3p0+skin", "coare3p6+skin", "ecmwf+skin"):
    t = traffic[k]
    alg = 88 if "+skin" not in k else (128 if k.startswith("ecmwf") else 176)
    extra = ""
    if f"{k}@nb30" in traffic:
        extra = f" ({traffic[f'{k}@nb30']['pipe_fp64_pct']:.1f} % at nb_iter 30)"
    rows.append(f"| {NAMES[k]}{' (Rsw > 0)' if '+skin' in k else ''} | {t['duration_us']:.1f} | {t['pipe_fp64_pct']:.1f} %{extra} | {t['issue_pct']:.1f} % | "
                f"{t['lanes_per_inst']:.1f} | {t['fp64_thread_inst_per_point']:.0f} | {t['registers']:.0f} | {t['spill_inst_per_point']:.0f} | {t['dram_bytes_per_point']:.1f} ({alg}) |")
c2 = traffic.get("coare3p6+skin@C2session")
if c2:
    rows.append(f"| COARE 3.6 + skin, mean of the 24 launches of a C2 session | {c2['duration_us']:.1f} | {c2['pipe_fp64_pct']:.1f} % | {c2['issue_pct']:.1f} % | "
                f"{c2['lanes_per_inst']:.1f} | {c2['fp64_thread_inst_per_point']:.0f} | 80 | – | – |")
ncu_table = "\n".join(rows)

# ---- headline
K = bench["kernels"]
cb = bench["cpu_baseline"]
gap = bench["ms_per_step"] - sum(k["avg_launch_ms"] for k in K)
fr = [k["fp64_frac"] for k in K]
head = "\n".join([
    "| | |", "|---|---|",
    f"| `value` (device-resident, 7 variants × 84 M) | **{bench['value'] / 1e9:.2f} Gpt/s**, {bench['ms_per_step']:.1f} ms per step (round 1 code on the same bench: 3.58 Gpt/s, 164.4 ms) |",
    "| flux kernels, ms per 84 M-point launch | " + " · ".join(f"{NAMES[k['variant']]} {k['avg_launch_ms']:.2f}" for k in K) + " |",
    "| FP64 roofline fraction per kernel (executed) | " + " · ".join(f"{f:.2f}" for f in fr) +
    f" -- `roofline.frac` = **{bench['roofline']['frac']:.2f}** ({NAMES[bench['roofline']['variant']]}, the longest) |",
    "| the same counting only active lanes (fraction × lanes per instruction / 32, ncu) | " + " · ".join(
        f"{k['fp64_frac'] * (k.get('ncu_lanes') or traffic[k['variant']]['lanes_per_inst']) / 32:.2f}" for k in K) + " |",
    f"| not flux: statistics ×7, classify ×6, small launches | {gap:.1f} ms of the step (round 1 code: 15.6 ms) |",
    f"| `e2e` pinned / pageable | {bench['e2e']['value'] / 1e9:.2f} / {bench['e2e_pageable']['value'] / 1e9:.2f} Gpt/s (PCIe-bound: 94.9 B per point evaluation) |",
    f"| CPU port, {cb['cores']} threads / 1 thread | {cb['value'] / 1e6:.2f} / {cb['serial_value'] / 1e6:.3f} Mpt/s → `e2e` ≈ {bench['e2e']['value'] / cb['value']:.0f}× the {cb['cores']}-thread figure, `value` ≈ {bench['value'] / cb['value']:.0f}× |",
    f"| in-bench parity probe (8 rows × 7 variants of the timed arrays) | max scaled error {bench['parity']['max_scaled_err']:.1e} (gate 1e-10) |",
])

# ---- launch shares
sh = {}
for l in open(P(f"launches_{tag}_summary.txt")):
    p = l.split()
    if not p or l.startswith("kernel"):
        continue
    sh[l[:60].strip()] = float(p[-1].rstrip("%"))
flux = sum(v for k, v in sh.items() if "flux_kernel" in k)
pick = lambda pre: next(v for k, v in sh.items() if k.startswith(pre))
shares = (f"The launch list (ncu, cold-cache and serialised, shares only; `profiles/launches_{tag}_summary.txt`) agrees: the seven `flux_kernel`\n"
          f"instantiations are {flux:.1f} % of the GPU time of the command, `stats_fast_kernel` {pick('stats_fast'):.1f} %, `classify_kernel` {pick('classify'):.1f} %\n"
          f"(the DFMA peak measurement {pick('dfma_peak'):.1f} %, everything else below 0.3 %).")

# ---- per_config
rows = ["| config | device-resident | flux kernel, roofline | end to end pinned / pageable | CPU 16 thr / 1 thr |", "|---|---|---|---|---|"]
for c in bench["per_config"]:
    cbc = c["cpu_baseline"]
    for j, x in enumerate(c["runs"]):
        name = c["config"] + " " + NAMES[x["variant"]] + (f" nb_iter {x['nb_iter']}" if c["config"] == "C4" else "") + (" × 24 steps" if c["config"] == "C2" else "")
        cpu = f"{cbc['value'] / 1e6:.2f} / {cbc['serial_value'] / 1e6:.3f} M" if j == 0 else ""
        fr_ = x["roofline"]["frac"]
        rows.append(f"| {name} ({c['grid'][0]}×{c['grid'][1]}) | {x['gpts']:.2f} Gpt/s ({x['ms']:.3f} ms) | {x['flux_kernel_avg_ms']:.3f} ms, {fr_:.2f} | "
                    f"{x['e2e']['pinned_gpts']:.2f} / {x['e2e']['pageable_gpts']:.2f} Gpt/s | {cpu} |")
per_config = "\n".join(rows)


# ---- kbench
def kb(path):
    out = {}
    for l in open(path):
        m = re.match(r"(\w+)\s+skin=(\d)\s+(\S+)\s*:\s*([\d.]+) ms\s+([\d.]+) Mpt/s", l)
        if m:
            out[(m.group(1), m.group(2) == "1", m.group(3))] = (float(m.group(4)), float(m.group(5)) / 1e3)
    return out


small, large = kb(P(f"kbench_1440x720_{ktag}.txt")), kb(P(f"kbench_4320x2160_{ktag}.txt"))
rows = ["| algorithm | 1440×720 (C2 size) | 4320×2160 (C3/C4 size) |", "|---|---|---|"]
one = lambda d, k: f"{d[k][0]:.3f} ms · {d[k][1]:.1f} Gpt/s"
two = lambda d, a, b: f"{d[a][0]:.3f} / {d[b][0]:.3f} ms · {d[a][1]:.1f} / {d[b][1]:.1f} Gpt/s"
rows.append(f"| NCAR | {one(small, ('ncar', False, '-'))} | {one(large, ('ncar', False, '-'))} |")
rows.append(f"| ANDREAS | {one(small, ('andreas', False, '-'))} | {one(large, ('andreas', False, '-'))} |")
rows.append(f"| COARE 3.0 / 3.6 | {two(small, ('coare3p0', False, '-'), ('coare3p6', False, '-'))} | {two(large, ('coare3p0', False, '-'), ('coare3p6', False, '-'))} |")
rows.append(f"| ECMWF | {one(small, ('ecmwf', False, '-'))} | {one(large, ('ecmwf', False, '-'))} |")
for a, n in (("coare3p6", "COARE 3.6"), ("ecmwf", "ECMWF")):
    rows.append(f"| {n} + skin, night / day | {two(small, (a, True, 'night'), (a, True, 'day'))} | {two(large, (a, True, 'night'), (a, True, 'day'))} |")
kbench = "\n".join(rows)

path = os.path.join(ROOT, "DESIGN.md")
old = open(path).read()
new = old
for name, text in (("ncu-table", ncu_table), ("headline-table", head), ("launch-shares", shares), ("per-config-table", per_config), ("kbench-table", kbench)):
    new = block(name, text, new)
if "--check" in sys.argv:
    print("DESIGN.md tables are current" if new == old else "DESIGN.md tables are STALE for tag " + tag)
    sys.exit(0 if new == old else 1)
open(path, "w").write(new)
print("DESIGN.md tables regenerated from tag", tag)
