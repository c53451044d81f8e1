"""Summary of scripts/r3_pruned_tail.sh: python scripts/r3_pruned_tail_summary.py <dir>  ->  markdown on stdout."""
import glob
import json
import os
import statistics
import sys

import numpy as np


def line(path):
    try:
        with open(path) as f:
            return json.loads(f.read().strip().splitlines()[-1])
    except Exception as e:            # a failed run is reported, not hidden
        return {"error": repr(e)}


def dumps_equal(d0, d1):
    names = sorted(os.path.basename(p) for p in glob.glob(os.path.join(d0, "*.npy")))
    if not names or names != sorted(os.path.basename(p) for p in glob.glob(os.path.join(d1, "*.npy"))):
        return False, names
    return all(np.array_equal(np.load(os.path.join(d0, n)), np.load(os.path.join(d1, n))) for n in names), names


def main(d):
    print("## Environment\n")
    print("```\n" + open(os.path.join(d, "env.txt")).read().strip() + "\n```\n")
    print("## Outputs, VB200_PRUNE=0 vs 1 (np.array_equal)\n")
    for w in ("vqa", "mt"):
        ok, names = dumps_equal(os.path.join(d, f"dump_{w}_p0"), os.path.join(d, f"dump_{w}_p1"))
        print(f"- {w}: {'identical' if ok else 'DIFFERENT'} ({', '.join(names)})")
    print()
    for steps in (200, 40):
        print(f"## {steps} steps, ABBA x 4\n")
        print("| run | arm | bf16 value | fp16 alt value | e2e | sm MHz median | clock reasons |")
        print("|---|---|---|---|---|---|---|")
        vals = {0: [], 1: [], "alt0": [], "alt1": []}
        for i in range(1, 5):
            order = (0, 1) if i % 2 else (1, 0)
            for a in order:
                r = line(os.path.join(d, f"s{steps}_p{a}_{i}.json"))
                if "value" not in r:
                    print(f"| {i} | {a} | failed: {r.get('error')} | | | | |")
                    continue
                alt = r.get("alt", {}).get("fp16", {})
                c = r.get("clocks", {})
                vals[a].append(r["value"])
                vals[f"alt{a}"].append(alt.get("value"))
                print(f"| {i} | {'B (pruned)' if a else 'A (full)'} | {r['value']:.0f} | {alt.get('value', 0):.0f} | "
                      f"{r.get('e2e', {}).get('value', 0):.0f} | {c.get('sm_mhz')} | {','.join(c.get('reasons', []))} |")
        if vals[0] and vals[1]:
            m0, m1 = statistics.median(vals[0]), statistics.median(vals[1])
            a0, a1 = statistics.median(vals["alt0"]), statistics.median(vals["alt1"])
            print(f"\nmedian bf16: A {m0:.0f}, B {m1:.0f} pairs/s ({100 * (m1 / m0 - 1):+.2f} %); every B > every A: "
                  f"{min(vals[1]) > max(vals[0])}")
            print(f"median fp16 alt: A {a0:.0f}, B {a1:.0f} pairs/s ({100 * (a1 / a0 - 1):+.2f} %)\n")
    print("## Reported, not gated\n")
    print("| run | A (full tail) | B (pruned) | change |")
    print("|---|---|---|---|")
    for tag, name in (("dump_mt", "multitask, 40 steps"), ("b512", "batch 512, 40 steps"), ("retr", "retrieval 250 x 250, 1 GPU")):
        r0, r1 = line(os.path.join(d, f"{tag}_p0.json")), line(os.path.join(d, f"{tag}_p1.json"))
        if "value" in r0 and "value" in r1:
            print(f"| {name} | {r0['value']:.0f} | {r1['value']:.0f} | {100 * (r1['value'] / r0['value'] - 1):+.2f} % |")
        else:
            print(f"| {name} | {r0.get('value', r0.get('error'))} | {r1.get('value', r1.get('error'))} | |")
    for a in (0, 1):
        r = line(os.path.join(d, f"dump_vqa_p{a}.json"))
        print(f"\nVQA batch 64, arm {'B' if a else 'A'}: launches/step {r.get('launches_per_step')}, "
              f"whole_step_tflops {r.get('roofline', {}).get('whole_step_tflops', r.get('whole_step_tflops'))}")
    print("\n## Per-launch table of the tail shapes (isolated replays, us per launch)\n")
    for a in (0, 1):
        p = os.path.join(d, f"ops_p{a}.jsonl")
        if not os.path.exists(p):
            continue
        rows = [json.loads(x) for x in open(p)]
        tail = [r for r in rows if r["dims"][0] == 64 or r["kind"] == "self_attention"]
        print(f"arm {'B' if a else 'A'}: " + "; ".join(f"{r['kind']} {r['dims']} x{r['launches']} {r['us']}" for r in tail))
        print(f"  serialised total {sum(r['total_us'] for r in rows):.1f} us\n")


if __name__ == "__main__":
    main(sys.argv[1])
