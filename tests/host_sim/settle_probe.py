"""TEST INFRASTRUCTURE: the site probe of the pending-carry settles of the verify window loops.

EDG_VERIFY_STEP (libeddsa_b200/csrc/ops.cuh) runs its public-data field operations in groups: each operation returns a
pending carry or borrow pN, the group ORs its flags, and one rarely taken branch settles the results with
pub_settle_add / pub_settle_sub.  This rewriter copies the headers and numbers those settle calls in text order (the
"sites", exactly SITES of them), so that a host build can count which sites a verification takes and can be mutated at
run time:

    if (pub_rare(p0 | p1)) { pub_settle_sub(e, p0); pub_settle_add(f, p1); }
 -> if (pub_rare(EDG_PROBE_FLAG(p0, 8) | EDG_PROBE_FLAG(p1, 9))) { EDG_PROBE_SETTLE(8, sub, e, p0, p1); EDG_PROBE_SETTLE(9, add, f, p1, p0); }

EDG_PROBE_SETTLE counts the site when its flag is set (and, separately, when no other flag of its group is), then
settles unless edg_probe_skip names the site; EDG_PROBE_FLAG leaves the flag out of the group's OR when edg_probe_drop
names the site.  Those two switches are the mutants: a settle that never runs, and a flag missing from its group.

    python settle_probe.py <src dir> <dst dir> [--ptx]    # --ptx: the inline PTX rewritten too (ptx_rewrite.py), so
                                                          # that the DEVICE paths build for the host
The product never sees any of this.
"""
import os
import re
import shutil
import subprocess
import sys

HS = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HS))
SITES = 28

GROUP_RE = re.compile(r"if \(pub_rare\(([^()]*)\)\) \{((?:\s*pub_settle_(?:add|sub)\([^;]*\);)+)\s*\}")
SETTLE_RE = re.compile(r"pub_settle_(add|sub)\(([^,()]+), (p\d)\);")

PRELUDE = """// settle probe (inserted by tests/host_sim/settle_probe.py)
#include <atomic>
#define EDG_PROBE_SITES %d
inline std::atomic<unsigned long long> edg_probe_hits[EDG_PROBE_SITES], edg_probe_alone[EDG_PROBE_SITES];   // all threads
inline thread_local unsigned edg_probe_taken = 0, edg_probe_taken_alone = 0;   // bit i: site i taken (alone in its group)
inline thread_local int edg_probe_skip = -1, edg_probe_drop = -1;              // the mutants of this thread: -1 = none
#define EDG_PROBE_FLAG(p, i) ((p) && edg_probe_drop != (i))
#define EDG_PROBE_SETTLE(i, kind, r, p, others)                                                                         \\
    do {                                                                                                                \\
        if (p) { edg_probe_hits[i].fetch_add(1, std::memory_order_relaxed); edg_probe_taken |= 1u << (i);               \\
                 if (!(others)) { edg_probe_alone[i].fetch_add(1, std::memory_order_relaxed); edg_probe_taken_alone |= 1u << (i); } } \\
        if (edg_probe_skip != (i)) pub_settle_##kind(r, p);                                                            \\
    } while (0)
// per-site counts since the last reset: taken, and taken with no other flag of its group set
extern "C" void edg_probe_counts(unsigned long long *hits, unsigned long long *alone, int reset) {
    for (int i = 0; i < EDG_PROBE_SITES; i++) {
        hits[i] = edg_probe_hits[i].load(); alone[i] = edg_probe_alone[i].load();
        if (reset) { edg_probe_hits[i] = 0; edg_probe_alone[i] = 0; }
    }
}
"""


def probe_ops(text):
    """ops.cuh -> (probed text, groups): groups[g] lists the sites of group g as (site, "add" | "sub", result, flag)."""
    groups, out, pos, site = [], [], 0, 0
    for m in GROUP_RE.finditer(text):
        flags = [f.strip() for f in m.group(1).split("|")]
        settles = SETTLE_RE.findall(m.group(2))
        assert len(settles) == len(flags) and sorted(f for _, _, f in settles) == sorted(flags), m.group(0)
        group = [(site + k, kind, res, flag) for k, (kind, res, flag) in enumerate(settles)]
        site += len(settles)
        of = {flag: s for s, _, _, flag in group}
        cond = " | ".join(f"EDG_PROBE_FLAG({f}, {of[f]})" for f in flags)
        body = " ".join(f"EDG_PROBE_SETTLE({s}, {kind}, {res}, {flag}, {' | '.join(o for o in flags if o != flag) or 'false'});"
                        for s, kind, res, flag in group)
        out.append(text[pos:m.start()])
        out.append(f"if (pub_rare({cond})) {{ {body} }}")
        pos = m.end()
        groups.append(group)
    out.append(text[pos:])
    new = "".join(out)
    if site != SITES or len(SETTLE_RE.findall(new)) != 0:
        raise SystemExit(f"settle_probe: found {site} settle sites in groups (and {len(SETTLE_RE.findall(new))} outside), "
                         f"expected {SITES}")
    assert new.count("#pragma once\n") == 1
    return new.replace("#pragma once\n", "#pragma once\n" + PRELUDE % SITES), groups


def probe_tree(src, dst, ptx=False):
    """Copy of the headers of src under dst with ops.cuh probed; ptx: the inline PTX rewritten as well.  Returns the groups."""
    if ptx:
        subprocess.run([sys.executable, os.path.join(HS, "ptx_rewrite.py"), src, dst], check=True, stdout=subprocess.DEVNULL)
    else:
        os.makedirs(dst, exist_ok=True)
        for f in os.listdir(src):
            if f.endswith((".cuh", ".h")):
                shutil.copy(os.path.join(src, f), os.path.join(dst, f))
    path = os.path.join(dst, "ops.cuh")
    new, groups = probe_ops(open(path).read())
    with open(path, "w") as fh:
        fh.write(new)
    return groups


def build(tmp, flavour, opt=("-O2",)):
    """settle_probe.cpp against a probed copy of the headers under tmp: flavour "host" (portable paths) or "device" (the
    device paths, inline PTX interpreted by ptx_emul.h).  Returns the path of the shared library."""
    gen = os.path.join(tmp, "gen_" + flavour)
    probe_tree(os.path.join(ROOT, "libeddsa_b200", "csrc"), os.path.join(gen, "libeddsa_b200", "csrc"), ptx=flavour == "device")
    so = os.path.join(tmp, f"libsettle_probe_{flavour}.so")
    cmd = ["g++", *opt, "-std=c++17", "-shared", "-fPIC", "-pthread", "-fno-gnu-unique", "-Wno-unknown-pragmas", "-I", gen]
    if flavour == "device":
        cmd += ["-D__CUDA_ARCH__=1000", "-D__CUDACC__", "-include", os.path.join(HS, "ptx_emul.h")]
    subprocess.run(cmd + ["-o", so, os.path.join(HS, "settle_probe.cpp")], check=True)
    return so


if __name__ == "__main__":
    args = [a for a in sys.argv[1:] if a != "--ptx"]
    g = probe_tree(args[0], args[1], ptx="--ptx" in sys.argv)
    print(f"probed {sum(len(x) for x in g)} settle sites in {len(g)} groups")
