"""tools/sass_regions.py [lib.so | obj.o | .cubin] [--kernel NAME] [--src frontier_pack.cu]: static SASS of one trip of
frontier_pack_kernel (one group of R runs), split the way the source splits it:

  ticket -> walk dispatch   ticket draw, barrier wait, header, planes, stages G / B / I, D-prep, stage C, walk table, the
                            first two prefetch links (load_sid, load_ent) and the format dispatch of the walk
  walk                      the walk functions (walk_items, walk_items_k, walk_items_any and what they inline), every
                            instance; below, the contiguous blocks of the 8-word byte-row branch of walk_items_k (one block per
                            K = 4 / 2 / 1 batch and failed-dependency instance)
  after the walk            cond masking and the fix-up loop, stage E, the head / defer branches and the re-arm (issue)

Instructions are attributed by `nvdisasm -gi` line info: a line of the source, or the line of the source a helper was
inlined at.  The prefetch lambdas are also inlined by the prologue; their instructions placed before the loop count as
prologue.  Counts are static (every branch once, rare ones included), so they compare builds, not trips.
Needs no GPU: `cuobjdump -xelf` + `nvdisasm` of the sm_100a cubin."""
import argparse
import collections
import glob
import os
import re
import subprocess
import sys
import tempfile

ap = argparse.ArgumentParser()
ap.add_argument("lib", nargs="?", default="bobrapet_b200/lib/obj/frontier_pack.cu.o")
ap.add_argument("--kernel", default="void bf::frontier_pack_kernel<false, false>(bf::KParams)")
ap.add_argument("--src", default=os.path.join(os.path.dirname(os.path.abspath(__file__)), "..", "bobrapet_b200", "csrc", "frontier_pack.cu"),
                help="the frontier_pack.cu the binary was compiled from (source anchors; for another build pass its source)")
a = ap.parse_args()

src = open(a.src).read().splitlines()


def find(pat, start=0):
    for i in range(start, len(src)):
        if re.search(pat, src[i]):
            return i + 1   # 1-based line
    sys.exit("anchor %r not found in %s" % (pat, a.src))


def body(start_pat, close="^}"):   # [first, last] line of a function / lambda whose header matches start_pat
    s = find(start_pat)
    return s, find(close, s)


walk_k = body(r"DI void walk_items_k\(")
walk_al = (find(r"if \(AL && FMT == FMT_ELL4B\)", walk_k[0]), find(r"^\s+return;", walk_k[0]))
walk_fns = [walk_k, body(r"DI void walk_items\("), body(r"DI void walk_items_any\(")]
lambdas = {name: body(r"auto %s = \[&\]" % name, "^  };") for name in ("load_sid", "load_ent", "issue")
           if any("auto %s = [&]" % name in x for x in src)}   # load_ent: builds before the slot entry went through shared memory
kern = find(r"frontier_pack_kernel\(const KParams P\)")
loop0 = find(r"^\s+for \(;;\) \{", kern)
after0 = find(r"met_w \|= FREE;", loop0)
loop1 = find(r"^  }$", after0)
general_i = None   # the general stage I, which groups of main-only runs skip
if any("if (main_only) {" in x for x in src):
    general_i = (find(r"^    \} else \{", find(r"if \(main_only\) \{", loop0)), find(r"^    \}$", find(r"if \(main_only\) \{", loop0) + 1))
lam_region = {"load_sid": "ticket -> walk dispatch", "load_ent": "ticket -> walk dispatch", "issue": "after the walk"}

with tempfile.TemporaryDirectory() as td:
    path = os.path.abspath(a.lib)
    if not path.endswith(".cubin"):
        subprocess.run(["cuobjdump", "-xelf", "all", path], cwd=td, check=True, capture_output=True)
        cubins = [c for c in glob.glob(os.path.join(td, "*.cubin")) if "sm_100" in c]
        cubins = [c for c in cubins if "frontier_pack" in os.path.basename(c)] or cubins
        if not cubins:
            sys.exit("no sm_100 cubin in %s" % path)
        path = cubins[0]
    dis = subprocess.run(["nvdisasm", "-gi", path], capture_output=True, text=True, check=True).stdout

base = os.path.basename(a.src)
ann_re = re.compile(r'//## File "([^"]+)", line (\d+)(?: inlined at "([^"]+)", line (\d+))?')
ins_re = re.compile(r"^\s+/\*([0-9a-f]{4,})\*/\s+(\S.*?)\s*;")
fn_re = re.compile(r"^\.text\.(\S+):$")
insts, cur, anns, fresh = [], None, [], False   # (address, [(file, line, inl_file, inl_line)], text) of the kernel
for ln in dis.splitlines():   # an annotation holds for every instruction up to the next one
    m = fn_re.match(ln)
    if m:
        name = subprocess.run(["c++filt", m.group(1)], capture_output=True, text=True).stdout.strip()
        cur = name == a.kernel
        continue
    if not cur:
        continue
    m = ann_re.search(ln)
    if m:
        if not fresh:
            anns, fresh = [], True
        anns.append((os.path.basename(m.group(1)), int(m.group(2)), m.group(3) and os.path.basename(m.group(3)),
                     int(m.group(4)) if m.group(4) else 0))
        continue
    m = ins_re.match(ln)
    if m:
        insts.append((int(m.group(1), 16), anns, m.group(2)))
        fresh = False
if not insts:
    sys.exit("kernel %r not found" % a.kernel)


def inside(line, rng):
    return rng[0] <= line <= rng[1]


def classify(anns):
    """-> (bucket, source line): the walk, a prefetch lambda, or a line of the kernel body"""
    for f, l, fi, li in anns:
        for ln in ((l if f == base else 0), (li if fi == base else 0)):
            if any(inside(ln, r) for r in walk_fns):
                return "walk", ln
    for f, l, fi, li in sorted(anns, key=lambda x: x[2] is None):   # prefer the annotation with inlining info
        ln = li if fi == base else (l if f == base else 0)
        for name, r in lambdas.items():
            if inside(ln, r) or (f == base and inside(l, r)):
                return name, ln
        if ln:
            return "kernel", ln
    return "other", 0


rows = [(addr, *classify(an), an, txt) for addr, an, txt in insts]
trip0 = min(addr for addr, b, ln, _, _ in rows if b == "kernel" and loop0 <= ln < after0)
trip1 = max(addr for addr, b, ln, _, _ in rows if b == "walk" or (b == "kernel" and loop0 <= ln <= loop1))
count = collections.Counter()
for addr, b, ln, an, txt in rows:
    if b == "walk":
        count["walk"] += 1
    elif b in lambdas:
        count[lam_region[b] if addr >= trip0 else "prologue"] += 1
    elif b == "kernel" and loop0 <= ln < after0:
        count["ticket -> walk dispatch"] += 1
        if general_i and inside(ln, general_i):
            count["  of which general stage I"] += 1
    elif b == "kernel" and after0 <= ln <= loop1:
        count["after the walk"] += 1
    elif b == "kernel" and trip0 <= addr <= trip1:
        count["setup lines inside the trip"] += 1   # loop invariants the register allocator rematerialises
    elif b == "kernel":
        count["outside the loop"] += 1
    else:
        count["no line of the source"] += 1   # a helper inlined into a helper (the walks of the other row formats)

# the 8-word byte-row batches: contiguous runs of instructions on lines of that branch (or inlined there)
blocks, run = [], 0
for addr, b, ln, an, txt in rows:
    hit = b == "walk" and any((f == base and inside(l, walk_al)) or (fi == base and inside(li, walk_al)) for f, l, fi, li in an)
    if hit:
        run += 1
    elif run:
        blocks.append(run)
        run = 0
if run:
    blocks.append(run)

print("# %s  %s  (source %s: loop %d-%d, walk dispatch ends / after-walk starts at %d)" %
      (os.path.basename(a.lib), a.kernel, base, loop0, loop1, after0))
for k in ("ticket -> walk dispatch", "  of which general stage I", "walk", "after the walk", "setup lines inside the trip", "prologue", "outside the loop",
          "no line of the source"):
    print("%-28s %6d" % (k, count[k]))
print("%-28s %6d" % ("trip outside the walk", count["ticket -> walk dispatch"] + count["after the walk"] + count["setup lines inside the trip"]))
print("%-28s %s" % ("8-word byte-row blocks", " ".join(str(x) for x in blocks if x >= 8)))
