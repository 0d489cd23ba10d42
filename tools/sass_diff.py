"""Compare the SASS of two builds of libhpdecode.so kernel by kernel.

usage: python tools/sass_diff.py OLD.so NEW.so [PATTERN ...]  ->  one line per kernel of OLD whose demangled name
contains one of the patterns (default: every kernel): "identical", "DIFFERS" or "missing", plus the kernels only NEW has.
A kernel of NEW that gained a trailing `float` template argument (the element type of the inputs) is compared with the
OLD kernel without it, and the aggregation kernels that lost their tag-map arguments with the OLD tag-less variants:
agg_nms_x2_kernel<E, NW, T, false> -> <NW, T>, agg_nms_ms_kernel<E, NW, NS, T> -> <NW, NS, T> (both E of OLD map to
the one NEW kernel), and track_kernel<false> with the untemplated OLD track_kernel.  Instruction text and encodings
are compared; only the offset comments and the padding between them are dropped.
Needs only the CUDA toolkit (cuobjdump, c++filt): no GPU.
"""
import re
import subprocess
import sys


def kernels(lib):
    txt = subprocess.run(["cuobjdump", "-sass", lib], capture_output=True, text=True, check=True).stdout
    out, cur = {}, None
    for line in txt.splitlines():
        m = re.match(r"\s*Function : (\S+)", line)
        if m:
            cur = out.setdefault(m.group(1), [])
            continue
        if cur is not None and line.strip().startswith("/*"):
            # cuobjdump pads the encoding comment to a column that depends on the listing: whitespace is not compared
            cur.append(re.sub(r"\s+", " ", re.sub(r"^\s*/\*[0-9a-f]{4,}\*/", "", line).strip()))
    names = subprocess.run(["c++filt"], input="\n".join(out), capture_output=True, text=True).stdout.splitlines()
    return {strip_params(re.sub(r"^void ", "", n)): v for n, v in zip(names, out.values())}


def strip_params(name):
    """Demangled signature -> name: drops the trailing parameter list, whose parentheses balance (a name may hold
    `(anonymous namespace)`)."""
    if not name.endswith(")"):
        return name
    depth = 0
    for i in range(len(name) - 1, -1, -1):
        depth += {")": 1, "(": -1}.get(name[i], 0)
        if depth == 0:
            return name[:i]
    return name


def without_tag_args(name):
    """OLD name of a kernel with tag-map template arguments -> its name without them."""
    name = re.sub(r"(agg_nms_x2_kernel)<\d, (.*), false>$", r"\1<\2>", name)
    return re.sub(r"(agg_nms_ms_kernel)<\d, (\d, \d, [^,]+)>$", r"\1<\2>", name)


def main(old_lib, new_lib, patterns):
    old, new = kernels(old_lib), kernels(new_lib)
    alias = {re.sub(r", float>$", ">", n): n for n in new}   # new name without the float element type -> new name
    alias.update({n[:-len("<false>")]: n for n in new if n.endswith("track_kernel<false>")})
    seen, rows = set(), []
    for name in sorted(old):
        if patterns and not any(p in name for p in patterns):
            continue
        twin = name if name in new else alias.get(name) or (without_tag_args(name) if without_tag_args(name) in new else None)
        if twin is None:
            rows.append(("missing", name, "", len(old[name])))
            continue
        seen.add(twin)
        rows.append(("identical" if old[name] == new[twin] else "DIFFERS", name, twin, len(old[name])))
    for name in sorted(new):
        if name not in seen and (not patterns or any(p in name for p in patterns)):
            rows.append(("new", "", name, len(new[name])))
    for status, o, n, lines in rows:
        print("%-9s %6d  %s%s" % (status, lines // 2, o or n, "  ->  " + n if o and n and n != o else ""))
    return 1 if any(r[0] in ("DIFFERS", "missing") for r in rows) else 0


if __name__ == "__main__":
    sys.exit(main(sys.argv[1], sys.argv[2], sys.argv[3:]))
