"""Compare the kernels of two builds of libvss_b200.so, kernel by kernel, from `cuobjdump -sass` listings.

Each kernel of the first listing is reported as byte-identical SASS, as the same instruction count per opcode (what
ptxas gives for the tcgen05 kernels of tc_gemm.cu / mlp_fused.cu from one source: two builds of the same commit differ
in uniform-register allocation), or as different; kernels only in the second listing are listed as new.

    cuobjdump -sass old/libvss_b200.so > old.sass; cuobjdump -sass new/libvss_b200.so > new.sass
    python profiles/sass_compare.py old.sass new.sass
"""
import collections
import re
import sys


def kernels(path):
    out, cur, buf = {}, None, []
    for line in open(path):
        m = re.match(r"\s+Function : (\S+)", line)
        if m:
            if cur:
                out.setdefault(cur, []).append("".join(buf))
            cur, buf = m.group(1), []
        elif cur is not None:
            buf.append(line)
    if cur:
        out.setdefault(cur, []).append("".join(buf))
    return out


def opcode_counts(text):
    c = collections.Counter()
    for line in text.splitlines():
        m = re.match(r"\s+/\*[0-9a-f]+\*/\s+(?:@!?U?P\w+\s+)?([A-Z][A-Z0-9_.]*)", line)
        if m:
            c[m.group(1)] += 1
    return c


def main(old_path, new_path):
    a, b = kernels(old_path), kernels(new_path)
    rows = collections.defaultdict(list)
    for k in a:
        if k not in b:
            rows["missing"].append(k)
        elif a[k] == b[k]:
            rows["byte-identical"].append(k)
        elif [opcode_counts(x) for x in a[k]] == [opcode_counts(x) for x in b[k]]:
            rows["same opcode counts"].append(k)
        else:
            rows["different"].append(k)
    rows["new"] = [k for k in b if k not in a]
    print(f"{len(a)} kernels in {old_path}: " + ", ".join(f"{len(v)} {k}" for k, v in rows.items()))
    for kind in ("same opcode counts", "different", "missing", "new"):
        for k in rows[kind]:
            print(f"  {kind}: {k}")
    for k in rows["byte-identical"]:
        print(f"  byte-identical: {k}")
    return 1 if rows["different"] or rows["missing"] else 0


if __name__ == "__main__":
    sys.exit(main(sys.argv[1], sys.argv[2]))
