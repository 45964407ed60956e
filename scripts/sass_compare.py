"""Compares the SASS of two builds kernel by kernel: `python scripts/sass_compare.py OLD.sass NEW.sass`, each the output
of `cuobjdump -sass` on an object file.  Instructions are compared with their addresses and encodings stripped; k_trunk4
instantiations are matched by their SINGLE / FP8 arguments, a missing FP8 argument counting as false (the bf16 tower) and
the image-slot / weight-stage arguments of older builds dropped when they are the 3 / 7 that is now fixed (other ring
sizes keep them), k_encode_rows by its bf16 form, and k_ab_items by its repetition argument, the untemplated kernel counting as false
(the plain search).  Prints one line per kernel: identical, DIFFERENT or new."""
import re
import sys


def functions(path):
    out, cur = {}, None
    for line in open(path):
        m = re.match(r"\s+Function : (\S+)", line)
        if m:
            cur = out.setdefault(m.group(1), [])
            continue
        m = re.match(r"\s+/\*[0-9a-f]+\*/\s+(.*?);", line)
        if cur is not None and m:
            cur.append(m.group(1).strip())
    return out


def key(name):
    m = re.match(r"_ZN3crl8k_trunk4I(?:Li(\d+)ELi(\d+)E)?Lb(\d)E(?:Lb(\d)E)?", name)
    if m:
        ring = "" if m.group(1) in (None, "3") and m.group(2) in (None, "7") else "%s,%s," % (m.group(1), m.group(2))
        return "k_trunk4<%s%s,%s>" % (ring, m.group(3), m.group(4) or "0")
    if re.match(r"_ZN3crl13k_encode_rows(ENS_5Pools|I13__nv_bfloat16E)", name):
        return "k_encode_rows<bf16>"
    m = re.match(r"_ZN3crl10k_ab_items(?:ILb(\d)EE)?", name)
    if m:
        return "k_ab_items<%s>" % (m.group(1) or "0")
    return name


def main(old, new):
    a = {key(k): v for k, v in functions(old).items()}
    b = {key(k): v for k, v in functions(new).items()}
    for k in sorted(a):
        print("%-9s %s (%d -> %d instructions)" % ("identical" if a[k] == b.get(k) else "DIFFERENT", k, len(a[k]),
                                                  len(b.get(k, []))))
    for k in sorted(set(b) - set(a)):
        print("new       %s (%d instructions)" % (k, len(b[k])))


if __name__ == "__main__":
    main(sys.argv[1], sys.argv[2])
