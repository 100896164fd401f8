"""Function-by-function comparison of the kernel images of two builds of libpom_b200.so (no GPU needed).

    python tools/sass_compare.py OLD.so NEW.so

For every kernel of OLD it finds the kernel of NEW that is the same instantiation, compares the SASS (cuobjdump -sass)
line by line, instruction encodings and their control bits included, and the resource usage (cuobjdump -res-usage:
registers, stack, shared, local and constant memory), and prints one JSON line per kernel and a summary line.  Exit code 0 when every kernel of OLD is in NEW unchanged.

Two names are the same instantiation when they differ only by trailing template arguments `false` that NEW added with
that default (a kernel template that gained `bool X = false`, or a plain kernel that became `template<bool X = false>`):
the default instantiation is the old kernel, so it must compile to the same code.  Kernels only NEW has are listed as
new."""
import json
import re
import subprocess
import sys

CUOBJDUMP = "/usr/local/cuda/bin/cuobjdump"


def _sections(text, head):
    out, name, body = {}, None, []
    for line in text.splitlines():
        m = re.match(r"\s*" + head + r"\s*:?\s*(\S+?):?\s*$", line)
        if m:
            if name:
                out[name] = body
            name, body = m.group(1), []
        elif name:
            body.append(line)
    if name:
        out[name] = body
    return out


def sass(lib):
    text = subprocess.run([CUOBJDUMP, "-sass", lib], capture_output=True, text=True, check=True).stdout
    out = {}
    for name, body in _sections(text, "Function").items():
        # every instruction with both 64-bit encoding words (the second carries the scheduling control bits)
        out[name] = [" ".join(line.split()) for line in body if "/* 0x" in line]
    return out


def res_usage(lib):
    text = subprocess.run([CUOBJDUMP, "-res-usage", lib], capture_output=True, text=True, check=True).stdout
    out, name = {}, None
    for line in text.splitlines():
        m = re.match(r"\s*Function\s+(\S+):\s*$", line)
        if m:
            name = m.group(1)
        elif name and "REG:" in line:
            out[name] = line.strip()
            name = None
    return out


def old_name(new, old_names):
    """the instantiation of OLD that NEW's kernel `new` stands for, or None"""
    n = new
    while n not in old_names:
        plain = n.replace("ILb0EEEv", "E", 1)                   # template<bool X = false> on a plain kernel
        if plain in old_names:
            return plain
        shorter = n.replace("Lb0EEEv", "EEv", 1)                # one trailing default argument less
        if shorter == n:
            return None
        n = shorter
    return n


def main(old_lib, new_lib):
    so, sn = sass(old_lib), sass(new_lib)
    ro, rn = res_usage(old_lib), res_usage(new_lib)
    mapped = {}
    for k in sn:
        o = old_name(k, so)
        if o is not None:
            mapped[o] = k
    same = 0
    for o in sorted(so):
        k = mapped.get(o)
        rec = {"old": o, "new": k}
        if k is None:
            rec["result"] = "missing"
        else:
            rec["sass_lines"] = len(so[o])
            rec["sass_same"] = so[o] == sn[k]
            rec["res_usage_same"] = ro.get(o) == rn.get(k)
            rec["res_usage"] = rn.get(k)
            rec["result"] = "same" if rec["sass_same"] and rec["res_usage_same"] else "DIFFERENT"
            same += rec["result"] == "same"
        print(json.dumps(rec))
    new_only = sorted(set(sn) - set(mapped.values()))
    for k in new_only:
        print(json.dumps({"new_only": k, "sass_lines": len(sn[k]), "res_usage": rn.get(k)}))
    print(json.dumps({"old_kernels": len(so), "unchanged": same, "new_kernels": len(new_only)}))
    return 0 if same == len(so) else 1


if __name__ == "__main__":
    sys.exit(main(sys.argv[1], sys.argv[2]))
