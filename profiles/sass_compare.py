"""Compare two builds of librenv_b200.so kernel by kernel (no GPU needed):

    python profiles/sass_compare.py OLD_DIR NEW_DIR > record.txt

Each directory is a random_envs_b200 package directory holding librenv_b200.so and the build's
librenv_b200.ptxas.log.  A kernel of OLD is SAME when its SASS (addresses ignored) and its ptxas registers, stack frame
and shared memory are identical in NEW; kernels only in NEW are listed with their statistics.
"""
import os
import re
import sys

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import sass_stats  # noqa: E402


def ptxas(path):
    out = {}
    for b in re.split(r"ptxas info\s+: Compiling entry function '", open(path).read())[1:]:
        name = b.split("'")[0]
        get = lambda pat: (re.search(pat, b).group(1) if re.search(pat, b) else "?")
        spills = re.search(r"(\d+) bytes spill stores, (\d+) bytes spill loads", b)
        out[name] = dict(regs=get(r"Used (\d+) registers"), stack=get(r"(\d+) bytes stack frame"),
                         smem=get(r"(\d+) bytes smem"), spills=(int(spills.group(1)), int(spills.group(2))) if spills else None)
    return out


def main():
    old_dir, new_dir = sys.argv[1], sys.argv[2]
    old = sass_stats.functions(os.path.join(old_dir, "librenv_b200.so"))
    new = sass_stats.functions(os.path.join(new_dir, "librenv_b200.so"))
    p_old = ptxas(os.path.join(old_dir, "librenv_b200.ptxas.log"))
    p_new = ptxas(os.path.join(new_dir, "librenv_b200.ptxas.log"))
    code = lambda rows: [(op, rest) for _, op, rest in rows]
    meta = lambda p, k: {f: p.get(k, {}).get(f) for f in ("regs", "stack", "smem")}
    lines, same, diff, missing = [], 0, 0, 0
    for name in new:
        if name not in old:
            m = p_new.get(name, {})
            lines.append("NEW %s instr=%d regs=%s stack=%s smem=%s spills=%s" % (
                name, len(new[name]), m.get("regs"), m.get("stack"), m.get("smem"), m.get("spills")))
    for name in old:
        if name not in new:
            missing += 1
            lines.append("MISSING %s" % name)
            continue
        ok = code(old[name]) == code(new[name]) and meta(p_old, name) == meta(p_new, name)
        same += ok
        diff += not ok
        m = meta(p_new, name)
        lines.append("%s %s instr=%d regs=%s stack=%s smem=%s" % ("SAME" if ok else "DIFF", name, len(new[name]),
                                                                 m["regs"], m["stack"], m["smem"]))
    print("librenv_b200.so of this change against a build of its parent commit, per kernel: SASS (addresses ignored, "
          "profiles/sass_stats.py) and the ptxas registers / stack / shared memory")
    print("Pre-existing kernels: %d, SASS + registers + shared memory + stack identical: %d, different: %d, missing: %d"
          % (len(old), same, diff, missing))
    print("\n".join(lines))


if __name__ == "__main__":
    main()
