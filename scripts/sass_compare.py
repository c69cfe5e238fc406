"""Compare the SASS of every kernel between two sets of `cuobjdump -sass` dumps (one .sass file per source file).

usage: python scripts/sass_compare.py OLD_DIR NEW_DIR [--widened NAME ...]

Each function is hashed over its instruction text without addresses and encoding comments; anonymous-namespace tags,
which hash the source path, are normalised.  A kernel template that gained a defaulted trailing flag (--widened NAME)
keeps its existing instantiations under a new mangled name: "...Lb0E" before the end of the template arguments, and a
trailing kernel parameter of a struct type; those names are mapped back before the comparison."""
import hashlib
import re
import sys
from pathlib import Path


def functions(path: Path) -> dict:
    out, name, body = {}, None, []
    for line in path.read_text().splitlines():
        m = re.match(r"\s*Function : (\S+)", line)
        if m:
            if name:
                out[name] = body
            name, body = re.sub(r"_GLOBAL__N__[0-9a-f]+_\d+_\w+?_cu_[0-9a-f]{8}", "_GLOBAL__N_", m.group(1)), []
            continue
        ins = re.match(r"\s*/\*[0-9a-f]{4,}\*/\s+(.*?);", line)
        if name and ins:
            body.append(ins.group(1).strip())
    if name:
        out[name] = body
    return {k: hashlib.sha256("\n".join(v).encode()).hexdigest()[:16] for k, v in out.items()}


def main(argv):
    old_dir, new_dir = Path(argv[0]), Path(argv[1])
    widened = argv[argv.index("--widened") + 1:] if "--widened" in argv else []

    def back(name: str) -> str:
        if not any(w in name for w in widened):
            return name
        name = name.replace("Lb0EEEv", "EEv", 1) if "Lb0EEEv" in name else name
        return re.sub(r"NS_8BoxMasksE$", "", name)

    old, new = {}, {}
    for f in sorted(old_dir.glob("*.sass")):
        old.update({(f.stem, k): v for k, v in functions(f).items()})
    for f in sorted(new_dir.glob("*.sass")):
        new.update({(f.stem, back(k)): (k, v) for k, v in functions(f).items()})
    same = [k for k in old if k in new and new[k][1] == old[k]]
    diff = [k for k in old if k in new and new[k][1] != old[k]]
    missing = [k for k in old if k not in new]
    added = [new[k][0] for k in new if k not in old]
    print(f"existing kernels: {len(old)}; identical: {len(same)}; different: {len(diff)}; missing: {len(missing)}")
    print(f"new kernels: {len(added)}")
    for k in diff:
        print(f"different  {k[0]}  {k[1]}")
    for k in missing:
        print(f"missing    {k[0]}  {k[1]}")
    for k in sorted(new):
        if k not in old:
            print(f"new        {new[k][1]}  {k[0]}.cu  {new[k][0]}")
    return 1 if diff or missing else 0


if __name__ == "__main__":
    sys.exit(main(sys.argv[1:]))
