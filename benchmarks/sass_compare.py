"""Compare the SASS of two builds of one CUDA object, function by function.

  python benchmarks/sass_compare.py OLD.o NEW.o [--trailing-default "(bool)1"]

Functions are matched by demangled name.  A template that gained trailing parameters with defaults (say
``sh_bwd_flush_kernel<3, 16, true>`` -> ``sh_bwd_flush_kernel<3, 16, true, true>``) is matched through
``--trailing-default``: an old function also matches the new one whose template arguments are the old ones followed
only by that value.  Every matched pair must have the same instructions (addresses, offsets of line info and the
function's own symbol are stripped); the script prints one line per function and exits non-zero on any difference or
any old function without a match.  New functions without an old counterpart are listed as added.
"""
import argparse
import re
import subprocess
import sys
from pathlib import Path

CUDA_BIN = Path("/usr/local/cuda/bin")


def _tool(name):
  p = CUDA_BIN / name
  return str(p) if p.exists() else name


def demangle(names):
  r = subprocess.run([_tool("cu++filt")], input="\n".join(names), stdout=subprocess.PIPE, text=True, check=True)
  return r.stdout.splitlines()


def sass_functions(obj):
  """{mangled name: [instruction text]} of every function in ``obj``."""
  out = subprocess.run([_tool("cuobjdump"), "-sass", str(obj)], stdout=subprocess.PIPE, text=True, check=True).stdout
  funcs, cur = {}, None
  for line in out.splitlines():
    m = re.match(r"\s*Function : (\S+)", line)
    if m:
      cur = m.group(1)
      funcs[cur] = []
      continue
    if cur is None:
      continue
    m = re.match(r"\s*/\*[0-9a-f]{4,}\*/\s+(.*?)\s*;?\s*(/\*.*\*/)?\s*$", line)
    if m and m.group(1):
      funcs[cur].append(m.group(1))
  return funcs


def split_template(name):
  """('gs::f', ['3', '16', 'true']) for 'void gs::f<3, 16, true>(args)'; (name, None) for a non-template."""
  depth, start, end = 0, None, None
  for i, c in enumerate(name):
    if c == "(" and depth == 0:   # the parameter list (casts such as "(int)3" sit inside the template brackets)
      break
    if c == "<":
      start = i if depth == 0 else start
      depth += 1
    elif c == ">":
      depth -= 1
      end = i if depth == 0 else end
  if start is None or end is None:
    return name.split("(", 1)[0], None
  head = name[:end + 1]
  args, depth, cur = [], 0, ""
  for c in head[start + 1:-1]:
    if c == "," and depth == 0:
      args.append(cur.strip())
      cur = ""
      continue
    depth += c == "<"
    depth -= c == ">"
    cur += c
  args.append(cur.strip())
  return head[:start].split(" ")[-1], args


def main():
  ap = argparse.ArgumentParser()
  ap.add_argument("old")
  ap.add_argument("new")
  ap.add_argument("--trailing-default", default="(bool)1")
  args = ap.parse_args()
  old, new = sass_functions(args.old), sass_functions(args.new)
  old_names = dict(zip(old, demangle(list(old))))
  new_names = dict(zip(new, demangle(list(new))))
  new_by_key = {}
  for m, d in new_names.items():
    new_by_key.setdefault(split_template(d)[0], []).append((m, d))

  def strip_self(instrs, mangled):
    return [i.replace(mangled, "<self>") for i in instrs]

  bad, matched = 0, set()
  for m, d in sorted(old_names.items(), key=lambda kv: kv[1]):
    target = m if m in new else None
    if target is None:
      base, targs = split_template(d)
      for m2, d2 in new_by_key.get(base, []):
        b2, a2 = split_template(d2)
        if targs is not None and a2 is not None and a2[:len(targs)] == targs and len(a2) > len(targs) \
            and all(a == args.trailing_default for a in a2[len(targs):]):
          target = m2
          break
    if target is None:
      print(f"MISSING  {d}")
      bad += 1
      continue
    matched.add(target)
    a, b = strip_self(old[m], m), strip_self(new[target], target)
    same = a == b
    bad += not same
    label = d if target == m else f"{d} -> {new_names[target].split('(')[0]}"
    print(f"{'same   ' if same else 'DIFFERS'}  {len(a):5d} -> {len(b):5d} instructions  {label}")
  for m, d in sorted(new_names.items(), key=lambda kv: kv[1]):
    if m not in matched:
      print(f"added    {len(new[m]):5d} instructions  {d}")
  print(f"{len(old)} old functions, {len(matched)} matched, {bad} differing or missing, "
        f"{len(new) - len(matched)} added")
  return 1 if bad else 0


if __name__ == "__main__":
  sys.exit(main())
