"""Diagnostics (not a test): compare the SASS of the learner's tensor-core kernels between a git commit and the working
tree.  Both sides are compiled for sm_100a with the Makefile's flags; kernels are paired by role and template
arguments (chain_fwd_tf32x3_kernel<1, true> <-> chain_fwd_kernel<1, true, Tf32x3>), and their instruction sequences
compared without addresses, encodings, branch targets and symbol names.  Registers and spill bytes from ptxas -v are
printed beside each pair.

  python tests/sass_compare.py [commit (default HEAD)] [file.cu ...]

Exit status 1 when a kernel differs or has no partner."""
import os
import re
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = "model-based-rl_b200/csrc"
FILES = ("mz_learner_tc.cu", "mz_learner_tf32.cu", "mz_fcnet_tf32.cu")
FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17", "-lineinfo", "-DMZ_BUILDING"]
CONTROL = re.compile(r"\b(BRA|BRX|BSSY|BSYNC|CALL|JMP|JMX|RET|BREAK|WARPSYNC)\b")


def tool(name):
  nvcc = os.environ.get("NVCC") or "/usr/local/cuda/bin/nvcc"
  return os.path.join(os.path.dirname(nvcc), name)


def compile_tree(tree, src, out):
  """(kernel -> normalised instructions, kernel -> (registers, spill bytes)) of one translation unit."""
  obj = os.path.join(out, src + ".o")
  err = subprocess.run([tool("nvcc"), *FLAGS, "-I" + os.path.join(tree, "include"), "-I" + os.path.join(tree, CSRC),
                        "-Xptxas", "-v", "-c", os.path.join(tree, CSRC, src), "-o", obj],
                       capture_output=True, text=True, check=True).stderr
  res, cur = {}, None
  for line in err.splitlines():
    m = re.search(r"Compiling entry function '(\S+)'", line)
    if m:
      cur = m.group(1)
    m = re.search(r"(\d+) bytes spill stores, (\d+) bytes spill loads", line)
    if m and cur:
      res.setdefault(cur, [0, 0])[1] = int(m.group(1)) + int(m.group(2))
    m = re.search(r"Used (\d+) registers", line)
    if m and cur:
      res.setdefault(cur, [0, 0])[0] = int(m.group(1))
  sass = subprocess.run([tool("cuobjdump"), "-sass", obj], capture_output=True, text=True, check=True).stdout
  code, cur = {}, None
  for line in sass.splitlines():
    m = re.search(r"Function : (\S+)", line)
    if m:
      cur = m.group(1)
      code[cur] = []
      continue
    m = re.match(r"\s*/\*[0-9a-f]{4,}\*/\s*(.*?)\s*;", line)
    if m and cur:
      ins = m.group(1)
      if CONTROL.search(ins):
        ins = re.sub(r"0x[0-9a-f]+", "<target>", ins)
      code[cur].append(ins)
  return code, res


def demangle(names):
  out = subprocess.run([tool("cu++filt")], input="\n".join(names), capture_output=True, text=True, check=True).stdout
  return dict(zip(names, out.splitlines()))


def key(src, pretty):
  """(file, role, template arguments without the format policy); the parent's tf32x3 heads_bwd had no TILES."""
  pretty = re.sub(r"^void ", "", pretty.replace("<unnamed>::", ""))
  m = re.match(r"([A-Za-z0-9_]+)(?:<(.*)>)?\(", pretty)
  args = [re.sub(r"^\((int|bool)\)", "", a.strip()) for a in (m.group(2) or "").split(",") if a.strip()]
  role, args = m.group(1), [{"true": "1", "false": "0"}.get(a, a) for a in args]
  tf32x3 = role.endswith("_tf32x3_kernel")
  role = role.replace("_tf32x3_kernel", "_kernel")
  args = [a for a in args if a not in ("Bf16", "Tf32x3")]
  if tf32x3 and role == "heads_bwd_kernel":
    args = ["1"] + args
  return src, role + "<" + ", ".join(args) + ">"


def main():
  commit = sys.argv[1] if len(sys.argv) > 1 else "HEAD"
  files = sys.argv[2:] or FILES
  bad = 0
  with tempfile.TemporaryDirectory() as d:
    base = os.path.join(d, "base")
    os.makedirs(base)
    subprocess.run(f"git -C {ROOT} archive {commit} include {CSRC} | tar -x -C {base}", shell=True, check=True)
    for src in files:
      sides = []
      for tree in (base, ROOT):
        out = tempfile.mkdtemp(dir=d)
        code, res = compile_tree(tree, src, out)
        names = demangle(sorted(code))
        sides.append({key(src, names[k]): (names[k], code[k], res.get(k, [0, 0])) for k in code})
      print(f"== {src}: {commit} {len(sides[0])} kernels, working tree {len(sides[1])} kernels")
      for k in sorted(set(sides[0]) | set(sides[1])):
        if k not in sides[0] or k not in sides[1]:
          bad += 1
          print(f"  UNPAIRED {k[1]}: only in {'the working tree' if k in sides[1] else commit}")
          continue
        (n0, c0, r0), (n1, c1, r1) = sides[0][k], sides[1][k]
        same = c0 == c1
        bad += not same
        print(f"  {'same' if same else 'DIFFERENT':9s} {len(c0):5d} / {len(c1):5d} instructions  registers {r0[0]} / {r1[0]}"
              f"  spill bytes {r0[1]} / {r1[1]}  {n0}  <->  {n1}")
        if not same:
          for i, (a, b) in enumerate(zip(c0, c1)):
            if a != b:
              print(f"      first difference at instruction {i}: {a!r} / {b!r}")
              break
  print("all kernels match" if not bad else f"{bad} kernel(s) differ or are unpaired")
  return 1 if bad else 0


if __name__ == "__main__":
  sys.exit(main())
