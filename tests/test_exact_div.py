"""CPU: the divide-free branch mean of the tensor-core epilogues (tc::div_exact in csrc/tc_ptx.cuh) equals the IEEE
quotient x / d bit for bit for every one of the 2^32 float inputs, subnormals, signed zeros and infinities included, for
each divisor the host accepts (tc_div_exact in csrc/conv_tc.cuh; d = 1 skips the division).  The same arithmetic is
compiled with the host compiler: no FMA contraction, libm fmaf, round-to-nearest and no flush to zero."""
import shutil
import subprocess


SRC = r"""
#include <math.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

static float bits(uint32_t u) { float f; memcpy(&f, &u, 4); return f; }
static uint32_t ubits(float f) { uint32_t u; memcpy(&u, &f, 4); return u; }

int main(int argc, char** argv) {
  const float d = (float)atof(argv[1]);
  volatile float dv = d;
  const float r = 1.0f / dv;
  uint64_t bad = 0;
  for (uint64_t i = 0; i <= 0xffffffffull; ++i) {
    const float v = bits((uint32_t)i);
    const float want = v / d;
    const float q0 = v * r;                         /* tc::div_exact */
    const float e = fmaf(-q0, d, v);
    const float got = fabsf(e) > 0.f ? fmaf(e, r, q0) : q0;
    if (ubits(got) != ubits(want) && !(isnan(got) && isnan(want))) {
      if (bad < 5) printf("x=%08x: %08x != %08x\n", (unsigned)i, ubits(got), ubits(want));
      ++bad;
    }
  }
  printf("d=%g: %llu mismatches\n", d, (unsigned long long)bad);
  return bad != 0;
}
"""


def test_div_exact_all_inputs(tmp_path):
    cc = shutil.which("cc") or shutil.which("gcc")
    assert cc, "a host C compiler is needed (the CUDA build needs one too)"
    src, exe = tmp_path / "div_exact.c", tmp_path / "div_exact"
    src.write_text(SRC)
    subprocess.run([cc, "-O2", "-ffp-contract=off", "-fno-fast-math", "-o", str(exe), str(src), "-lm"], check=True)
    procs = [subprocess.Popen([str(exe), d], stdout=subprocess.PIPE, text=True) for d in ("2", "3", "4")]
    outs = [(p.communicate()[0], p.returncode) for p in procs]
    for out, rc in outs:
        print(out.strip())
        assert rc == 0, out
