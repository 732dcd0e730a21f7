// Exhaustive host check of hypot_glibc_int (stair_step_detector_b200/csrc/ssd_device.cuh, the denominator of the device's line fits)
// against the host's libm hypot, which the reference calls: every integer pair (a, b) with |a| <= 5109 and |b| <= 9349, the
// largest line coefficients of the largest frame ssd_gpu_create accepts (a: row difference, b: column difference). Host code only.
//   nvcc -O2 -std=c++17 -Xcompiler -ffp-contract=off -o hypot_glibc_check tools/hypot_glibc_check.cu && ./hypot_glibc_check
// Prints the number of pairs compared, of mismatches (must be 0) and of pairs where libm is not the correctly rounded square root.
#include <cmath>
#include <cstdio>
#include "../stair_step_detector_b200/csrc/ssd_device.cuh"

int main()
{
  const int AMAX = 5109, BMAX = 9349;
  long long n = 0, bad = 0, not_cr = 0;
  for(int a = -AMAX; a <= AMAX; a++)
    for(int b = -BMAX; b <= BMAX; b++)
    {
      const double l = hypot((double)a, (double)b), g = hypot_glibc_int(a, b);
      n++;
      if(l != g && bad++ < 10)
        std::printf("mismatch a=%d b=%d libm=%a device=%a\n", a, b, l, g);
      not_cr += l != std::sqrt((double)a * a + (double)b * b);
    }
  std::printf("pairs %lld mismatches %lld libm_not_correctly_rounded %lld\n", n, bad, not_cr);
  return bad != 0;
}
