// xsb_x86nan.cuh -- IEEE double arithmetic whose NaN results carry the bits x86-64 gives them: the first NaN
// operand, quieted; an invalid operation on non-NaN operands (Inf - Inf, 0 * Inf) gives the negative default NaN.
// The device's own NaN results differ, and nzval is compared bit for bit with the reference's host arithmetic.
#pragma once
#include "xsb_internal.h"

namespace xsb {

__device__ __forceinline__ double quiet(double x)
{
    return __longlong_as_double(__double_as_longlong(x) | 0x0008000000000000ll);
}

// r = a op b as the device computed it -> the same value with x86-64's NaN bits
__device__ __forceinline__ double x86_nan(double r, double a, double b)
{
    if (r == r)
        return r;
    if (a != a)
        return quiet(a);
    if (b != b)
        return quiet(b);
    return __longlong_as_double((long long)0xfff8000000000000ull);
}

// a + b (OP == kAlgAdd) or a - b (OP == kAlgSub)
template <int OP> __device__ __forceinline__ double apply(double a, double b)
{
    return x86_nan(OP == kAlgSub ? __dsub_rn(a, b) : __dadd_rn(a, b), a, b);
}

__device__ __forceinline__ double mul_x86(double a, double b) { return x86_nan(__dmul_rn(a, b), a, b); }

} // namespace xsb
