// tests/lossy_ref_excerpt.cpp -- the statements of the reference's lossy pre-conditioner whose meaning depends on how the
// compiler treats undefined behaviour, in functions of the same shape, for tests/test_lossy_extremes.py to compile with the
// reference's stock flags (g++ -std=c++14 -O3 -DNDEBUG, no -march) and run next to oracle/oracle.c's restatement:
//   * stdDev (h264.cpp:1993-2036): `sum_diff2 += diff * diff` with int diff, which overflows for |diff| >= 46341;
//   * the bound update of addImageLossyNoCamera (:2367-2376) and of addLoss (:2559-2567): `lowError -= (int)round(...)`,
//     where the double is NaN after an empty background / foreground split, or beyond int range for a large stdFactor.
// Test code only: the product never builds or loads it.
#include <cmath>
#include <cstdlib>

extern "C" {

// stdDev(prev, img, n, img_dl, background): img_dl == nullptr is the un-split form used while fewer than 40 spreads are in
void excerpt_std_dev(const unsigned short* prev, const unsigned short* img, int n, const unsigned short* img_dl,
                     unsigned background, double* out)
{
    if (!img_dl) {
        double sum_diff2 = 0, sum_diff = 0;
        for (int i = 0; i < n; ++i) {
            int diff = std::abs((int)img[i] - (int)prev[i]);
            sum_diff2 += diff * diff;
            sum_diff += diff;
        }
        double res = std::sqrt((sum_diff * sum_diff - sum_diff2)) / n;
        out[0] = out[1] = res;
    } else {
        double sum_diff2 = 0, sum_diff = 0, b_sum_diff2 = 0, b_sum_diff = 0;
        int b_sum = 0, sum = 0;
        for (int i = 0; i < n; ++i) {
            int diff = std::abs((int)img[i] - (int)prev[i]);
            if (img_dl[i] > background) {
                sum_diff2 += diff * diff;
                sum_diff += diff;
                sum++;
            } else {
                b_sum_diff2 += diff * diff;
                b_sum_diff += diff;
                b_sum++;
            }
        }
        out[0] = std::sqrt((b_sum_diff * b_sum_diff - b_sum_diff2)) / b_sum;
        out[1] = std::sqrt((sum_diff * sum_diff - sum_diff2)) / sum;
    }
}

// addImageLossyNoCamera's bound update; errors = {lowValueError, highValueError} in, {lowError, highError} out
void excerpt_bounds_add_image_lossy(const double* stdDevs, const double* mean, double stdFactor, int* errors)
{
    int lowError = errors[0];
    int highError = errors[1];
    highError -= (int)round(std::abs(stdDevs[1] - mean[1]) * stdFactor);
    lowError -= (int)round(std::abs(stdDevs[0] - mean[0]) * stdFactor);
    if (highError < 0) highError = 0;
    if (lowError < highError) lowError = highError;
    errors[0] = lowError;
    errors[1] = highError;
}

// addLoss's: only a spread above its running mean tightens the bound
void excerpt_bounds_add_loss(const double* stdDevs, const double* mean, double stdFactor, int* errors)
{
    int lowError = errors[0];
    int highError = errors[1];
    double diff_high = stdDevs[1] < mean[1] ? 0 : stdDevs[1] - mean[1];
    double diff_low = stdDevs[0] < mean[0] ? 0 : stdDevs[0] - mean[0];
    highError -= (int)round(diff_high * stdFactor);
    lowError -= (int)round(diff_low * stdFactor);
    if (highError < 0) highError = 0;
    if (lowError < highError) lowError = highError;
    errors[0] = lowError;
    errors[1] = highError;
}

// the two constructs on their own, with the operands out of the optimiser's sight
int excerpt_square(volatile int* diff)
{
    int d = *diff;
    return d * d;
}
int excerpt_round_to_int(volatile double* x)
{
    return (int)round(*x);
}
}
