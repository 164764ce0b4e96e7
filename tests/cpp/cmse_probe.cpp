// tests/cpp/cmse_probe.cpp — prints the CMSE_FLAGS enumerators (DirectXTex.h:1022-1038); built against the C++ mirror, and with
// -DPROBE_REFERENCE against the reference's own header (tests/test_cpu_analysis.py compares the two)
#include <cstdio>
#ifdef PROBE_REFERENCE
#include "DirectXTex.h"
#else
#include "DirectXTexB200.h"
#endif
using namespace DirectX;

int main()
{
#define P(e) std::printf("%s %u\n", #e, static_cast<unsigned>(e))
    P(CMSE_DEFAULT); P(CMSE_IMAGE1_SRGB); P(CMSE_IMAGE2_SRGB); P(CMSE_IGNORE_RED); P(CMSE_IGNORE_GREEN); P(CMSE_IGNORE_BLUE);
    P(CMSE_IGNORE_ALPHA); P(CMSE_IMAGE1_X2_BIAS); P(CMSE_IMAGE2_X2_BIAS);
    return 0;
}
