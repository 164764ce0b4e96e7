// tests/cpp/alpha_probe.cpp — a shared library exposing ScratchImage::IsAlphaAllOpaque and ComputeMSE to ctypes.  Built against the
// C++ mirror (DirectXTexB200.h, linked with libdxtex_b200.so) and, with -DPROBE_REFERENCE, against the reference's own DirectXTex.h
// (through oracle/compat, linked with the reference build oracle/_ref/libdxtex_ref.so) to record the reference's answers.
#include <cstdint>
#include <cstring>
#ifdef PROBE_REFERENCE
#include "DirectXTex.h"
#else
#include "DirectXTexB200.h"
#endif
using namespace DirectX;

extern "C" {

// the member's answer for a 2D texture packed in ScratchImage::Initialize2D(fmt, w, h, arraySize, mipLevels) order
__attribute__((visibility("default")))
int32_t probe_is_alpha_all_opaque(const uint8_t* pixels, size_t pixelBytes, uint32_t fmt, size_t w, size_t h, size_t arraySize,
                                  size_t mipLevels, int32_t* opaque)
{
    ScratchImage img;
    HRESULT hr = img.Initialize2D(static_cast<DXGI_FORMAT>(fmt), w, h, arraySize, mipLevels);
    if (FAILED(hr)) return hr;
    if (img.GetPixelsSize() != pixelBytes) return E_INVALIDARG;
    memcpy(img.GetPixels(), pixels, pixelBytes);
    *opaque = img.IsAlphaAllOpaque() ? 1 : 0;
    return S_OK;
}

// ComputeMSE of two tightly packed single images; out = { mse, mseV[0..3] }
__attribute__((visibility("default")))
int32_t probe_compute_mse(const uint8_t* a, uint32_t fmtA, const uint8_t* b, uint32_t fmtB, size_t w, size_t h, uint32_t flags, float* out)
{
    Image ia = {}, ib = {};
    ia.width = ib.width = w; ia.height = ib.height = h;
    ia.format = static_cast<DXGI_FORMAT>(fmtA); ib.format = static_cast<DXGI_FORMAT>(fmtB);
    ComputePitch(ia.format, w, h, ia.rowPitch, ia.slicePitch);
    ComputePitch(ib.format, w, h, ib.rowPitch, ib.slicePitch);
    ia.pixels = const_cast<uint8_t*>(a); ib.pixels = const_cast<uint8_t*>(b);
    return ComputeMSE(ia, ib, out[0], out + 1, static_cast<CMSE_FLAGS>(flags));
}

}
