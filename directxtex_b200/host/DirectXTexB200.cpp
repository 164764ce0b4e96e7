// DirectXTexB200.cpp — implementation of the C++ mirror (DirectXTexB200.h): validation and destination
// allocation as the reference's entry points do them, compute through the C ABI (include/dxtex_b200.h).
// Reference behaviour restated (not copied): Compress/CompressEx DirectXTexCompress.cpp:632-845, Convert/ConvertEx
// DirectXTexConvert.cpp:5091-5404, GenerateMipMaps DirectXTexMipmaps.cpp:2828-3247 + Setup2DMips :851-904,
// ScratchImage DirectXTexImage.cpp:300-455, TexMetadata::ComputeIndex DirectXTexUtil.cpp:1695-1741.
#include "DirectXTexB200.h"
#include "../../include/dxtex_b200.h"

#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <new>
#include <vector>
#include <string>

namespace
{
    inline dxb200_image to_c(const DirectX::Image& im)
    {
        dxb200_image c; c.width = im.width; c.height = im.height; c.format = static_cast<uint32_t>(im.format);
        c.rowPitch = im.rowPitch; c.slicePitch = im.slicePitch; c.pixels = im.pixels;
        return c;
    }
    inline bool implemented_pixel_format(DXGI_FORMAT f)
    {
        size_t r = 0, s = 0;
        return dxb200_compute_pitch(static_cast<uint32_t>(f), 1, 1, &r, &s) == 0;
    }
}

namespace
{

// ---- format utilities (DirectXTex.h:72-99, 144-154; DirectXTexUtil.cpp:760-960, 1186-1690) -----------------------------------------
// The reference answers these from one switch statement per question.  Here every answer is derived from the format's NAME: a DXGI
// name is a list of channel groups (a letter and a bit count each: R8G8B8A8, D24 + S8, R9G9B9E5, X8X24 ...) followed by a type
// (UNORM, FLOAT, TYPELESS, ... SRGB), so bits per pixel is the sum of the bit counts, bits per colour their maximum, "has alpha" an A
// channel, BGR a leading B channel, and the Make* conversions are look-ups of the sibling name.  The video / planar / palettized /
// block-compressed formats, whose names are not channel lists, have one small table.  tests/test_cpu_abi.py compares all of it, for
// every value 0..200, with the reference's own functions.
struct FormatName { uint32_t value; const char* name; };
const FormatName kFormatNames[] = {
#define DXB_X(name, value) { value, #name },
    DXB_DXGI_FORMATS(DXB_X)
#undef DXB_X
    // extension values the reference classifies although they are not DXGI_FORMAT enumerators (XBOX_DXGI_FORMAT_*, DirectXTexP.h:188-204;
    // 189 / 190 take the Xbox meaning there, which shadows the sampler-feedback names of the public enum: listed first = found first)
};
const FormatName kExtensionNames[] = {
    { 116, "R10G10B10_7E3_A2_FLOAT" }, { 117, "R10G10B10_6E4_A2_FLOAT" }, { 118, "D16_UNORM_S8_UINT" }, { 119, "R16_UNORM_X8_TYPELESS" },
    { 120, "X16_TYPELESS_G8_UINT" }, { 189, "R10G10B10_SNORM_A2_UNORM" }, { 190, "R4G4_UNORM" },
};
const char* format_name(DXGI_FORMAT f)
{
    for (const FormatName& e : kExtensionNames) if (e.value == static_cast<uint32_t>(f)) return e.name;
    for (const FormatName& e : kFormatNames) if (e.value == static_cast<uint32_t>(f)) return e.name;
    return nullptr;
}
DXGI_FORMAT format_by_name(const std::string& n, DXGI_FORMAT fallback)
{
    for (const FormatName& e : kFormatNames) if (n == e.name) return static_cast<DXGI_FORMAT>(e.value);
    return fallback;
}
struct FormatClass
{
    bool known = false, regular = false;            // regular: the name is a channel list
    bool typeless = false, partialTypeless = false, srgb = false, depth = false, stencilPlane = false, xboxPlanar = false, alpha = false, bgr = false;
    size_t bits = 0, maxBits = 0;
    int bc = 0;                                     // 1..7 for BCn
    std::string family;                             // name without its trailing type tokens ("R8G8B8A8", "BC6H")
};
bool is_type_token(const std::string& t)
{
    return t == "TYPELESS" || t == "UNORM" || t == "SNORM" || t == "UINT" || t == "SINT" || t == "FLOAT" || t == "SRGB" || t == "UF16" || t == "SF16" ||
           t == "SHAREDEXP";
}
// "R32G8X24" -> channels; false when the token is not (letter, digits)+
bool parse_group(const std::string& t, FormatClass& c, bool first)
{
    size_t i = 0, sum = 0, mx = 0, posB = 99, posR = 99, idx = 0; bool a = false, d = false, any = false;
    while (i < t.size())
    {
        const char ch = t[i];
        if (!(ch == 'R' || ch == 'G' || ch == 'B' || ch == 'A' || ch == 'X' || ch == 'D' || ch == 'S' || ch == 'E')) return false;
        size_t k = i + 1, v = 0;
        while (k < t.size() && t[k] >= '0' && t[k] <= '9') { v = v * 10 + size_t(t[k] - '0'); ++k; }
        if (k == i + 1) return false;
        if (ch == 'A') a = true;
        if (ch == 'D') d = true;
        if (ch == 'B' && posB == 99) posB = idx;
        if (ch == 'R' && posR == 99) posR = idx;
        mx = std::max(mx, v);                       // padding (X) planes count: X32_TYPELESS_G8X24_UINT answers 32
        sum += v; i = k; any = true; ++idx;
    }
    if (!any) return false;
    c.bits += sum; c.maxBits = std::max(c.maxBits, mx); c.alpha |= a; c.depth |= d;
    if (first) c.bgr = (posB < posR && posR != 99);   // blue stored before red: B8G8R8A8, B5G6R5, A4B4G4R4
    return true;
}
FormatClass classify_name(DXGI_FORMAT f);
// every value 0..255 is classified once (the names are parsed on first use); anything else is unknown
const FormatClass& classify(DXGI_FORMAT f)
{
    static const std::vector<FormatClass> table = []() { std::vector<FormatClass> t(256); for (uint32_t v = 0; v < 256; ++v) t[v] = classify_name(static_cast<DXGI_FORMAT>(v)); return t; }();
    static const FormatClass unknown;
    const uint32_t v = static_cast<uint32_t>(f);
    return (v < 256u) ? table[v] : unknown;
}
FormatClass classify_name(DXGI_FORMAT f)
{
    FormatClass c;
    const char* nm = format_name(f);
    if (!nm || f == DXGI_FORMAT_UNKNOWN) return c;
    c.known = true;
    std::vector<std::string> tok;
    { std::string cur; for (const char* p = nm;; ++p) { if (*p == '_' || *p == 0) { tok.push_back(cur); cur.clear(); if (!*p) break; } else cur += *p; } }
    if (tok[0].size() >= 3 && tok[0][0] == 'B' && tok[0][1] == 'C' && tok[0][2] >= '1' && tok[0][2] <= '7')
    {
        c.bc = tok[0][2] - '0';
        c.bits = (c.bc == 1 || c.bc == 4) ? 4 : 8;
        c.maxBits = (c.bc == 6) ? 16 : (c.bc == 7) ? 7 : (c.bc <= 3) ? 6 : 8;          // 5:6:5 end points; mode-dependent 4..8 for BC7
        c.alpha = (c.bc == 1 || c.bc == 2 || c.bc == 3 || c.bc == 7);
    }
    else
    {
        bool all = true, first = true; size_t groups = 0, types = 0;
        FormatClass t = c;
        for (const std::string& s : tok)
        {
            if (is_type_token(s)) { ++types; continue; }
            if (s == "XR" || s == "BIAS" || s == "7E3" || s == "6E4") continue;      // R10G10B10_XR_BIAS_A2_UNORM, the Xbox 7e3 / 6e4 floats
            if (!parse_group(s, t, first)) { all = false; break; }
            first = false; ++groups;
        }
        if (all && groups > 0) { c = t; c.regular = true; }
        (void)types;
    }
    size_t ntypes = 0;
    for (const std::string& s : tok) if (is_type_token(s)) { ++ntypes; if (s == "TYPELESS") c.typeless = true; if (s == "SRGB") c.srgb = true; }
    c.partialTypeless = c.typeless && ntypes > 1;
    // a stencil plane next to a 24 / 32-bit depth plane: the D3D12 planar depth formats (R32G8X24, R24G8 and their views)
    { const std::string n(nm); c.stencilPlane = n.find("G8X24") != std::string::npos || n.find("S8X24") != std::string::npos || n.find("X8X24") != std::string::npos ||
                                               n.find("R24G8") != std::string::npos || n.find("D24_UNORM_S8") != std::string::npos || n.find("R24_UNORM_X8") != std::string::npos ||
                                               n.find("X24_TYPELESS_G8") != std::string::npos;
      c.xboxPlanar = n.find("D16_UNORM_S8") != std::string::npos || n.find("R16_UNORM_X8") != std::string::npos || n.find("X16_TYPELESS_G8") != std::string::npos;
      c.stencilPlane |= c.xboxPlanar;
      if (n == "R9G9B9E5_SHAREDEXP") c.maxBits = 14; }        // 9 mantissa + 5 shared exponent bits
    // family = the name up to (not including) its trailing run of type tokens
    size_t last = tok.size();
    while (last > 0 && is_type_token(tok[last - 1])) --last;
    for (size_t k = 0; k < last; ++k) c.family += (k ? "_" : "") + tok[k];
    return c;
}
// formats whose names are not channel lists: { bits per pixel, bits per colour (0: palettized), alpha, video, planar, palettized, packed }
struct OddFormat { DXGI_FORMAT f; uint8_t bpp, bpc; bool alpha, video, planar, pal, packed; };
const OddFormat kOdd[] = {
    { DXGI_FORMAT_AYUV, 32, 8, true, true, false, false, false },   { DXGI_FORMAT_Y410, 32, 10, true, true, false, false, false },
    { DXGI_FORMAT_Y416, 64, 16, true, true, false, false, false },  { DXGI_FORMAT_NV12, 12, 8, false, true, true, false, false },
    { DXGI_FORMAT_P010, 24, 10, false, true, true, false, false },  { DXGI_FORMAT_P016, 24, 16, false, true, true, false, false },
    { DXGI_FORMAT_420_OPAQUE, 12, 8, false, true, true, false, false }, { DXGI_FORMAT_YUY2, 32, 8, false, true, false, false, true },
    { DXGI_FORMAT_Y210, 64, 10, false, true, false, false, true },  { DXGI_FORMAT_Y216, 64, 16, false, true, false, false, true },
    { DXGI_FORMAT_NV11, 12, 8, false, true, true, false, false },   { DXGI_FORMAT_AI44, 8, 0, true, true, false, true, false },
    { DXGI_FORMAT_IA44, 8, 0, true, true, false, true, false },     { DXGI_FORMAT_P8, 8, 0, false, true, false, true, false },
    { DXGI_FORMAT_A8P8, 16, 0, true, true, false, true, false },    { DXGI_FORMAT_P208, 16, 8, false, true, true, false, false },
    { DXGI_FORMAT_V208, 16, 8, false, true, true, false, false },   { DXGI_FORMAT_V408, 24, 8, false, true, true, false, false },
};
const OddFormat* odd(DXGI_FORMAT f) { for (const OddFormat& o : kOdd) if (o.f == f) return &o; return nullptr; }
}   // namespace

namespace DirectX
{

bool IsValid(DXGI_FORMAT fmt) noexcept { const uint32_t v = static_cast<uint32_t>(fmt); return v >= 1u && v <= 191u; }
bool IsCompressed(DXGI_FORMAT fmt) noexcept { return classify(fmt).bc != 0; }
bool IsPacked(DXGI_FORMAT fmt) noexcept
{
    if (fmt == DXGI_FORMAT_R8G8_B8G8_UNORM || fmt == DXGI_FORMAT_G8R8_G8B8_UNORM) return true;
    const OddFormat* o = odd(fmt); return o && o->packed;
}
bool IsVideo(DXGI_FORMAT fmt) noexcept { const OddFormat* o = odd(fmt); return o && o->video; }
bool IsPlanar(DXGI_FORMAT fmt, bool isd3d12) noexcept
{
    const OddFormat* o = odd(fmt);
    if (o) return o->planar;
    const FormatClass& c = classify(fmt);
    return c.xboxPlanar || (isd3d12 && c.stencilPlane);
}
bool IsPalettized(DXGI_FORMAT fmt) noexcept { const OddFormat* o = odd(fmt); return o && o->pal; }
bool IsDepthStencil(DXGI_FORMAT fmt) noexcept { const FormatClass& c = classify(fmt); return c.regular && (c.depth || c.stencilPlane); }
bool IsSRGB(DXGI_FORMAT fmt) noexcept { return classify(fmt).srgb; }
bool IsBGR(DXGI_FORMAT fmt) noexcept { const FormatClass& c = classify(fmt); return c.regular && c.bgr; }
bool IsTypeless(DXGI_FORMAT fmt, bool partialTypeless) noexcept
{
    const FormatClass& c = classify(fmt);
    if (!c.typeless) return false;
    return c.partialTypeless ? partialTypeless : true;
}
bool HasAlpha(DXGI_FORMAT fmt) noexcept
{
    const OddFormat* o = odd(fmt);
    if (o) return o->alpha;
    return classify(fmt).alpha;
}
size_t BitsPerPixel(DXGI_FORMAT fmt) noexcept
{
    const OddFormat* o = odd(fmt);
    if (o) return o->bpp;
    return classify(fmt).bits;
}
size_t BitsPerColor(DXGI_FORMAT fmt) noexcept
{
    const OddFormat* o = odd(fmt);
    if (o) return o->bpc;
    return classify(fmt).maxBits;
}
FORMAT_TYPE FormatDataType(DXGI_FORMAT fmt) noexcept
{
    // any TYPELESS part makes the format typeless; otherwise the first type token of the name decides (D24_UNORM_S8_UINT is UNORM,
    // BC6H_UF16 / SHAREDEXP are FLOAT); the non-planar YUV formats count as UNORM, the other video formats and the Xbox depth planes as typeless
    const char* nm = format_name(fmt);
    if (!nm) return FORMAT_TYPE_TYPELESS;
    const std::string n(nm);
    if (n.find("TYPELESS") != std::string::npos || classify(fmt).xboxPlanar) return FORMAT_TYPE_TYPELESS;
    if (const OddFormat* o = odd(fmt)) return (!o->planar && !o->pal) ? FORMAT_TYPE_UNORM : FORMAT_TYPE_TYPELESS;
    size_t best = std::string::npos; FORMAT_TYPE t = FORMAT_TYPE_TYPELESS;
    const struct { const char* tok; FORMAT_TYPE ty; } types[] = {
        { "_FLOAT", FORMAT_TYPE_FLOAT }, { "_UF16", FORMAT_TYPE_FLOAT }, { "_SF16", FORMAT_TYPE_FLOAT }, { "_SHAREDEXP", FORMAT_TYPE_FLOAT },
        { "_UNORM", FORMAT_TYPE_UNORM }, { "_SNORM", FORMAT_TYPE_SNORM }, { "_UINT", FORMAT_TYPE_UINT }, { "_SINT", FORMAT_TYPE_SINT }, { "_TYPELESS", FORMAT_TYPE_TYPELESS } };
    for (const auto& e : types)
    {
        const size_t p = n.find(e.tok);
        if (p != std::string::npos && p < best) { best = p; t = e.ty; }
    }
    return t;
}
size_t ComputeScanlines(DXGI_FORMAT fmt, size_t height) noexcept
{
    if (fmt == DXGI_FORMAT_UNKNOWN) return 0;
    if (IsCompressed(fmt)) return std::max<size_t>(1, (height + 3) / 4);
    if (classify(fmt).xboxPlanar) return height + ((height + 1) >> 1);                        // 16-bit depth plane + half-height stencil rows
    switch (fmt)
    {
    case DXGI_FORMAT_NV11: case DXGI_FORMAT_P208: return height * 2;                          // 4:1:1 / 4:2:2 planar: a full-height chroma plane
    case DXGI_FORMAT_V208: return height + (((height + 1) >> 1) * 2);                         // two half-height chroma planes
    case DXGI_FORMAT_V408: return height + ((height >> 1) * 4);
    case DXGI_FORMAT_NV12: case DXGI_FORMAT_P010: case DXGI_FORMAT_P016: case DXGI_FORMAT_420_OPAQUE: return height + ((height + 1) >> 1);   // 4:2:0
    default: return height;
    }
}
DXGI_FORMAT MakeSRGB(DXGI_FORMAT fmt) noexcept
{
    const char* n = format_name(fmt);
    return n ? format_by_name(std::string(n) + "_SRGB", fmt) : fmt;
}
DXGI_FORMAT MakeLinear(DXGI_FORMAT fmt) noexcept
{
    const char* n = format_name(fmt);
    if (!n) return fmt;
    const std::string s(n);
    return (s.size() > 5 && s.compare(s.size() - 5, 5, "_SRGB") == 0) ? format_by_name(s.substr(0, s.size() - 5), fmt) : fmt;
}
DXGI_FORMAT MakeTypeless(DXGI_FORMAT fmt) noexcept
{
    const FormatClass& c = classify(fmt);
    if (!c.known || c.typeless || c.family.empty()) return fmt;
    const uint32_t v = static_cast<uint32_t>(fmt);
    if (v == 116u || v == 117u || v == 189u) return DXGI_FORMAT_R10G10B10A2_TYPELESS;        // the Xbox 10:10:10:2 variants
    if (v == 190u) return DXGI_FORMAT_R8_TYPELESS;                                            // R4G4
    if (c.depth) return (c.family == "D32") ? DXGI_FORMAT_R32_TYPELESS : (c.family == "D16") ? DXGI_FORMAT_R16_TYPELESS : fmt;
    return format_by_name(c.family + "_TYPELESS", fmt);
}
DXGI_FORMAT MakeTypelessUNORM(DXGI_FORMAT fmt) noexcept
{
    const FormatClass& c = classify(fmt);
    if (!c.known || !c.typeless || c.partialTypeless) return fmt;
    return format_by_name(c.family + "_UNORM", fmt);
}
DXGI_FORMAT MakeTypelessFLOAT(DXGI_FORMAT fmt) noexcept
{
    const FormatClass& c = classify(fmt);
    if (!c.known || !c.typeless || c.partialTypeless) return fmt;
    return format_by_name(c.family + "_FLOAT", fmt);
}

// DirectXTexUtil.cpp:961-1183 for EVERY format and every CP_FLAGS rule.  Three layouts cover all of them:
//   blocks        4x4 texels in 8 or 16 bytes (BAD_DXTN_TAILS: whole blocks only, at least one byte)
//   pixel groups  the packed and planar video formats: a row is ceil(width / g) groups of b bytes, a slice is ComputeScanlines rows
//                 (the planar formats' chroma planes are the extra rows); 4:2:0 needs an even height
//   pixels        everything else: ceil(width * bpp / A) units of A bits, A from the alignment flag (8 without one); the 24 / 16 / 8 BPP
//                 flags override the format's bits per pixel
// With no flags the result equals dxb200_compute_pitch for the formats the backend implements (tests/test_cpu_capi.py).
HRESULT ComputePitch(DXGI_FORMAT fmt, size_t width, size_t height, size_t& rowPitch, size_t& slicePitch, CP_FLAGS flags) noexcept
{
    if (fmt == DXGI_FORMAT_UNKNOWN) return E_INVALIDARG;
    const FormatClass& c = classify(fmt);
    uint64_t pitch = 0, slice = 0;
    struct Group { DXGI_FORMAT f; uint32_t px, bytes; bool evenHeight; };
    static const Group groups[] = {
        { DXGI_FORMAT_R8G8_B8G8_UNORM, 2, 4, false }, { DXGI_FORMAT_G8R8_G8B8_UNORM, 2, 4, false }, { DXGI_FORMAT_YUY2, 2, 4, false },
        { DXGI_FORMAT_Y210, 2, 8, false }, { DXGI_FORMAT_Y216, 2, 8, false },
        { DXGI_FORMAT_NV12, 2, 2, true }, { DXGI_FORMAT_420_OPAQUE, 2, 2, true }, { DXGI_FORMAT_P010, 2, 4, true }, { DXGI_FORMAT_P016, 2, 4, true },
        { static_cast<DXGI_FORMAT>(118), 2, 4, false }, { static_cast<DXGI_FORMAT>(119), 2, 4, false }, { static_cast<DXGI_FORMAT>(120), 2, 4, false },   // Xbox D16 + S8 planes
        { DXGI_FORMAT_NV11, 4, 4, false }, { DXGI_FORMAT_P208, 2, 2, false }, { DXGI_FORMAT_V208, 1, 1, true }, { DXGI_FORMAT_V408, 1, 1, false },
    };
    const Group* g = nullptr;
    for (const Group& e : groups) if (e.f == fmt) g = &e;
    if (c.bc)
    {
        const uint64_t bytes = (c.bits == 4) ? 8u : 16u;
        if (flags & CP_FLAGS_BAD_DXTN_TAILS)
        {
            pitch = std::max<uint64_t>(1u, uint64_t(width >> 2) * bytes);
            slice = std::max<uint64_t>(1u, pitch * uint64_t(height >> 2));
        }
        else
        {
            pitch = std::max<uint64_t>(1u, (uint64_t(width) + 3u) / 4u) * bytes;
            slice = pitch * std::max<uint64_t>(1u, (uint64_t(height) + 3u) / 4u);
        }
    }
    else if (g)
    {
        if (g->evenHeight && (height & 1u)) return E_INVALIDARG;
        pitch = ((uint64_t(width) + g->px - 1u) / g->px) * g->bytes;
        slice = pitch * uint64_t(ComputeScanlines(fmt, height));
    }
    else
    {
        const uint64_t bpp = (flags & CP_FLAGS_24BPP) ? 24u : (flags & CP_FLAGS_16BPP) ? 16u : (flags & CP_FLAGS_8BPP) ? 8u : uint64_t(BitsPerPixel(fmt));
        if (!bpp) return E_INVALIDARG;
        const uint64_t align = (flags & CP_FLAGS_PAGE4K) ? 32768u : (flags & CP_FLAGS_ZMM) ? 512u : (flags & CP_FLAGS_YMM) ? 256u : (flags & CP_FLAGS_PARAGRAPH) ? 128u :
                               (flags & CP_FLAGS_LEGACY_DWORD) ? 32u : 8u;          // bits; the largest requested alignment wins
        pitch = ((uint64_t(width) * bpp + align - 1u) / align) * (align / 8u);
        slice = pitch * uint64_t(height);
    }
    rowPitch = static_cast<size_t>(pitch); slicePitch = static_cast<size_t>(slice);
    return S_OK;
}

bool CalculateMipLevels(size_t width, size_t height, size_t& mipLevels) noexcept
{
    return dxb200_calculate_mip_levels(width, height, &mipLevels) == 0;
}

size_t TexMetadata::ComputeIndex(size_t mip, size_t item, size_t slice) const noexcept
{
    if (mip >= mipLevels || dimension == TEX_DIMENSION_TEXTURE3D) return size_t(-1);
    if (slice > 0 || item >= arraySize) return size_t(-1);
    return item * mipLevels + mip;
}

// ---------------------------------------------------------------------------------------------------
ScratchImage& ScratchImage::operator=(ScratchImage&& o) noexcept
{
    if (this != &o)
    {
        Release();
        m_nimages = o.m_nimages; m_size = o.m_size; m_metadata = o.m_metadata; m_image = o.m_image; m_memory = o.m_memory;
        o.m_nimages = 0; o.m_size = 0; o.m_image = nullptr; o.m_memory = nullptr;
    }
    return *this;
}

void ScratchImage::Release() noexcept
{
    m_nimages = 0; m_size = 0;
    delete[] m_image; m_image = nullptr;
    if (m_memory) { std::free(m_memory); m_memory = nullptr; }
    std::memset(&m_metadata, 0, sizeof(m_metadata));
}

HRESULT ScratchImage::Initialize(const TexMetadata& mdata, CP_FLAGS flags) noexcept
{
    if (mdata.dimension != TEX_DIMENSION_TEXTURE2D && mdata.dimension != TEX_DIMENSION_TEXTURE1D) return HRESULT_E_NOT_SUPPORTED;   // no volume maps on this path
    if (!mdata.width || !mdata.height || mdata.depth != 1 || !mdata.arraySize) return E_INVALIDARG;
    if ((mdata.miscFlags & 0x4u) && (mdata.arraySize % 6) != 0) return E_INVALIDARG;      // TEX_MISC_TEXTURECUBE (DirectXTexImage.cpp:324-328)
    size_t mipLevels = mdata.mipLevels;
    if (!CalculateMipLevels(mdata.width, mdata.height, mipLevels)) return E_INVALIDARG;
    Release();
    // item-major, mip-minor; every image occupies slicePitch bytes; one zero-filled 16-byte aligned block
    size_t total = 0;
    {
        size_t w = mdata.width, h = mdata.height;
        for (size_t l = 0; l < mipLevels; ++l)
        {
            size_t row = 0, slice = 0;
            const HRESULT hr = ComputePitch(mdata.format, w, h, row, slice, flags);
            if (FAILED(hr)) return hr;
            total += slice;
            if (h > 1) h >>= 1;
            if (w > 1) w >>= 1;
        }
        total *= mdata.arraySize;
    }
    const size_t nimages = mdata.arraySize * mipLevels;
    m_image = new (std::nothrow) Image[nimages];
    if (!m_image) return E_OUTOFMEMORY;
    m_memory = static_cast<uint8_t*>(std::aligned_alloc(16, (total + 15) & ~size_t(15)));
    if (!m_memory) { Release(); return E_OUTOFMEMORY; }
    std::memset(m_memory, 0, total);
    m_nimages = nimages; m_size = total;
    m_metadata = mdata; m_metadata.mipLevels = mipLevels; m_metadata.depth = 1;
    uint8_t* p = m_memory;
    size_t idx = 0;
    for (size_t item = 0; item < mdata.arraySize; ++item)
    {
        size_t w = mdata.width, h = mdata.height;
        for (size_t l = 0; l < mipLevels; ++l, ++idx)
        {
            size_t row = 0, slice = 0;
            ComputePitch(mdata.format, w, h, row, slice, flags);
            Image& im = m_image[idx];
            im.width = w; im.height = h; im.format = mdata.format; im.rowPitch = row; im.slicePitch = slice; im.pixels = p;
            p += slice;
            if (h > 1) h >>= 1;
            if (w > 1) w >>= 1;
        }
    }
    return S_OK;
}

HRESULT ScratchImage::Initialize2D(DXGI_FORMAT fmt, size_t width, size_t height, size_t arraySize, size_t mipLevels, CP_FLAGS flags) noexcept
{
    TexMetadata m{};
    m.width = width; m.height = height; m.depth = 1; m.arraySize = arraySize; m.mipLevels = mipLevels;
    m.format = fmt; m.dimension = TEX_DIMENSION_TEXTURE2D;
    return Initialize(m, flags);
}

// DirectXTexImage.cpp:400-455, 510-640: the 1D / cube / from-images variants are the 2D array case plus a dimension or cube flag and a
// row-by-row copy of the callers' pixels (min of the two pitches per row, ComputeScanlines rows).
HRESULT ScratchImage::Initialize1D(DXGI_FORMAT fmt, size_t length, size_t arraySize, size_t mipLevels, CP_FLAGS flags) noexcept
{
    if (!length || !arraySize) return E_INVALIDARG;
    const HRESULT hr = Initialize2D(fmt, length, 1, arraySize, mipLevels, flags);
    if (SUCCEEDED(hr)) m_metadata.dimension = TEX_DIMENSION_TEXTURE1D;
    return hr;
}

HRESULT ScratchImage::InitializeCube(DXGI_FORMAT fmt, size_t width, size_t height, size_t nCubes, size_t mipLevels, CP_FLAGS flags) noexcept
{
    if (!width || !height || !nCubes) return E_INVALIDARG;
    const HRESULT hr = Initialize2D(fmt, width, height, nCubes * 6, mipLevels, flags);
    if (SUCCEEDED(hr)) m_metadata.miscFlags |= 0x4u;                     // TEX_MISC_TEXTURECUBE
    return hr;
}

namespace
{
    HRESULT copy_rows(const Image& src, const Image& dst)
    {
        const size_t rows = ComputeScanlines(src.format, src.height);
        if (!rows) return static_cast<HRESULT>(0x8000FFFF);               // E_UNEXPECTED
        if (!src.pixels || !dst.pixels) return E_POINTER;
        const size_t n = dst.rowPitch < src.rowPitch ? dst.rowPitch : src.rowPitch;
        for (size_t y = 0; y < rows; ++y) std::memcpy(dst.pixels + y * dst.rowPitch, src.pixels + y * src.rowPitch, n);
        return S_OK;
    }
}

HRESULT ScratchImage::InitializeFromImage(const Image& src, bool allow1D, CP_FLAGS flags) noexcept
{
    const HRESULT hr = (src.height > 1 || !allow1D) ? Initialize2D(src.format, src.width, src.height, 1, 1, flags) : Initialize1D(src.format, src.width, 1, 1, flags);
    if (FAILED(hr)) return hr;
    return copy_rows(src, m_image[0]);
}

HRESULT ScratchImage::InitializeArrayFromImages(const Image* images, size_t nImages, bool allow1D, CP_FLAGS flags) noexcept
{
    if (!images || !nImages) return E_INVALIDARG;
    for (size_t i = 0; i < nImages; ++i)
    {
        if (!images[i].pixels) return E_POINTER;
        if (images[i].format != images[0].format || images[i].width != images[0].width || images[i].height != images[0].height) return E_FAIL;   // one format and size
    }
    const Image& f = images[0];
    HRESULT hr = (f.height > 1 || !allow1D) ? Initialize2D(f.format, f.width, f.height, nImages, 1, flags) : Initialize1D(f.format, f.width, nImages, 1, flags);
    for (size_t i = 0; i < nImages && SUCCEEDED(hr); ++i) hr = copy_rows(images[i], m_image[i]);
    return hr;
}

HRESULT ScratchImage::InitializeCubeFromImages(const Image* images, size_t nImages, CP_FLAGS flags) noexcept
{
    if (!images || !nImages || (nImages % 6) != 0) return E_INVALIDARG;  // whole cubes only
    const HRESULT hr = InitializeArrayFromImages(images, nImages, false, flags);
    if (SUCCEEDED(hr)) m_metadata.miscFlags |= 0x4u;
    return hr;
}

bool ScratchImage::OverrideFormat(DXGI_FORMAT f) noexcept
{
    if (!m_image || !IsValid(f) || IsPlanar(f) || IsPalettized(f)) return false;
    for (size_t i = 0; i < m_nimages; ++i) m_image[i].format = f;
    m_metadata.format = f;
    return true;
}

const Image* ScratchImage::GetImage(size_t mip, size_t item, size_t slice) const noexcept
{
    const size_t i = m_metadata.ComputeIndex(mip, item, slice);
    return (i < m_nimages) ? &m_image[i] : nullptr;
}

// ---------------------------------------------------------------------------------------------------
// Compress
namespace
{
    // std::function status callback -> the C ABI's (done, total, user) callback
    int status_trampoline(size_t done, size_t total, void* user)
    {
        auto* f = static_cast<std::function<bool(size_t, size_t)>*>(user);
        try { return (*f)(done, total) ? 1 : 0; } catch (...) { return 0; }
    }
}

HRESULT Compress(const Image& src, DXGI_FORMAT format, TEX_COMPRESS_FLAGS compress, float threshold, ScratchImage& image) noexcept
{
    CompressOptions o{ compress, threshold, TEX_ALPHA_WEIGHT_DEFAULT };
    try { return CompressEx(src, format, o, image, nullptr); } catch (...) { return E_FAIL; }
}

HRESULT Compress(const Image* srcImages, size_t nimages, const TexMetadata& metadata, DXGI_FORMAT format, TEX_COMPRESS_FLAGS compress, float threshold, ScratchImage& cImages) noexcept
{
    CompressOptions o{ compress, threshold, TEX_ALPHA_WEIGHT_DEFAULT };
    try { return CompressEx(srcImages, nimages, metadata, format, o, cImages, nullptr); } catch (...) { return E_FAIL; }
}

HRESULT CompressEx(const Image& src, DXGI_FORMAT format, const CompressOptions& options, ScratchImage& image, std::function<bool(size_t, size_t)> cb)
{
    if (IsCompressed(src.format) || !IsCompressed(format)) return E_INVALIDARG;
    if (!implemented_pixel_format(src.format)) return HRESULT_E_NOT_SUPPORTED;
    HRESULT hr = image.Initialize2D(format, src.width, src.height, 1, 1);
    if (FAILED(hr)) return hr;
    const Image* img = image.GetImage(0, 0, 0);
    if (!img) { image.Release(); return E_POINTER; }
    // the C ABI reports (rows done, height) before every band of block rows and (height, height) at the end, and returns E_ABORT
    // between bands when the callback says stop (DirectXTexCompress.cpp:115-121, 690-724)
    const dxb200_image s = to_c(src), d = to_c(*img);
    hr = dxb200_compress_ex(&s, 1, static_cast<uint32_t>(format), static_cast<uint32_t>(options.flags), options.threshold, options.alphaWeight, &d,
                            cb ? status_trampoline : nullptr, cb ? &cb : nullptr);
    if (FAILED(hr)) { image.Release(); return hr; }
    return S_OK;
}

HRESULT CompressEx(const Image* srcImages, size_t nimages, const TexMetadata& metadata, DXGI_FORMAT format, const CompressOptions& options,
                   ScratchImage& cImages, std::function<bool(size_t, size_t)> cb)
{
    if (!srcImages || !nimages) return E_INVALIDARG;
    if (IsCompressed(metadata.format) || !IsCompressed(format)) return E_INVALIDARG;
    if (!implemented_pixel_format(metadata.format)) return HRESULT_E_NOT_SUPPORTED;
    cImages.Release();
    if (cb && nimages == 1 && !metadata.IsVolumemap() && metadata.mipLevels == 1 && metadata.arraySize == 1)
        return CompressEx(srcImages[0], format, options, cImages, cb);
    TexMetadata m2 = metadata; m2.format = format;
    HRESULT hr = cImages.Initialize(m2);
    if (FAILED(hr)) return hr;
    if (nimages != cImages.GetImageCount()) { cImages.Release(); return E_FAIL; }
    const Image* dest = cImages.GetImages();
    // images of one mip level share a size; the C ABI takes arbitrary per-image sizes in one batch
    std::vector<dxb200_image> s(nimages), d(nimages);
    for (size_t i = 0; i < nimages; ++i)
    {
        if (srcImages[i].width != dest[i].width || srcImages[i].height != dest[i].height) { cImages.Release(); return E_FAIL; }
        s[i] = to_c(srcImages[i]); d[i] = to_c(dest[i]);
    }
    hr = dxb200_compress_ex(s.data(), nimages, static_cast<uint32_t>(format), static_cast<uint32_t>(options.flags), options.threshold, options.alphaWeight, d.data(),
                            cb ? status_trampoline : nullptr, cb ? &cb : nullptr);          // (images done, nimages), :785-837
    if (FAILED(hr)) { cImages.Release(); return hr; }
    return S_OK;
}

// ---------------------------------------------------------------------------------------------------
// ComputeMSE (DirectXTexMisc.cpp:388-468) and ScratchImage::IsAlphaAllOpaque (DirectXTexImage.cpp:800-852)
HRESULT ComputeMSE(const Image& image1, const Image& image2, float& mse, float* mseV, CMSE_FLAGS flags) noexcept
{
    const dxb200_image a = to_c(image1), b = to_c(image2);
    return dxb200_compute_mse(&a, &b, 1, static_cast<uint32_t>(flags), &mse, mseV);
}

bool ScratchImage::IsAlphaAllOpaque() const noexcept
{
    if (!m_image) return false;
    if (!HasAlpha(m_metadata.format)) return true;
    DXGI_FORMAT f = m_metadata.format;
    switch (f)                     // IsAlphaAllOpaqueBC promotes the typeless BC formats (DirectXTexCompress.cpp:545-553)
    {
    case DXGI_FORMAT_BC1_TYPELESS: f = DXGI_FORMAT_BC1_UNORM; break;
    case DXGI_FORMAT_BC2_TYPELESS: f = DXGI_FORMAT_BC2_UNORM; break;
    case DXGI_FORMAT_BC3_TYPELESS: f = DXGI_FORMAT_BC3_UNORM; break;
    case DXGI_FORMAT_BC7_TYPELESS: f = DXGI_FORMAT_BC7_UNORM; break;
    default: break;
    }
    std::vector<dxb200_image> imgs(m_nimages);
    for (size_t i = 0; i < m_nimages; ++i) { imgs[i] = to_c(m_image[i]); imgs[i].format = static_cast<uint32_t>(f); }
    int32_t opaque = 0;
    if (FAILED(dxb200_is_alpha_all_opaque(imgs.data(), imgs.size(), &opaque))) return false;
    return opaque != 0;
}

// ---------------------------------------------------------------------------------------------------
// Decompress
HRESULT Decompress(const Image& cImage, DXGI_FORMAT format, ScratchImage& image) noexcept
{
    if (!IsCompressed(cImage.format) || IsCompressed(format)) return E_INVALIDARG;
    if (format == DXGI_FORMAT_UNKNOWN)
    {
        switch (cImage.format)         // DefaultDecompress, DirectXTexCompress.cpp:377-421
        {
        case DXGI_FORMAT_BC4_UNORM: format = DXGI_FORMAT_R8_UNORM; break;
        case DXGI_FORMAT_BC4_SNORM: format = DXGI_FORMAT_R8_SNORM; break;
        case DXGI_FORMAT_BC5_UNORM: format = DXGI_FORMAT_R8G8_UNORM; break;
        case DXGI_FORMAT_BC5_SNORM: format = DXGI_FORMAT_R8G8_SNORM; break;
        case DXGI_FORMAT_BC6H_UF16: case DXGI_FORMAT_BC6H_SF16: format = DXGI_FORMAT_R32G32B32A32_FLOAT; break;
        default: format = IsSRGB(cImage.format) ? DXGI_FORMAT_R8G8B8A8_UNORM_SRGB : DXGI_FORMAT_R8G8B8A8_UNORM; break;
        }
    }
    HRESULT hr = image.Initialize2D(format, cImage.width, cImage.height, 1, 1);
    if (FAILED(hr)) return hr;
    const dxb200_image s = to_c(cImage), d = to_c(*image.GetImage(0, 0, 0));
    hr = dxb200_decompress(&s, 1, static_cast<uint32_t>(format), &d);
    if (FAILED(hr)) image.Release();
    return hr;
}

HRESULT Decompress(const Image* cImages, size_t nimages, const TexMetadata& metadata, DXGI_FORMAT format, ScratchImage& images) noexcept
{
    if (!cImages || !nimages) return E_INVALIDARG;
    if (!IsCompressed(metadata.format) || IsCompressed(format) || format == DXGI_FORMAT_UNKNOWN) return E_INVALIDARG;
    images.Release();
    TexMetadata m2 = metadata; m2.format = format;
    HRESULT hr = images.Initialize(m2);
    if (FAILED(hr)) return hr;
    if (nimages != images.GetImageCount()) { images.Release(); return E_FAIL; }
    std::vector<dxb200_image> s(nimages), d(nimages);
    for (size_t i = 0; i < nimages; ++i) { s[i] = to_c(cImages[i]); d[i] = to_c(images.GetImages()[i]); }
    hr = dxb200_decompress(s.data(), nimages, static_cast<uint32_t>(format), d.data());
    if (FAILED(hr)) images.Release();
    return hr;
}

// ---------------------------------------------------------------------------------------------------
// Convert
HRESULT Convert(const Image& src, DXGI_FORMAT format, TEX_FILTER_FLAGS filter, float threshold, ScratchImage& image) noexcept
{
    ConvertOptions o{ filter, threshold };
    try { return ConvertEx(src, format, o, image, nullptr); } catch (...) { return E_FAIL; }
}

HRESULT Convert(const Image* srcImages, size_t nimages, const TexMetadata& metadata, DXGI_FORMAT format, TEX_FILTER_FLAGS filter, float threshold, ScratchImage& result) noexcept
{
    ConvertOptions o{ filter, threshold };
    try { return ConvertEx(srcImages, nimages, metadata, format, o, result, nullptr); } catch (...) { return E_FAIL; }
}

HRESULT ConvertEx(const Image& src, DXGI_FORMAT format, const ConvertOptions& options, ScratchImage& image, std::function<bool(size_t, size_t)> cb)
{
    if (src.format == format || IsCompressed(src.format) || IsCompressed(format)) return E_INVALIDARG;
    if (!implemented_pixel_format(src.format) || !implemented_pixel_format(format)) return HRESULT_E_NOT_SUPPORTED;
    if (src.width > 0xFFFFFFFFull || src.height > 0xFFFFFFFFull) return E_INVALIDARG;
    HRESULT hr = image.Initialize2D(format, src.width, src.height, 1, 1);
    if (FAILED(hr)) return hr;
    const Image* rimage = image.GetImage(0, 0, 0);
    if (!rimage) { image.Release(); return E_POINTER; }
    const dxb200_image s = to_c(src), d = to_c(*rimage);
    hr = dxb200_convert_ex(&s, 1, static_cast<uint32_t>(format), static_cast<uint32_t>(options.filter), options.threshold, &d,
                           cb ? status_trampoline : nullptr, cb ? &cb : nullptr);
    if (FAILED(hr)) { image.Release(); return hr; }
    return S_OK;
}

HRESULT ConvertEx(const Image* srcImages, size_t nimages, const TexMetadata& metadata, DXGI_FORMAT format, const ConvertOptions& options,
                  ScratchImage& result, std::function<bool(size_t, size_t)> cb)
{
    if (!srcImages || !nimages || metadata.format == format) return E_INVALIDARG;
    if (IsCompressed(metadata.format) || IsCompressed(format)) return E_INVALIDARG;
    if (!implemented_pixel_format(metadata.format) || !implemented_pixel_format(format)) return HRESULT_E_NOT_SUPPORTED;
    TexMetadata m2 = metadata; m2.format = format;
    HRESULT hr = result.Initialize(m2);
    if (FAILED(hr)) return hr;
    if (nimages != result.GetImageCount()) { result.Release(); return E_FAIL; }
    std::vector<dxb200_image> s(nimages), d(nimages);
    for (size_t i = 0; i < nimages; ++i) { s[i] = to_c(srcImages[i]); d[i] = to_c(result.GetImages()[i]); }
    hr = dxb200_convert_ex(s.data(), nimages, static_cast<uint32_t>(format), static_cast<uint32_t>(options.filter), options.threshold, d.data(),
                           cb ? status_trampoline : nullptr, cb ? &cb : nullptr);
    if (FAILED(hr)) { result.Release(); return hr; }
    return S_OK;
}

// ---------------------------------------------------------------------------------------------------
// GenerateMipMaps
HRESULT GenerateMipMaps(const Image& baseImage, TEX_FILTER_FLAGS filter, size_t levels, ScratchImage& mipChain, bool) noexcept
{
    TexMetadata m{};
    m.width = baseImage.width; m.height = baseImage.height; m.depth = 1; m.arraySize = 1; m.mipLevels = 1;
    m.format = baseImage.format; m.dimension = TEX_DIMENSION_TEXTURE2D;
    try { return GenerateMipMaps(&baseImage, 1, m, filter, levels, mipChain); } catch (...) { return E_FAIL; }
}

HRESULT GenerateMipMaps(const Image* srcImages, size_t nimages, const TexMetadata& metadata, TEX_FILTER_FLAGS filter, size_t levels, ScratchImage& mipChain)
{
    if (!srcImages || !nimages || !metadata.width || !metadata.height) return E_INVALIDARG;
    if (metadata.IsVolumemap() || IsCompressed(metadata.format)) return HRESULT_E_NOT_SUPPORTED;
    if (!CalculateMipLevels(metadata.width, metadata.height, levels)) return E_INVALIDARG;
    if (levels <= 1) return E_INVALIDARG;
    if (!implemented_pixel_format(metadata.format)) return HRESULT_E_NOT_SUPPORTED;
    // the base image of every item through ComputeIndex(0, item, 0) (DirectXTexMipmaps.cpp:3040-3059): the caller may pass a
    // ScratchImage that still carries its old mip levels (nimages = arraySize * mipLevels) or just the base images
    std::vector<const Image*> base(metadata.arraySize);
    for (size_t item = 0; item < metadata.arraySize; ++item)
    {
        const size_t index = metadata.ComputeIndex(0, item, 0);
        if (index >= nimages) return E_FAIL;
        const Image& src = srcImages[index];
        if (!src.pixels) return E_POINTER;
        if (src.format != metadata.format || src.width != metadata.width || src.height != metadata.height) return E_FAIL;
        base[item] = &src;
    }
    TexMetadata m2 = metadata; m2.mipLevels = levels;
    HRESULT hr = mipChain.Initialize(m2);
    if (FAILED(hr)) return hr;
    // copy the base image of each item to the top of its chain (Setup2DMips)
    for (size_t item = 0; item < metadata.arraySize; ++item)
    {
        const Image& src = *base[item];
        const Image* dest = mipChain.GetImage(0, item, 0);
        if (!dest) { mipChain.Release(); return E_POINTER; }
        const size_t n = dest->rowPitch < src.rowPitch ? dest->rowPitch : src.rowPitch;
        for (size_t y = 0; y < src.height; ++y) std::memcpy(dest->pixels + y * dest->rowPitch, src.pixels + y * src.rowPitch, n);
    }
    std::vector<dxb200_image> chain(mipChain.GetImageCount());
    for (size_t i = 0; i < chain.size(); ++i) chain[i] = to_c(mipChain.GetImages()[i]);
    hr = dxb200_generate_mipmaps(chain.data(), metadata.arraySize, levels, static_cast<uint32_t>(filter));
    if (FAILED(hr)) mipChain.Release();
    return hr;
}

// ---------------------------------------------------------------------------------------------------
// Resize (DirectXTexResize.cpp:854-935, 942-1120): 2D textures and arrays, top level only (the result has one mip level)
HRESULT Resize(const Image& srcImage, size_t width, size_t height, TEX_FILTER_FLAGS filter, ScratchImage& image) noexcept
{
    if (width == 0 || height == 0) return E_INVALIDARG;
    if (!srcImage.pixels) return E_POINTER;
    TexMetadata m{};
    m.width = srcImage.width; m.height = srcImage.height; m.depth = 1; m.arraySize = 1; m.mipLevels = 1;
    m.format = srcImage.format; m.dimension = TEX_DIMENSION_TEXTURE2D;
    return Resize(&srcImage, 1, m, width, height, filter, image);
}

HRESULT Resize(const Image* srcImages, size_t nimages, const TexMetadata& metadata, size_t width, size_t height, TEX_FILTER_FLAGS filter, ScratchImage& result) noexcept
{
    if (!srcImages || !nimages || width == 0 || height == 0) return E_INVALIDARG;
    if (metadata.IsVolumemap()) return HRESULT_E_NOT_SUPPORTED;
    if (IsCompressed(metadata.format)) return HRESULT_E_NOT_SUPPORTED;
    if (!implemented_pixel_format(metadata.format)) return HRESULT_E_NOT_SUPPORTED;
    try
    {
        TexMetadata m2 = metadata;
        m2.width = width; m2.height = height; m2.mipLevels = 1;
        HRESULT hr = result.Initialize(m2);
        if (FAILED(hr)) return hr;
        // the base image of every array item (metadata.ComputeIndex(0, item, 0) in the reference)
        std::vector<dxb200_image> src(metadata.arraySize), dst(metadata.arraySize);
        for (size_t item = 0; item < metadata.arraySize; ++item)
        {
            const size_t srcIndex = item * metadata.mipLevels;
            if (srcIndex >= nimages) { result.Release(); return E_FAIL; }
            const Image* d = result.GetImage(0, item, 0);
            if (!d) { result.Release(); return E_POINTER; }
            if (srcImages[srcIndex].format != metadata.format) { result.Release(); return E_FAIL; }
            src[item] = to_c(srcImages[srcIndex]); dst[item] = to_c(*d);
        }
        hr = dxb200_resize(src.data(), src.size(), static_cast<uint32_t>(filter), dst.data());
        if (FAILED(hr)) result.Release();
        return hr;
    }
    catch (...) { return E_FAIL; }
}

// ---------------------------------------------------------------------------------------------------
// PremultiplyAlpha (DirectXTexPMAlpha.cpp:214-344)
HRESULT PremultiplyAlpha(const Image& srcImage, TEX_PMALPHA_FLAGS flags, ScratchImage& image) noexcept
{
    if (!srcImage.pixels) return E_POINTER;
    if (IsCompressed(srcImage.format) || !implemented_pixel_format(srcImage.format)) return HRESULT_E_NOT_SUPPORTED;
    try
    {
        HRESULT hr = image.Initialize2D(srcImage.format, srcImage.width, srcImage.height, 1, 1);
        if (FAILED(hr)) return hr;
        const Image* r = image.GetImage(0, 0, 0);
        if (!r) { image.Release(); return E_POINTER; }
        const dxb200_image s = to_c(srcImage), d = to_c(*r);
        hr = dxb200_premultiply_alpha(&s, 1, static_cast<uint32_t>(flags), &d);
        if (FAILED(hr)) image.Release();
        return hr;
    }
    catch (...) { return E_FAIL; }
}

HRESULT PremultiplyAlpha(const Image* srcImages, size_t nimages, const TexMetadata& metadata, TEX_PMALPHA_FLAGS flags, ScratchImage& result) noexcept
{
    if (!srcImages || !nimages) return E_INVALIDARG;
    if (IsCompressed(metadata.format) || !implemented_pixel_format(metadata.format)) return HRESULT_E_NOT_SUPPORTED;
    if (metadata.IsPMAlpha() != ((flags & TEX_PMALPHA_REVERSE) != 0)) return E_FAIL;                       // :297-298
    try
    {
        TexMetadata m2 = metadata;
        m2.SetAlphaMode((flags & TEX_PMALPHA_REVERSE) ? TEX_ALPHA_MODE_STRAIGHT : TEX_ALPHA_MODE_PREMULTIPLIED);
        HRESULT hr = result.Initialize(m2);
        if (FAILED(hr)) return hr;
        if (nimages != result.GetImageCount()) { result.Release(); return E_FAIL; }
        std::vector<dxb200_image> src(nimages), dst(nimages);
        for (size_t i = 0; i < nimages; ++i)
        {
            const Image& s = srcImages[i]; const Image& d = result.GetImages()[i];
            if (s.format != metadata.format) { result.Release(); return E_FAIL; }
            if (s.width != d.width || s.height != d.height) { result.Release(); return E_FAIL; }
            src[i] = to_c(s); dst[i] = to_c(d);
        }
        // mip levels have different sizes: one call per distinct size keeps every call uniform
        size_t i = 0;
        while (i < nimages && SUCCEEDED(hr))
        {
            size_t k = i + 1;
            while (k < nimages && src[k].width == src[i].width && src[k].height == src[i].height) ++k;
            hr = dxb200_premultiply_alpha(src.data() + i, k - i, static_cast<uint32_t>(flags), dst.data() + i);
            i = k;
        }
        if (FAILED(hr)) result.Release();
        return hr;
    }
    catch (...) { return E_FAIL; }
}

// ---------------------------------------------------------------------------------------------------
// ScaleMipMapsAlphaForCoverage (DirectXTexMipmaps.cpp:3483-3552): srcImages = the mip levels of one item, mipChain = an
// initialised chain of the same shape whose item `item` receives the result
HRESULT ScaleMipMapsAlphaForCoverage(const Image* srcImages, size_t nimages, const TexMetadata& metadata, size_t item, float alphaReference, ScratchImage& mipChain) noexcept
{
    if (!srcImages || !nimages || nimages > metadata.mipLevels || !mipChain.GetImages()) return E_INVALIDARG;
    if (metadata.IsVolumemap() || IsCompressed(metadata.format) || !implemented_pixel_format(metadata.format)) return HRESULT_E_NOT_SUPPORTED;
    if (srcImages[0].format != metadata.format || srcImages[0].width != metadata.width || srcImages[0].height != metadata.height) return E_FAIL;
    if (nimages < metadata.mipLevels) return E_FAIL;                                             // :3535-3536 (level >= nimages)
    try
    {
        std::vector<dxb200_image> src(metadata.mipLevels), dst(metadata.mipLevels);
        for (size_t level = 0; level < metadata.mipLevels; ++level)
        {
            const Image* d = mipChain.GetImage(level, item, 0);
            if (!d || !d->pixels) return E_POINTER;
            src[level] = to_c(srcImages[level]); dst[level] = to_c(*d);
        }
        return dxb200_scale_mipmaps_alpha_for_coverage(src.data(), src.size(), alphaReference, dst.data());
    }
    catch (...) { return E_OUTOFMEMORY; }
}

// ---------------------------------------------------------------------------------------------------
// DDS container (DirectXTexDDS.cpp); the format logic lives behind the C ABI (host/dxb_dds.cpp)
Blob& Blob::operator=(Blob&& o) noexcept
{
    if (this != &o) { Release(); m_buffer = o.m_buffer; m_size = o.m_size; o.m_buffer = nullptr; o.m_size = 0; }
    return *this;
}
HRESULT Blob::Initialize(size_t size) noexcept
{
    if (!size) return E_INVALIDARG;
    Release();
    m_buffer = static_cast<uint8_t*>(std::malloc(size));
    if (!m_buffer) return E_OUTOFMEMORY;
    m_size = size;
    return S_OK;
}
void Blob::Release() noexcept { std::free(m_buffer); m_buffer = nullptr; m_size = 0; }

namespace {
    dxb200_metadata md_to_c(const TexMetadata& m) noexcept
    {
        return { m.width, m.height, m.depth, m.arraySize, m.mipLevels, m.miscFlags, m.miscFlags2, static_cast<uint32_t>(m.format), static_cast<uint32_t>(m.dimension) };
    }
    TexMetadata from_c(const dxb200_metadata& m) noexcept
    {
        TexMetadata r{};
        r.width = m.width; r.height = m.height; r.depth = m.depth; r.arraySize = m.arraySize; r.mipLevels = m.mipLevels;
        r.miscFlags = m.miscFlags; r.miscFlags2 = m.miscFlags2; r.format = static_cast<DXGI_FORMAT>(m.format); r.dimension = static_cast<TEX_DIMENSION>(m.dimension);
        return r;
    }
    HRESULT read_file(const char* path, std::vector<uint8_t>& data) noexcept
    {
        if (!path) return E_INVALIDARG;
        FILE* f = std::fopen(path, "rb");
        if (!f) return static_cast<HRESULT>(0x80070002);                     // HRESULT_FROM_WIN32(ERROR_FILE_NOT_FOUND)
        std::fseek(f, 0, SEEK_END); const long n = std::ftell(f); std::fseek(f, 0, SEEK_SET);
        HRESULT hr = S_OK;
        try { data.resize(n > 0 ? static_cast<size_t>(n) : 0); } catch (...) { hr = E_OUTOFMEMORY; }
        if (SUCCEEDED(hr) && std::fread(data.data(), 1, data.size(), f) != data.size()) hr = E_FAIL;
        std::fclose(f);
        return hr;
    }
}

HRESULT GetMetadataFromDDSMemory(const uint8_t* pSource, size_t size, DDS_FLAGS flags, TexMetadata& metadata) noexcept
{
    if (!pSource || !size) return E_INVALIDARG;
    dxb200_metadata m;
    const HRESULT hr = dxb200_dds_get_metadata(pSource, size, static_cast<uint32_t>(flags), &m, nullptr);
    if (SUCCEEDED(hr)) metadata = from_c(m);
    return hr;
}
HRESULT GetMetadataFromDDSFile(const char* szFile, DDS_FLAGS flags, TexMetadata& metadata) noexcept
{
    std::vector<uint8_t> data;
    const HRESULT hr = read_file(szFile, data);
    return FAILED(hr) ? hr : GetMetadataFromDDSMemory(data.data(), data.size(), flags, metadata);
}
HRESULT LoadFromDDSMemory(const uint8_t* pSource, size_t size, DDS_FLAGS flags, TexMetadata* metadata, ScratchImage& image) noexcept
{
    if (!pSource || !size) return E_INVALIDARG;
    image.Release();
    dxb200_metadata m;
    HRESULT hr = dxb200_dds_get_metadata(pSource, size, static_cast<uint32_t>(flags), &m, nullptr);
    if (FAILED(hr)) return hr;
    try
    {
        const TexMetadata md = from_c(m);
        hr = image.Initialize(md);
        if (FAILED(hr)) return hr;
        std::vector<dxb200_image> imgs(image.GetImageCount());
        for (size_t i = 0; i < imgs.size(); ++i) imgs[i] = to_c(image.GetImages()[i]);
        hr = dxb200_dds_load_memory(pSource, size, static_cast<uint32_t>(flags), imgs.data(), imgs.size());
        if (FAILED(hr)) { image.Release(); return hr; }
        if (metadata) *metadata = md;
        return S_OK;
    }
    catch (...) { image.Release(); return E_OUTOFMEMORY; }
}
HRESULT LoadFromDDSFile(const char* szFile, DDS_FLAGS flags, TexMetadata* metadata, ScratchImage& image) noexcept
{
    std::vector<uint8_t> data;
    const HRESULT hr = read_file(szFile, data);
    return FAILED(hr) ? hr : LoadFromDDSMemory(data.data(), data.size(), flags, metadata, image);
}
HRESULT SaveToDDSMemory(const Image* images, size_t nimages, const TexMetadata& metadata, DDS_FLAGS flags, Blob& blob) noexcept
{
    if (!images || !nimages) return E_INVALIDARG;
    try
    {
        std::vector<dxb200_image> imgs(nimages);
        for (size_t i = 0; i < nimages; ++i) imgs[i] = to_c(images[i]);
        const dxb200_metadata m = md_to_c(metadata);
        size_t need = 0;
        HRESULT hr = dxb200_dds_save_memory(imgs.data(), nimages, &m, static_cast<uint32_t>(flags), nullptr, 0, &need);
        if (FAILED(hr)) return hr;
        blob.Release();
        hr = blob.Initialize(need);
        if (FAILED(hr)) return hr;
        hr = dxb200_dds_save_memory(imgs.data(), nimages, &m, static_cast<uint32_t>(flags), blob.GetBufferPointer(), blob.GetBufferSize(), &need);
        if (FAILED(hr)) blob.Release();
        return hr;
    }
    catch (...) { return E_OUTOFMEMORY; }
}
HRESULT SaveToDDSMemory(const Image& image, DDS_FLAGS flags, Blob& blob) noexcept
{
    TexMetadata m{};
    m.width = image.width; m.height = image.height; m.depth = 1; m.arraySize = 1; m.mipLevels = 1;
    m.format = image.format; m.dimension = TEX_DIMENSION_TEXTURE2D;
    return SaveToDDSMemory(&image, 1, m, flags, blob);
}
HRESULT SaveToDDSFile(const Image* images, size_t nimages, const TexMetadata& metadata, DDS_FLAGS flags, const char* szFile) noexcept
{
    if (!szFile) return E_INVALIDARG;
    Blob blob;
    HRESULT hr = SaveToDDSMemory(images, nimages, metadata, flags, blob);
    if (FAILED(hr)) return hr;
    FILE* f = std::fopen(szFile, "wb");
    if (!f) return E_FAIL;
    if (std::fwrite(blob.GetConstBufferPointer(), 1, blob.GetBufferSize(), f) != blob.GetBufferSize()) hr = E_FAIL;
    std::fclose(f);
    return hr;
}
HRESULT SaveToDDSFile(const Image& image, DDS_FLAGS flags, const char* szFile) noexcept
{
    Blob blob;
    HRESULT hr = SaveToDDSMemory(image, flags, blob);
    if (FAILED(hr)) return hr;
    TexMetadata m{};
    m.width = image.width; m.height = image.height; m.depth = 1; m.arraySize = 1; m.mipLevels = 1;
    m.format = image.format; m.dimension = TEX_DIMENSION_TEXTURE2D;
    return SaveToDDSFile(&image, 1, m, flags, szFile);
}

// ---- wchar_t paths (the reference's signatures, DirectXTex.h:588-616): converted to UTF-8 and forwarded
namespace
{
    bool to_utf8(const wchar_t* w, std::string& out)
    {
        if (!w) return false;
        out.clear();
        for (; *w; ++w)
        {
            uint32_t c = static_cast<uint32_t>(*w);
            if (sizeof(wchar_t) == 2 && c >= 0xD800 && c <= 0xDBFF && w[1] >= 0xDC00 && w[1] <= 0xDFFF)
            {
                c = 0x10000u + ((c - 0xD800u) << 10) + (static_cast<uint32_t>(w[1]) - 0xDC00u); ++w;
            }
            if (c < 0x80) out.push_back(static_cast<char>(c));
            else if (c < 0x800) { out.push_back(static_cast<char>(0xC0 | (c >> 6))); out.push_back(static_cast<char>(0x80 | (c & 0x3F))); }
            else if (c < 0x10000) { out.push_back(static_cast<char>(0xE0 | (c >> 12))); out.push_back(static_cast<char>(0x80 | ((c >> 6) & 0x3F))); out.push_back(static_cast<char>(0x80 | (c & 0x3F))); }
            else { out.push_back(static_cast<char>(0xF0 | (c >> 18))); out.push_back(static_cast<char>(0x80 | ((c >> 12) & 0x3F))); out.push_back(static_cast<char>(0x80 | ((c >> 6) & 0x3F))); out.push_back(static_cast<char>(0x80 | (c & 0x3F))); }
        }
        return true;
    }
}
HRESULT GetMetadataFromDDSFile(const wchar_t* szFile, DDS_FLAGS flags, TexMetadata& metadata) noexcept
{
    try { std::string p; return to_utf8(szFile, p) ? GetMetadataFromDDSFile(p.c_str(), flags, metadata) : E_INVALIDARG; } catch (...) { return E_OUTOFMEMORY; }
}
HRESULT LoadFromDDSFile(const wchar_t* szFile, DDS_FLAGS flags, TexMetadata* metadata, ScratchImage& image) noexcept
{
    try { std::string p; return to_utf8(szFile, p) ? LoadFromDDSFile(p.c_str(), flags, metadata, image) : E_INVALIDARG; } catch (...) { return E_OUTOFMEMORY; }
}
HRESULT SaveToDDSFile(const Image& image, DDS_FLAGS flags, const wchar_t* szFile) noexcept
{
    try { std::string p; return to_utf8(szFile, p) ? SaveToDDSFile(image, flags, p.c_str()) : E_INVALIDARG; } catch (...) { return E_OUTOFMEMORY; }
}
HRESULT SaveToDDSFile(const Image* images, size_t nimages, const TexMetadata& metadata, DDS_FLAGS flags, const wchar_t* szFile) noexcept
{
    try { std::string p; return to_utf8(szFile, p) ? SaveToDDSFile(images, nimages, metadata, flags, p.c_str()) : E_INVALIDARG; } catch (...) { return E_OUTOFMEMORY; }
}

} // namespace DirectX
