// DirectXTexB200.h — C++ host-side mirror of the part of the DirectXTex public API that the B200 backend
// accelerates.  A program written against the reference's DirectXTex.h for this path
//     ScratchImage out;  HRESULT hr = DirectX::Compress(img, DXGI_FORMAT_BC7_UNORM, TEX_COMPRESS_DEFAULT, 0.5f, out);
// compiles against this header unchanged and links libdxtex_b200.so instead of libDirectXTex.  Names, argument
// meaning, memory layout, ownership and HRESULTs follow the reference (citations: DirectXTex/DirectXTex.h of
// microsoft/DirectXTex @ 0bb96f0); the implementation (DirectXTexB200.cpp) is new code that validates,
// allocates the destination exactly like the reference and forwards to the C ABI in include/dxtex_b200.h.
// Provided besides the accelerated operations: the containers (ScratchImage / Image / TexMetadata / Blob with every constructor of the 2D
// path), every DXGI format utility, ComputePitch with all CP_FLAGS, the DDS container.  Not provided (out of the hot path, SURVEY.md 8):
// WIC / TGA / HDR / EXR codecs, D3D interop, 3D textures, normal maps, TransformImage / EvaluateImage / CopyRectangle / FlipRotate.
// ComputeMSE and ScratchImage::IsAlphaAllOpaque run on the device (BC data decoded in the kernel).
#pragma once
#include <cstddef>
#include <cstdint>
#include <functional>

#if defined(__GNUC__)
#define DXTEXB200_API __attribute__((visibility("default")))
#else
#define DXTEXB200_API
#endif

typedef int32_t HRESULT;
#ifndef S_OK
#define S_OK            static_cast<HRESULT>(0)
#define E_NOTIMPL       static_cast<HRESULT>(0x80004001)
#define E_POINTER       static_cast<HRESULT>(0x80004003)
#define E_ABORT         static_cast<HRESULT>(0x80004004)
#define E_FAIL          static_cast<HRESULT>(0x80004005)
#define E_OUTOFMEMORY   static_cast<HRESULT>(0x8007000E)
#define E_INVALIDARG    static_cast<HRESULT>(0x80070057)
#define SUCCEEDED(hr)   (static_cast<HRESULT>(hr) >= 0)
#define FAILED(hr)      (static_cast<HRESULT>(hr) < 0)
#endif
#define HRESULT_E_NOT_SUPPORTED static_cast<HRESULT>(0x80070032)

// DXGI_FORMAT: the full public list (dxb_dxgi_formats.h); the backend implements the subset listed in DESIGN.md section 1
#include "dxb_dxgi_formats.h"
enum DXGI_FORMAT : uint32_t
{
#define DXB_X(name, value) DXGI_FORMAT_##name = value,
    DXB_DXGI_FORMATS(DXB_X)
#undef DXB_X
    DXGI_FORMAT_FORCE_UINT = 0xffffffff
};

namespace DirectX
{
    // ---- format utilities (DirectXTex.h:72-99, 144-154) for EVERY DXGI format: callers like texconv classify formats the backend
    // does not convert as well.  Classified from the format's name (channel list, type suffix), see DirectXTexB200.cpp.
    DXTEXB200_API bool IsValid(DXGI_FORMAT fmt) noexcept;
    DXTEXB200_API bool IsCompressed(DXGI_FORMAT fmt) noexcept;
    DXTEXB200_API bool IsPacked(DXGI_FORMAT fmt) noexcept;
    DXTEXB200_API bool IsVideo(DXGI_FORMAT fmt) noexcept;
    DXTEXB200_API bool IsPlanar(DXGI_FORMAT fmt, bool isd3d12 = false) noexcept;
    DXTEXB200_API bool IsPalettized(DXGI_FORMAT fmt) noexcept;
    DXTEXB200_API bool IsDepthStencil(DXGI_FORMAT fmt) noexcept;
    DXTEXB200_API bool IsSRGB(DXGI_FORMAT fmt) noexcept;
    DXTEXB200_API bool IsBGR(DXGI_FORMAT fmt) noexcept;
    DXTEXB200_API bool IsTypeless(DXGI_FORMAT fmt, bool partialTypeless = true) noexcept;
    DXTEXB200_API bool HasAlpha(DXGI_FORMAT fmt) noexcept;
    DXTEXB200_API size_t BitsPerPixel(DXGI_FORMAT fmt) noexcept;
    DXTEXB200_API size_t BitsPerColor(DXGI_FORMAT fmt) noexcept;
    enum FORMAT_TYPE : uint32_t { FORMAT_TYPE_TYPELESS, FORMAT_TYPE_FLOAT, FORMAT_TYPE_UNORM, FORMAT_TYPE_SNORM, FORMAT_TYPE_UINT, FORMAT_TYPE_SINT };
    DXTEXB200_API FORMAT_TYPE FormatDataType(DXGI_FORMAT fmt) noexcept;      // DirectXTex.h:92-102
    DXTEXB200_API size_t ComputeScanlines(DXGI_FORMAT fmt, size_t height) noexcept;
    DXTEXB200_API DXGI_FORMAT MakeSRGB(DXGI_FORMAT fmt) noexcept;
    DXTEXB200_API DXGI_FORMAT MakeLinear(DXGI_FORMAT fmt) noexcept;
    DXTEXB200_API DXGI_FORMAT MakeTypeless(DXGI_FORMAT fmt) noexcept;
    DXTEXB200_API DXGI_FORMAT MakeTypelessUNORM(DXGI_FORMAT fmt) noexcept;
    DXTEXB200_API DXGI_FORMAT MakeTypelessFLOAT(DXGI_FORMAT fmt) noexcept;

    // row-pitch rules of ComputePitch / ScratchImage::Initialize* (DirectXTex.h:104-138)
    enum CP_FLAGS : uint32_t
    {
        CP_FLAGS_NONE = 0, CP_FLAGS_LEGACY_DWORD = 0x1, CP_FLAGS_PARAGRAPH = 0x2, CP_FLAGS_YMM = 0x4, CP_FLAGS_ZMM = 0x8, CP_FLAGS_PAGE4K = 0x200,
        CP_FLAGS_BAD_DXTN_TAILS = 0x1000, CP_FLAGS_24BPP = 0x10000, CP_FLAGS_16BPP = 0x20000, CP_FLAGS_8BPP = 0x40000, CP_FLAGS_LIMIT_4GB = 0x10000000,
    };
    DXTEXB200_API HRESULT ComputePitch(DXGI_FORMAT fmt, size_t width, size_t height, size_t& rowPitch, size_t& slicePitch, CP_FLAGS flags = CP_FLAGS_NONE) noexcept;   // DirectXTex.h:141-143
    DXTEXB200_API bool CalculateMipLevels(size_t width, size_t height, size_t& mipLevels) noexcept;                                                                   // DirectXTex.h:147

    // ---- metadata (DirectXTex.h:160-216)
    enum TEX_DIMENSION : uint32_t { TEX_DIMENSION_TEXTURE1D = 2, TEX_DIMENSION_TEXTURE2D = 3, TEX_DIMENSION_TEXTURE3D = 4 };

    struct DXTEXB200_API TexMetadata
    {
        size_t width, height, depth, arraySize, mipLevels;
        uint32_t miscFlags, miscFlags2;
        DXGI_FORMAT format;
        TEX_DIMENSION dimension;
        size_t ComputeIndex(size_t mip, size_t item, size_t slice) const noexcept;     // DirectXTexUtil.cpp:1695-1741 (2D only)
        bool IsCubemap() const noexcept { return (miscFlags & 0x4u) != 0; }            // TEX_MISC_TEXTURECUBE
        bool IsVolumemap() const noexcept { return dimension == TEX_DIMENSION_TEXTURE3D; }
        // alpha mode lives in the low 3 bits of miscFlags2 (TEX_MISC2_ALPHA_MODE_MASK, DirectXTex.h:169-185, 214-216)
        bool IsPMAlpha() const noexcept { return (miscFlags2 & 0x7u) == 2u; }
        void SetAlphaMode(uint32_t mode) noexcept { miscFlags2 = (miscFlags2 & ~0x7u) | (mode & 0x7u); }
        uint32_t GetAlphaMode() const noexcept { return miscFlags2 & 0x7u; }
        // D3D subresource index: mip + item * mipLevels (+ plane * mipLevels * arraySize); uint32_t(-1) when out of range (DirectXTexUtil.cpp:1744-1807)
        uint32_t CalculateSubresource(size_t mip, size_t item) const noexcept { return CalculateSubresource(mip, item, 0); }
        uint32_t CalculateSubresource(size_t mip, size_t item, size_t plane) const noexcept
        {
            if (mip >= mipLevels) return uint32_t(-1);
            if (dimension == TEX_DIMENSION_TEXTURE3D) return (item == 0) ? static_cast<uint32_t>(mip + plane * mipLevels) : uint32_t(-1);
            if (dimension != TEX_DIMENSION_TEXTURE1D && dimension != TEX_DIMENSION_TEXTURE2D) return uint32_t(-1);
            return (item < arraySize) ? static_cast<uint32_t>(mip + item * mipLevels + plane * mipLevels * arraySize) : uint32_t(-1);
        }
    };
    enum TEX_MISC_FLAG : uint32_t { TEX_MISC_TEXTURECUBE = 0x4 };
    enum TEX_MISC_FLAG2 : uint32_t { TEX_MISC2_ALPHA_MODE_MASK = 0x7 };
    enum TEX_ALPHA_MODE : uint32_t { TEX_ALPHA_MODE_UNKNOWN = 0, TEX_ALPHA_MODE_STRAIGHT = 1, TEX_ALPHA_MODE_PREMULTIPLIED = 2, TEX_ALPHA_MODE_OPAQUE = 3, TEX_ALPHA_MODE_CUSTOM = 4 };

    // ---- flags (DirectXTex.h:741-797, 887-917)
    enum TEX_FILTER_FLAGS : uint32_t
    {
        TEX_FILTER_DEFAULT = 0,
        TEX_FILTER_WRAP_U = 0x1, TEX_FILTER_WRAP_V = 0x2, TEX_FILTER_WRAP_W = 0x4, TEX_FILTER_WRAP = 0x7,
        TEX_FILTER_MIRROR_U = 0x10, TEX_FILTER_MIRROR_V = 0x20, TEX_FILTER_MIRROR_W = 0x40, TEX_FILTER_MIRROR = 0x70,
        TEX_FILTER_SEPARATE_ALPHA = 0x100, TEX_FILTER_FLOAT_X2BIAS = 0x200,
        TEX_FILTER_RGB_COPY_RED = 0x1000, TEX_FILTER_RGB_COPY_GREEN = 0x2000, TEX_FILTER_RGB_COPY_BLUE = 0x4000, TEX_FILTER_RGB_COPY_ALPHA = 0x8000,
        TEX_FILTER_DITHER = 0x10000, TEX_FILTER_DITHER_DIFFUSION = 0x20000,
        TEX_FILTER_POINT = 0x100000, TEX_FILTER_LINEAR = 0x200000, TEX_FILTER_CUBIC = 0x300000, TEX_FILTER_BOX = 0x400000,
        TEX_FILTER_FANT = 0x400000, TEX_FILTER_TRIANGLE = 0x500000,
        TEX_FILTER_SRGB_IN = 0x1000000, TEX_FILTER_SRGB_OUT = 0x2000000, TEX_FILTER_SRGB = 0x3000000,
        TEX_FILTER_FORCE_NON_WIC = 0x10000000, TEX_FILTER_FORCE_WIC = 0x20000000,      // accepted and ignored: there is no WIC path here
    };
    // DirectXTex.h:864-879
    enum TEX_PMALPHA_FLAGS : uint32_t
    {
        TEX_PMALPHA_DEFAULT = 0, TEX_PMALPHA_IGNORE_SRGB = 0x1, TEX_PMALPHA_REVERSE = 0x2,
        TEX_PMALPHA_SRGB_IN = 0x1000000, TEX_PMALPHA_SRGB_OUT = 0x2000000, TEX_PMALPHA_SRGB = 0x3000000,
    };
    enum TEX_COMPRESS_FLAGS : uint32_t
    {
        TEX_COMPRESS_DEFAULT = 0,
        TEX_COMPRESS_RGB_DITHER = 0x10000, TEX_COMPRESS_A_DITHER = 0x20000, TEX_COMPRESS_DITHER = 0x30000,
        TEX_COMPRESS_UNIFORM = 0x40000, TEX_COMPRESS_BC7_USE_3SUBSETS = 0x80000, TEX_COMPRESS_BC7_QUICK = 0x100000,
        TEX_COMPRESS_SRGB_IN = 0x1000000, TEX_COMPRESS_SRGB_OUT = 0x2000000, TEX_COMPRESS_SRGB = 0x3000000,
        TEX_COMPRESS_PARALLEL = 0x10000000,
    };
    constexpr TEX_FILTER_FLAGS operator|(TEX_FILTER_FLAGS a, TEX_FILTER_FLAGS b) noexcept { return static_cast<TEX_FILTER_FLAGS>(static_cast<uint32_t>(a) | static_cast<uint32_t>(b)); }
    constexpr TEX_COMPRESS_FLAGS operator|(TEX_COMPRESS_FLAGS a, TEX_COMPRESS_FLAGS b) noexcept { return static_cast<TEX_COMPRESS_FLAGS>(static_cast<uint32_t>(a) | static_cast<uint32_t>(b)); }

    constexpr float TEX_THRESHOLD_DEFAULT = 0.5f;
    constexpr float TEX_ALPHA_WEIGHT_DEFAULT = 1.0f;

    struct ConvertOptions { TEX_FILTER_FLAGS filter; float threshold; };
    struct CompressOptions { TEX_COMPRESS_FLAGS flags; float threshold; float alphaWeight; };

    // ---- bitmap container (DirectXTex.h:437-498): same members, same layout, same ownership
    struct Image
    {
        size_t width, height;
        DXGI_FORMAT format;
        size_t rowPitch, slicePitch;
        uint8_t* pixels;
    };

    class DXTEXB200_API ScratchImage
    {
    public:
        ScratchImage() noexcept : m_nimages(0), m_size(0), m_metadata{}, m_image(nullptr), m_memory(nullptr) {}
        ScratchImage(ScratchImage&& moveFrom) noexcept : ScratchImage() { *this = static_cast<ScratchImage&&>(moveFrom); }
        ~ScratchImage() { Release(); }
        ScratchImage& operator=(ScratchImage&& moveFrom) noexcept;
        ScratchImage(const ScratchImage&) = delete;
        ScratchImage& operator=(const ScratchImage&) = delete;

        HRESULT Initialize(const TexMetadata& mdata, CP_FLAGS flags = CP_FLAGS_NONE) noexcept;
        HRESULT Initialize1D(DXGI_FORMAT fmt, size_t length, size_t arraySize, size_t mipLevels, CP_FLAGS flags = CP_FLAGS_NONE) noexcept;
        HRESULT Initialize2D(DXGI_FORMAT fmt, size_t width, size_t height, size_t arraySize, size_t mipLevels, CP_FLAGS flags = CP_FLAGS_NONE) noexcept;
        HRESULT InitializeCube(DXGI_FORMAT fmt, size_t width, size_t height, size_t nCubes, size_t mipLevels, CP_FLAGS flags = CP_FLAGS_NONE) noexcept;
        HRESULT InitializeFromImage(const Image& srcImage, bool allow1D = false, CP_FLAGS flags = CP_FLAGS_NONE) noexcept;
        HRESULT InitializeArrayFromImages(const Image* images, size_t nImages, bool allow1D = false, CP_FLAGS flags = CP_FLAGS_NONE) noexcept;
        HRESULT InitializeCubeFromImages(const Image* images, size_t nImages, CP_FLAGS flags = CP_FLAGS_NONE) noexcept;
        void Release() noexcept;
        bool OverrideFormat(DXGI_FORMAT f) noexcept;

        const TexMetadata& GetMetadata() const noexcept { return m_metadata; }
        const Image* GetImage(size_t mip, size_t item, size_t slice) const noexcept;
        const Image* GetImages() const noexcept { return m_image; }
        size_t GetImageCount() const noexcept { return m_nimages; }
        uint8_t* GetPixels() const noexcept { return m_memory; }
        size_t GetPixelsSize() const noexcept { return m_size; }
        // DirectXTexImage.cpp:800-852: false without images, true for formats without alpha, else the scan of every image on the
        // device (dxb200_is_alpha_all_opaque); false on any failure, the reference's failure value
        bool IsAlphaAllOpaque() const noexcept;

    private:
        size_t m_nimages, m_size;
        TexMetadata m_metadata;
        Image* m_image;
        uint8_t* m_memory;
    };

    // ---- DDS container (DirectXTex.h:232-279 DDS_FLAGS, :425-435 Blob, :518-560 the DDS I/O functions); host-side only
    enum DDS_FLAGS : uint32_t
    {
        DDS_FLAGS_NONE = 0, DDS_FLAGS_LEGACY_DWORD = 0x1, DDS_FLAGS_NO_LEGACY_EXPANSION = 0x2, DDS_FLAGS_NO_R10B10G10A2_FIXUP = 0x4, DDS_FLAGS_FORCE_RGB = 0x8,
        DDS_FLAGS_NO_16BPP = 0x10, DDS_FLAGS_EXPAND_LUMINANCE = 0x20, DDS_FLAGS_BAD_DXTN_TAILS = 0x40, DDS_FLAGS_PERMISSIVE = 0x80, DDS_FLAGS_IGNORE_MIPS = 0x100,
        DDS_FLAGS_FORCE_DX10_EXT = 0x10000, DDS_FLAGS_FORCE_DX10_EXT_MISC2 = 0x20000, DDS_FLAGS_FORCE_DX9_LEGACY = 0x40000,
        DDS_FLAGS_FORCE_DXT5_RXGB = 0x80000, DDS_FLAGS_FORCE_24BPP_RGB = 0x100000, DDS_FLAGS_ALLOW_LARGE_FILES = 0x1000000,
    };
    class DXTEXB200_API Blob
    {
    public:
        Blob() noexcept : m_buffer(nullptr), m_size(0) {}
        Blob(Blob&& o) noexcept : m_buffer(o.m_buffer), m_size(o.m_size) { o.m_buffer = nullptr; o.m_size = 0; }
        Blob& operator=(Blob&& o) noexcept;
        Blob(const Blob&) = delete;
        Blob& operator=(const Blob&) = delete;
        ~Blob() { Release(); }
        HRESULT Initialize(size_t size) noexcept;
        void Release() noexcept;
        uint8_t* GetBufferPointer() const noexcept { return m_buffer; }
        const uint8_t* GetConstBufferPointer() const noexcept { return m_buffer; }
        size_t GetBufferSize() const noexcept { return m_size; }
    private:
        uint8_t* m_buffer; size_t m_size;
    };
    DXTEXB200_API HRESULT GetMetadataFromDDSMemory(const uint8_t* pSource, size_t size, DDS_FLAGS flags, TexMetadata& metadata) noexcept;
    DXTEXB200_API HRESULT GetMetadataFromDDSFile(const char* szFile, DDS_FLAGS flags, TexMetadata& metadata) noexcept;
    DXTEXB200_API HRESULT LoadFromDDSMemory(const uint8_t* pSource, size_t size, DDS_FLAGS flags, TexMetadata* metadata, ScratchImage& image) noexcept;
    DXTEXB200_API HRESULT LoadFromDDSFile(const char* szFile, DDS_FLAGS flags, TexMetadata* metadata, ScratchImage& image) noexcept;
    DXTEXB200_API HRESULT SaveToDDSMemory(const Image& image, DDS_FLAGS flags, Blob& blob) noexcept;
    DXTEXB200_API HRESULT SaveToDDSMemory(const Image* images, size_t nimages, const TexMetadata& metadata, DDS_FLAGS flags, Blob& blob) noexcept;
    DXTEXB200_API HRESULT SaveToDDSFile(const Image& image, DDS_FLAGS flags, const char* szFile) noexcept;
    DXTEXB200_API HRESULT SaveToDDSFile(const Image* images, size_t nimages, const TexMetadata& metadata, DDS_FLAGS flags, const char* szFile) noexcept;
    // the reference's own signatures (DirectXTex.h:588-616): wchar_t paths, converted to UTF-8
    DXTEXB200_API HRESULT GetMetadataFromDDSFile(const wchar_t* szFile, DDS_FLAGS flags, TexMetadata& metadata) noexcept;
    DXTEXB200_API HRESULT LoadFromDDSFile(const wchar_t* szFile, DDS_FLAGS flags, TexMetadata* metadata, ScratchImage& image) noexcept;
    DXTEXB200_API HRESULT SaveToDDSFile(const Image& image, DDS_FLAGS flags, const wchar_t* szFile) noexcept;
    DXTEXB200_API HRESULT SaveToDDSFile(const Image* images, size_t nimages, const TexMetadata& metadata, DDS_FLAGS flags, const wchar_t* szFile) noexcept;

    // ---- the accelerated operations: same signatures as DirectXTex.h:818-832, 841-846, 929-944, 965-968
    DXTEXB200_API HRESULT Convert(const Image& srcImage, DXGI_FORMAT format, TEX_FILTER_FLAGS filter, float threshold, ScratchImage& image) noexcept;
    DXTEXB200_API HRESULT Convert(const Image* srcImages, size_t nimages, const TexMetadata& metadata, DXGI_FORMAT format, TEX_FILTER_FLAGS filter, float threshold, ScratchImage& result) noexcept;
    DXTEXB200_API HRESULT ConvertEx(const Image& srcImage, DXGI_FORMAT format, const ConvertOptions& options, ScratchImage& image, std::function<bool(size_t, size_t)> statusCallBack = nullptr);
    DXTEXB200_API HRESULT ConvertEx(const Image* srcImages, size_t nimages, const TexMetadata& metadata, DXGI_FORMAT format, const ConvertOptions& options, ScratchImage& result, std::function<bool(size_t, size_t)> statusCallBack = nullptr);

    DXTEXB200_API HRESULT GenerateMipMaps(const Image& baseImage, TEX_FILTER_FLAGS filter, size_t levels, ScratchImage& mipChain, bool allow1D = false) noexcept;
    DXTEXB200_API HRESULT GenerateMipMaps(const Image* srcImages, size_t nimages, const TexMetadata& metadata, TEX_FILTER_FLAGS filter, size_t levels, ScratchImage& mipChain);

    // DirectXTex.h:800-806 (Resize)
    DXTEXB200_API HRESULT Resize(const Image& srcImage, size_t width, size_t height, TEX_FILTER_FLAGS filter, ScratchImage& image) noexcept;
    DXTEXB200_API HRESULT Resize(const Image* srcImages, size_t nimages, const TexMetadata& metadata, size_t width, size_t height, TEX_FILTER_FLAGS filter, ScratchImage& result) noexcept;

    // DirectXTex.h:848-851 (ScaleMipMapsAlphaForCoverage)
    DXTEXB200_API HRESULT ScaleMipMapsAlphaForCoverage(const Image* srcImages, size_t nimages, const TexMetadata& metadata, size_t item, float alphaReference, ScratchImage& mipChain) noexcept;

    // DirectXTex.h:881-885 (PremultiplyAlpha)
    DXTEXB200_API HRESULT PremultiplyAlpha(const Image& srcImage, TEX_PMALPHA_FLAGS flags, ScratchImage& image) noexcept;
    DXTEXB200_API HRESULT PremultiplyAlpha(const Image* srcImages, size_t nimages, const TexMetadata& metadata, TEX_PMALPHA_FLAGS flags, ScratchImage& result) noexcept;

    DXTEXB200_API HRESULT Compress(const Image& srcImage, DXGI_FORMAT format, TEX_COMPRESS_FLAGS compress, float threshold, ScratchImage& cImage) noexcept;
    DXTEXB200_API HRESULT Compress(const Image* srcImages, size_t nimages, const TexMetadata& metadata, DXGI_FORMAT format, TEX_COMPRESS_FLAGS compress, float threshold, ScratchImage& cImages) noexcept;
    DXTEXB200_API HRESULT CompressEx(const Image& srcImage, DXGI_FORMAT format, const CompressOptions& options, ScratchImage& cImage, std::function<bool(size_t, size_t)> statusCallBack = nullptr);
    DXTEXB200_API HRESULT CompressEx(const Image* srcImages, size_t nimages, const TexMetadata& metadata, DXGI_FORMAT format, const CompressOptions& options, ScratchImage& cImages, std::function<bool(size_t, size_t)> statusCallBack = nullptr);

    // DirectXTex.h:1022-1041 (ComputeMSE): mseV within 4 fp32 ulp of the exact mean of the reference's per-pixel squares, see
    // include/dxtex_b200.h (dxb200_compute_mse)
    enum CMSE_FLAGS : uint32_t
    {
        CMSE_DEFAULT = 0,
        CMSE_IMAGE1_SRGB = 0x1, CMSE_IMAGE2_SRGB = 0x2,
        CMSE_IGNORE_RED = 0x10, CMSE_IGNORE_GREEN = 0x20, CMSE_IGNORE_BLUE = 0x40, CMSE_IGNORE_ALPHA = 0x80,
        CMSE_IMAGE1_X2_BIAS = 0x100, CMSE_IMAGE2_X2_BIAS = 0x200,
    };
    constexpr CMSE_FLAGS operator|(CMSE_FLAGS a, CMSE_FLAGS b) noexcept { return static_cast<CMSE_FLAGS>(static_cast<uint32_t>(a) | static_cast<uint32_t>(b)); }
    DXTEXB200_API HRESULT ComputeMSE(const Image& image1, const Image& image2, float& mse, float* mseV, CMSE_FLAGS flags = CMSE_DEFAULT) noexcept;

    DXTEXB200_API HRESULT Decompress(const Image& cImage, DXGI_FORMAT format, ScratchImage& image) noexcept;
    DXTEXB200_API HRESULT Decompress(const Image* cImages, size_t nimages, const TexMetadata& metadata, DXGI_FORMAT format, ScratchImage& images) noexcept;
}
