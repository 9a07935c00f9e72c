// dev_mem.h -- ownership of the CUDA resources of the library's handles (host code only).
//
// Every buffer of tsar_ctx, tsar_fusion and tsar_eval only grows: cudaMalloc / cudaFree synchronise the whole device and
// would serialise contexts that pipeline views on other streams (DESIGN.md 4.4), so a call at sizes the handle has seen
// before allocates nothing.
#pragma once
#include <cuda_runtime.h>
#include <stdio.h>
#include <string.h>

#include <string>
#include <utility>

#include "../../include/tsar_b200.h"

namespace tsar {

// One allocation of device (or, with Pinned, page-locked host) memory, never zeroed.  Move-only; a move leaves the
// source empty.
template <class T, bool Pinned = false>
class DeviceBuf {
  public:
    DeviceBuf() = default;
    DeviceBuf(const DeviceBuf &) = delete;
    DeviceBuf &operator=(const DeviceBuf &) = delete;
    DeviceBuf(DeviceBuf &&o) noexcept : p_(std::exchange(o.p_, nullptr)), cap_(std::exchange(o.cap_, 0)) {}
    DeviceBuf &operator=(DeviceBuf &&o) noexcept {
        if (this != &o) {
            release();
            p_ = std::exchange(o.p_, nullptr);
            cap_ = std::exchange(o.cap_, 0);
        }
        return *this;
    }
    ~DeviceBuf() { release(); }

    // Room for n elements.  No CUDA call when they fit; otherwise the old block is freed first (the peak is the new size,
    // not old + new), and on failure the buffer is left empty.
    cudaError_t reserve(size_t n) {
        if (n <= cap_) return cudaSuccess;
        release();
        void *p = nullptr;
        const cudaError_t e = Pinned ? cudaMallocHost(&p, n * sizeof(T)) : cudaMalloc(&p, n * sizeof(T));
        if (e != cudaSuccess) return e;
        p_ = static_cast<T *>(p);
        cap_ = n;
        return cudaSuccess;
    }
    T *get() const { return p_; }
    size_t capacity() const { return cap_; }

  private:
    void release() {
        if (p_) Pinned ? cudaFreeHost(p_) : cudaFree(p_);
        p_ = nullptr;
        cap_ = 0;
    }
    T *p_ = nullptr;
    size_t cap_ = 0;
};

template <class T>
using PinnedBuf = DeviceBuf<T, true>;

// A W x H cudaArray behind a texture object with linear filtering and unnormalised coordinates.  Move-only; a move
// leaves the source empty (std::vector<Texture2D> moves its elements when it grows).
class Texture2D {
  public:
    Texture2D() = default;
    Texture2D(const Texture2D &) = delete;
    Texture2D &operator=(const Texture2D &) = delete;
    Texture2D(Texture2D &&o) noexcept : arr_(std::exchange(o.arr_, nullptr)), tex_(std::exchange(o.tex_, 0)) {}
    Texture2D &operator=(Texture2D &&o) noexcept {
        if (this != &o) {
            release();
            arr_ = std::exchange(o.arr_, nullptr);
            tex_ = std::exchange(o.tex_, 0);
        }
        return *this;
    }
    ~Texture2D() { release(); }

    cudaError_t create(int W, int H, const cudaChannelFormatDesc &cd, cudaTextureAddressMode address,
                       cudaTextureReadMode read) {
        release();
        cudaError_t e = cudaMallocArray(&arr_, &cd, W, H);
        if (e != cudaSuccess) {
            arr_ = nullptr;
            return e;
        }
        cudaResourceDesc rd;
        memset(&rd, 0, sizeof(rd));
        rd.resType = cudaResourceTypeArray;
        rd.res.array.array = arr_;
        cudaTextureDesc td;
        memset(&td, 0, sizeof(td));
        td.addressMode[0] = td.addressMode[1] = address;
        td.filterMode = cudaFilterModeLinear;
        td.readMode = read;
        td.normalizedCoords = 0;
        e = cudaCreateTextureObject(&tex_, &rd, &td, NULL);
        if (e != cudaSuccess) tex_ = 0;
        return e;
    }
    cudaArray_t array() const { return arr_; }
    cudaTextureObject_t tex() const { return tex_; }

  private:
    void release() {  // the texture object goes before the array it reads
        if (tex_) cudaDestroyTextureObject(tex_);
        if (arr_) cudaFreeArray(arr_);
        tex_ = 0;
        arr_ = nullptr;
    }
    cudaArray_t arr_ = nullptr;
    cudaTextureObject_t tex_ = 0;
};

// Device, stream and last error message of a handle (tsar_ctx, tsar_fusion, tsar_eval derive from it).  Its buffers are
// members of the derived handle, so they are freed before an owned stream is destroyed.
struct HandleCore {
    int device = 0;
    cudaStream_t stream = nullptr;
    bool own_stream = false;
    std::string err;

    HandleCore() = default;
    HandleCore(const HandleCore &) = delete;
    HandleCore &operator=(const HandleCore &) = delete;
    ~HandleCore() {
        if (own_stream) cudaStreamDestroy(stream);
    }

    // TSAR_ERR_NODEVICE (with a message on stderr) unless `dev` is an sm_100 device; then makes it current and uses
    // `user_stream`, or a new non-blocking stream of its own when that is NULL.
    int open(int dev, void *user_stream) {
        int ndev = 0;
        if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0 || dev < 0 || dev >= ndev) {
            cudaGetLastError();
            fprintf(stderr, "[tsar_b200] no usable CUDA device (requested %d of %d); this library has no CPU path\n", dev, ndev);
            return TSAR_ERR_NODEVICE;
        }
        cudaDeviceProp prop;
        if (cudaGetDeviceProperties(&prop, dev) != cudaSuccess || prop.major != 10) {
            fprintf(stderr, "[tsar_b200] device %d is sm_%d%d; this build contains sm_100a code only\n", dev, prop.major, prop.minor);
            return TSAR_ERR_NODEVICE;
        }
        device = dev;
        if (cudaSetDevice(dev) != cudaSuccess) return TSAR_ERR_CUDA;
        if (user_stream) {
            stream = (cudaStream_t)user_stream;
            return TSAR_OK;
        }
        if (cudaStreamCreateWithFlags(&stream, cudaStreamNonBlocking) != cudaSuccess) return TSAR_ERR_CUDA;
        own_stream = true;
        return TSAR_OK;
    }

    // Records "file:line call: error" and clears the runtime's last error, so that it does not surface in a later call
    // that itself succeeded.
    int cuda_failed(cudaError_t e, const char *file, int line, const char *call) {
        char buf[512];
        snprintf(buf, sizeof(buf), "%s:%d %s: %s", file, line, call, cudaGetErrorString(e));
        err = buf;
        cudaGetLastError();
        return e == cudaErrorMemoryAllocation ? TSAR_ERR_NOMEM : TSAR_ERR_CUDA;
    }
};

}  // namespace tsar

#define TSAR_CK(handle, call)                                                          \
    do {                                                                               \
        const cudaError_t e_ = (call);                                                 \
        if (e_ != cudaSuccess) return (handle)->cuda_failed(e_, __FILE__, __LINE__, #call); \
    } while (0)

#define TSAR_FAIL(handle, code, msg) \
    do {                             \
        (handle)->err = (msg);       \
        return (code);               \
    } while (0)
