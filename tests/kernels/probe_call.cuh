// probe_call.cuh -- the host side shared by the test-only kernel probes (contract_probe.cu, linalg_probe.cu).
//
// A Call owns the device buffers and the private stream of one probe call and releases them in its destructor, whatever
// path the call leaves by.  Buffers from guarded() sit between two sentinel regions of GUARD_BYTES; finish() checks them
// once the stream has drained, so a kernel that writes past either end of a buffer fails the call (-2, probe_last_error
// names the buffer) instead of corrupting a neighbour silently.
#pragma once
#include <cuda_runtime.h>

#include <cstring>
#include <string>
#include <vector>

namespace probe {

inline std::string &last_error()
{
    static std::string e;
    return e;
}

constexpr size_t GUARD_BYTES = 256;                 // keeps the guarded buffer itself 256-byte aligned
constexpr unsigned char GUARD_BYTE = 0xA5;

struct Call {
    struct Guarded { const unsigned char *base; size_t bytes; const char *name; };
    cudaStream_t stream = nullptr;
    std::vector<void *> bufs;
    std::vector<Guarded> guards;
    cudaError_t err = cudaSuccess;
    Call() { note(cudaStreamCreateWithFlags(&stream, cudaStreamNonBlocking)); }
    ~Call()
    {
        if (stream) cudaStreamSynchronize(stream);
        for (void *p : bufs) cudaFree(p);
        if (stream) cudaStreamDestroy(stream);
    }
    Call(const Call &) = delete;
    Call &operator=(const Call &) = delete;
    bool note(cudaError_t e)
    {
        if (e != cudaSuccess && err == cudaSuccess) { err = e; last_error() = cudaGetErrorString(e); }
        return err == cudaSuccess;
    }
    template <class T>
    T *alloc(size_t n)
    {
        void *p = nullptr;
        if (!note(cudaMalloc(&p, n * sizeof(T) + 16))) return nullptr;
        bufs.push_back(p);
        note(cudaMemsetAsync(p, 0, n * sizeof(T) + 16, stream));
        return static_cast<T *>(p);
    }
    // n elements, every byte set to `fill` (0xFF: NaN doubles, -1 ints), between two guard regions
    template <class T>
    T *guarded(size_t n, const char *name, unsigned char fill = 0xFF)
    {
        const size_t bytes = n * sizeof(T);
        void *p = nullptr;
        if (!note(cudaMalloc(&p, bytes + 2 * GUARD_BYTES))) return nullptr;
        bufs.push_back(p);
        unsigned char *b = static_cast<unsigned char *>(p);
        note(cudaMemsetAsync(b, GUARD_BYTE, GUARD_BYTES, stream));
        note(cudaMemsetAsync(b + GUARD_BYTES, fill, bytes, stream));
        note(cudaMemsetAsync(b + GUARD_BYTES + bytes, GUARD_BYTE, GUARD_BYTES, stream));
        guards.push_back({b, bytes, name});
        return reinterpret_cast<T *>(b + GUARD_BYTES);
    }
    template <class T>
    T *upload(const T *h, size_t n)
    {
        T *d = alloc<T>(n);
        if (d && h && n) note(cudaMemcpyAsync(d, h, n * sizeof(T), cudaMemcpyHostToDevice, stream));
        return d;
    }
    template <class T>
    T *upload_guarded(const T *h, size_t n, const char *name)
    {
        T *d = guarded<T>(n, name);
        if (d && h && n) note(cudaMemcpyAsync(d, h, n * sizeof(T), cudaMemcpyHostToDevice, stream));
        return d;
    }
    template <class T>
    void download(T *h, const T *d, size_t n)
    {
        if (h && d && n && err == cudaSuccess) note(cudaMemcpyAsync(h, d, n * sizeof(T), cudaMemcpyDeviceToHost, stream));
    }
    // 0, a positive cudaError_t, or -2 when a kernel wrote into a guard region
    int finish()
    {
        if (err == cudaSuccess) note(cudaGetLastError());
        if (err == cudaSuccess) note(cudaStreamSynchronize(stream));
        if (err != cudaSuccess) return (int)err;
        std::vector<unsigned char> h(2 * GUARD_BYTES);
        for (const Guarded &g : guards) {
            if (!note(cudaMemcpy(h.data(), g.base, GUARD_BYTES, cudaMemcpyDeviceToHost))) return (int)err;
            if (!note(cudaMemcpy(h.data() + GUARD_BYTES, g.base + GUARD_BYTES + g.bytes, GUARD_BYTES, cudaMemcpyDeviceToHost))) return (int)err;
            for (size_t i = 0; i < h.size(); i++)
                if (h[i] != GUARD_BYTE) {
                    last_error() = std::string("guard region overwritten: ") + g.name + (i < GUARD_BYTES ? " (before the buffer)" : " (after the buffer)");
                    return -2;
                }
        }
        return 0;
    }
};

inline int bad(const char *msg) { last_error() = msg; return -1; }

}  // namespace probe
