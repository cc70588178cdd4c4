// pndf_host.h -- host-side bookkeeping shared by pndf_capi.cu and pndf_tc.cu: the device buffers a handle owns and the layout of the
// flat parameter vector.  No device code.
#pragma once
#include <cuda_runtime.h>

#include <string>
#include <utility>

#include "../../include/pndf.h"
#include "pndf_kernel.cuh"

namespace pndf {

// records `msg` as pndf_last_error() and returns 1 (pndf_capi.cu)
int fail(const std::string& msg);

// One device allocation of `size()` elements of T, freed with its owner.  It only grows: reserve(n) replaces the buffer when n does
// not fit.  A failed grow leaves it empty (size 0), so the next call grows again instead of using a freed pointer, and it clears the
// runtime's last error so that no later call reports it as its own.
template <class T>
class DevBuf {
public:
    DevBuf() = default;
    DevBuf(DevBuf&& o) noexcept : p_(o.p_), n_(o.n_) { o.p_ = nullptr; o.n_ = 0; }
    DevBuf& operator=(DevBuf&& o) noexcept {
        std::swap(p_, o.p_);
        std::swap(n_, o.n_);
        return *this;
    }
    ~DevBuf() { cudaFree(p_); }

    T* get() const { return p_; }
    size_t size() const { return n_; }

    // make room for n elements (old contents are not kept); `zero` fills a new buffer with zero bytes
    int reserve(size_t n, const char* name, bool zero = false) {
        if (n <= n_) return 0;
        cudaFree(p_);
        p_ = nullptr;
        n_ = 0;
        const size_t bytes = n * sizeof(T);
        cudaError_t e = cudaMalloc(&p_, bytes);
        if (e == cudaSuccess && zero) e = cudaMemset(p_, 0, bytes);
        if (e != cudaSuccess) {
            cudaFree(p_);
            p_ = nullptr;
            cudaGetLastError();
            return fail(std::string("cannot allocate ") + name + " (" + std::to_string(bytes) + " bytes): " + cudaGetErrorString(e));
        }
        n_ = n;
        return 0;
    }

private:
    T* p_ = nullptr;
    size_t n_ = 0;
};

// The flat parameter vector in reference state_dict order (pndf_set_weights): [encoder] W0 b0 W1 b1 ... W6 b6, where W_l is
// [width[l + 1]][width[l]] row-major and the encoder block (kEncFloats with the structure encoder, else empty) comes first.
struct ParamLayout {
    int width[8];               // in_dim, 256, 512, 1024, 512, 256, 64, 1
    int enc_floats;
    long long w_off[7], b_off[7];
    long long total;

    explicit ParamLayout(const pndf_config& c) : width{c.in_dim, 256, 512, 1024, 512, 256, 64, 1} {
        enc_floats = c.use_enc ? kEncFloats : 0;
        long long off = enc_floats;
        for (int l = 0; l < 7; ++l) {
            w_off[l] = off; off += (long long)width[l + 1] * width[l];
            b_off[l] = off; off += width[l + 1];
        }
        total = off;
    }
};

}  // namespace pndf
