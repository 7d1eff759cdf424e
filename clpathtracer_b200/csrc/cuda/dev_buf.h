// dev_buf.h -- a device array with the library's two growth policies (internal).
#pragma once

#include <cuda_runtime.h>
#include <stddef.h>

#include "CLHandler.h"

// Bumped by every (re)allocation of any DevBuf.  A recorded CUDA graph holds raw pointers, so
// whoever replays one keeps this count in the graph's key and records again when it changed.
inline size_t clpt_devbuf_reallocations = 0;

template <typename T>
struct DevBuf {
    T *ptr = nullptr;
    size_t count = 0, capacity = 0;

    void release() {
        if (ptr) HANDLE_ERR(cudaFree(ptr));
        ptr = nullptr;
        count = capacity = 0;
    }
    // The reference frees and re-creates every buffer at its exact size on each
    // upload (resize_buffer, src/CLState.c:92-102).  cudaFree/cudaMalloc cost a
    // device synchronisation each, which dominates re-uploads of an animated scene,
    // so the allocation is kept while it is big enough and not more than 2x too big.
    void resize(size_t n) {
        if (n > capacity || n * 2 < capacity) reallocate(n);
        count = n;
    }
    // Grow-only, with a quarter of headroom: buffers whose size follows the scene (the
    // traversal layout, the device builder's workspace), which an animated scene re-sizes
    // every frame by a little either way.
    void reserve(size_t n) {
        if (n > capacity) reallocate(n + n / 4 + 1024);
        count = n;
    }
    // reserve(n), keeping the first `keep` elements.
    void grow_keep(size_t n, size_t keep, cudaStream_t s) {
        if (n > capacity) {
            DevBuf old = *this;
            ptr = nullptr;
            capacity = 0;
            reserve(n);
            if (keep) {
                HANDLE_ERR(cudaMemcpyAsync(ptr, old.ptr, keep * sizeof(T), cudaMemcpyDeviceToDevice, s));
                HANDLE_ERR(cudaStreamSynchronize(s));
            }
            old.release();
        }
        count = n;
    }
    void upload(const T *src, size_t n, cudaStream_t s) {
        resize(n);
        if (n) {
            HANDLE_ERR(cudaMemcpyAsync(ptr, src, n * sizeof(T), cudaMemcpyHostToDevice, s));
            HANDLE_ERR(cudaStreamSynchronize(s));
        }
    }

  private:
    void reallocate(size_t n) {
        release();
        if (n) {
            HANDLE_ERR(cudaMalloc((void **)&ptr, n * sizeof(T)));
            clpt_devbuf_reallocations++;
        }
        capacity = n;
    }
};
