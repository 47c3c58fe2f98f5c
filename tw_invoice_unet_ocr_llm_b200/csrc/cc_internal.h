// Entry points of components.cu that other translation units of libunetb200.so enqueue (csrc/morph.cu,
// csrc/match.cu).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

// scipy.ndimage.binary_fill_holes of every plane on the union-find of components.cu: out = in | the 4-connected
// background components that touch no border pixel.  Arguments already validated by unetb200_mask_morph (sizes as
// unetb200_mask_components, packed sides with w % 32 == 0, workspace >= unetb200_components_workspace_bytes).
// Only the first pass reads `in`, so in == out works.  Returns a UNETB200_* code (a grid too large for the batch is
// UNETB200_EINVAL, a failed launch UNETB200_ECUDA) with the message prefixed by `who`.
__attribute__((visibility("hidden"))) int cc_fill_holes(const char* who, const uint8_t* in, int in_packed,
                                                        uint8_t* out, int out_packed, int n_planes, int h, int w,
                                                        void* workspace, cudaStream_t s);

// What cc_label leaves in its workspace, per plane p: parent[p * h * w + i] encodes the component of pixel i
// (cc_pixel_id) and count[p * cap + id] is the pixel count of component id (ids 0 .. n_comps[p] - 1 in raster order
// of their first pixel, i.e. scipy.ndimage.label's labels minus one).
struct CcLabels {
    const int* parent;
    const int* count;
    int cap;              // statistics rows per plane, ceil(h * w / 2)
};

// True when cc_label accepts the batch (h, w >= 1, h * w < 2^31 and every labelling grid below 2^31 blocks).
__attribute__((visibility("hidden"))) bool cc_batch_fits(int n_planes, int h, int w);

// The labelling passes of unetb200_mask_components (pack, local, merge, flatten, scan, number, stats) without the
// selection: mask as unetb200_mask_components (packed = 1: w % 32 == 0), workspace >=
// unetb200_components_workspace_bytes and 16-byte aligned, n_comps int32 [n_planes] on the device.  Enqueued on `s`.
// Returns a UNETB200_* code as cc_fill_holes.
__attribute__((visibility("hidden"))) int cc_label(const char* who, const uint8_t* mask, int packed, int n_planes,
                                                   int h, int w, int connectivity, void* workspace, int32_t* n_comps,
                                                   cudaStream_t s, CcLabels* out);

#ifdef __CUDACC__
// Component id of pixel i of a cc_label plane (-1 = background).  Entries: -1 background, -(id + 2) the root of
// component id, otherwise the raster index of the pixel's root.
__device__ __forceinline__ int cc_pixel_id(const int* __restrict__ par, int i) {
    const int v = par[i];
    if (v == -1) return -1;
    return v < -1 ? -v - 2 : -par[v] - 2;
}
#endif
