// Entry point of components.cu that another translation unit of libunetb200.so enqueues (csrc/morph.cu).
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
