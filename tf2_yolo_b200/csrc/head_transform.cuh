// The head transform of the v3/v4 models (yolov4/models/__init__.py:42-60, yolov3/models/__init__.py:36-63):
// sigmoid on x, y, objectness and the class scores, anchor * exp on w, h.  This is the one definition of
// "the activation of a raw head": the from-logits instances of the loss kernel and yb_activate_head both
// call it, and both are compiled in loss.cu under the same flags, so a raw head decoded inside the
// train-and-evaluate step and the same head activated on the device give the same float32 bits.
#pragma once

namespace yb {

__device__ __forceinline__ float sigmoidf_(float z) { return 1.f / (1.f + expf(-z)); }

// value j of a box's [x, y, w, h, c, p_0 .. p_{C-1}]; a = the box's anchor side for j = 2 (w) / 3 (h)
__device__ __forceinline__ float head_act(float v, int j, float a) {
    return (j == 2 || j == 3) ? a * expf(v) : sigmoidf_(v);
}

}  // namespace yb
