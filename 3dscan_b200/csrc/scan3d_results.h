// scan3d_results.h -- which of a context's results are current (host only, no CUDA include).
//
// When a result is recomputed, every result computed from it is stale.  INPUTS below is the one place that says what
// is computed from what.  Every entry of the C ABI checks the results it requires with has(), drops the results it
// will overwrite before its first allocation or launch, and produces what it made after its last launch succeeds.
#pragma once
#include <stdint.h>

namespace s3d {

// Enumerated so that every result comes after its inputs.
enum Result : int {
    WRAPPED_V, WRAPPED_H,          // the direction's wrapped phase and mask
    UNWRAPPED_V, UNWRAPPED_H,      // the direction's unwrapped phase and code planes
    CPMAP, VALID, XYZ,
    POINTS,                        // the compacted points and their count
    POINT_COLOURS,                 // the points' colours from the texture set when they were computed
    MESH,                          // the camera-grid mesh of the points and its point normals
    ACCUMULATOR,                   // a voxel begin has run
    VOXELS,                        // the finish outputs of the adds since begin
    SURFACE,                       // the held voxel surface
    COMPONENTS,                    // the component table of the held surface
    SIMPLIFIED, SMOOTHED,          // the held surface has been simplified / smoothed
    RESULT_COUNT
};

constexpr uint32_t bit(Result r) { return 1u << r; }

// the direct inputs of each result
constexpr uint32_t INPUTS[RESULT_COUNT] = {
    /* WRAPPED_V     */ 0,
    /* WRAPPED_H     */ 0,
    /* UNWRAPPED_V   */ bit(WRAPPED_V),
    /* UNWRAPPED_H   */ bit(WRAPPED_H),
    /* CPMAP         */ bit(UNWRAPPED_V) | bit(UNWRAPPED_H),
    /* VALID         */ bit(UNWRAPPED_V) | bit(UNWRAPPED_H),
    /* XYZ           */ bit(CPMAP) | bit(VALID),
    /* POINTS        */ bit(XYZ),
    /* POINT_COLOURS */ bit(POINTS),
    /* MESH          */ bit(POINTS),
    /* ACCUMULATOR   */ 0,
    /* VOXELS        */ bit(ACCUMULATOR),
    /* SURFACE       */ bit(VOXELS),
    /* COMPONENTS    */ bit(SURFACE),
    /* SIMPLIFIED    */ bit(SURFACE),
    /* SMOOTHED      */ bit(SURFACE),
};

// DOWNSTREAM.of[r]: every result computed from r, directly or through others.  One pass in enumeration order is
// enough because every result comes after its inputs.
struct Downstream {
    uint32_t of[RESULT_COUNT];
};
constexpr Downstream downstream()
{
    Downstream d{};
    for (int r = 0; r < RESULT_COUNT; r++) {
        uint32_t from_r = bit((Result)r);
        for (int s = r + 1; s < RESULT_COUNT; s++)
            if (INPUTS[s] & from_r) from_r |= bit((Result)s);
        d.of[r] = from_r & ~bit((Result)r);
    }
    return d;
}
constexpr bool inputs_come_first()
{
    for (int s = 0; s < RESULT_COUNT; s++)
        if (INPUTS[s] >> s) return false;
    return true;
}
static_assert(inputs_come_first(), "a result must come after its inputs in enum Result");
constexpr Downstream DOWNSTREAM = downstream();

// the set of current results; a new context has none
class Results {
  public:
    bool has(Result r) const { return (bits_ & bit(r)) != 0; }
    // r and everything computed from it are no longer current
    void drop(Result r) { bits_ &= ~(bit(r) | DOWNSTREAM.of[r]); }
    // r was just computed: what was computed from the old r is stale
    void produce(Result r) { bits_ = (bits_ & ~DOWNSTREAM.of[r]) | bit(r); }

  private:
    uint32_t bits_ = 0;
};

}  // namespace s3d
