// Driver of tests/test_results_host.py: replays drop and produce operations on s3d::Results
// (3dscan_b200/csrc/scan3d_results.h).  Each argument is "drop:NAME" or "produce:NAME"; after each operation one line
// lists the current results in enumeration order ("-" for none).
#include <stdio.h>
#include <string.h>

#include "../3dscan_b200/csrc/scan3d_results.h"

static const char* const NAMES[] = {"WRAPPED_V", "WRAPPED_H", "UNWRAPPED_V", "UNWRAPPED_H", "CPMAP", "VALID", "XYZ",
                                    "POINTS", "POINT_COLOURS", "MESH", "ACCUMULATOR", "VOXELS", "SURFACE",
                                    "COMPONENTS", "SIMPLIFIED", "SMOOTHED"};
static_assert(sizeof(NAMES) / sizeof(NAMES[0]) == s3d::RESULT_COUNT, "one name per result");

static int find(const char* name)
{
    for (int r = 0; r < s3d::RESULT_COUNT; r++)
        if (!strcmp(NAMES[r], name)) return r;
    return -1;
}

int main(int argc, char** argv)
{
    s3d::Results results;
    for (int i = 1; i < argc; i++) {
        const char* colon = strchr(argv[i], ':');
        const int r = colon ? find(colon + 1) : -1;
        if (r < 0) {
            fprintf(stderr, "bad operation %s\n", argv[i]);
            return 2;
        }
        if (!strncmp(argv[i], "drop:", 5)) results.drop((s3d::Result)r);
        else if (!strncmp(argv[i], "produce:", 8)) results.produce((s3d::Result)r);
        else {
            fprintf(stderr, "bad operation %s\n", argv[i]);
            return 2;
        }
        int any = 0;
        for (int k = 0; k < s3d::RESULT_COUNT; k++)
            if (results.has((s3d::Result)k)) printf(any++ ? " %s" : "%s", NAMES[k]);
        printf(any ? "\n" : "-\n");
    }
    return 0;
}
