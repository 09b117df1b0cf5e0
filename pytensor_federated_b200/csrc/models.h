// Plain-old-data descriptors shared between the host runtime and the kernels.
#pragma once
#include <cstdint>

struct LinregShard {
    const void* x;        // [n] float64 or float32
    const void* y;        // [n]
    long long n;
    double sigma;
    int theta_offset;     // index (in doubles) of this shard's (intercept, slope) pair in theta
    int _pad;
};

// One contiguous block of rows of a generalised linear model ("shard" / "group").
struct GlmSegment {
    const void* X;        // [n_rows, ld] row-major; bf16 (or fp8 e4m3 for the block-scaled kernel)
    const float* y;       // [n_rows] response (0/1 for logistic)
    const void* scales;   // fp8 only: per-(row, 32-feature block) ue8m0 scales, else null
    long long n_rows;
    long long first_tile; // prefix sum over segments of ceil(n_rows / tile_rows)
    int group;            // which intercept this segment uses
    int out_group;        // which output block this segment's [LL, grads] go to (0 unless per-node outputs are kept)
};

struct GlmParams {
    int n_segments;
    int n_features;       // P
    int ld;               // row stride of X in elements
    int n_groups;         // G intercepts; theta = [intercept[G], beta[P], phi[D]] per chain
    int n_chains;         // K parameter vectors evaluated per launch (theta is [K][G+P+D])
    int family;           // 0 = logistic (Bernoulli), 1 = Poisson (log link), 2 = Gaussian (identity, unit variance);
                          // tensor-core kernel only: 3 = normal (sigma), 4 = Student-t (sigma, nu), 5 = negative binomial (alpha)
    long long total_tiles;
    int n_out;            // output blocks: 1 = everything summed; > 1 = one [K][1+G+P+D] block per node (tensor-core kernel)
    int early_loads;      // tensor-core kernels: claim + load the first tiles before theta arrives (B200FED_NO_EARLY_LOADS=1: off)
    int n_family_params;  // D fitted family parameters phi (0 for families 0-2); the result per chain is [LL, gi[G], g[P], dphi[D]]
};

// Unit of work of the dynamically scheduled tensor-core GLM kernel: n_tiles consecutive 128-row tiles of one
// segment starting at tile first_tile (n_tiles is even; the last one may lie past the segment's rows).
struct GlmChunk {
    int seg;
    int first_tile;
    int n_tiles;
    int _pad;
};

// Lotka-Volterra parameter estimation: every series i starts from its own (known) state
// y0[:, i] and is observed at the shared time grid t[0..n_t).
struct OdeShard {
    const float* t;       // [n_t] observation times (ascending, t[0] > 0; integration starts at 0)
    const float* y0;      // [2, n_series]   initial prey / predator densities
    const float* y_obs;   // [n_t, 2, n_series] noisy observations (series index fastest)
    int n_series;
    int n_t;
    float sigma;          // observation noise (Gaussian)
    int substeps;         // RK4 steps between consecutive observation times
    int theta_offset;     // first float of this shard's parameter vector in theta (per-node parameters)
    int out_offset;       // first double of this shard's [LL, dLL/dtheta] block in the result
};
