// A WINDOW of a VE plan: m consecutive binary eliminations run as ONE launch (contract_chain.cu).
//
// The window's first step reads a wide intermediate, the HEAD H, whose m fastest axes are the variables the m steps
// eliminate, in their order (the canonical layout of ve.cu: the next variable to be eliminated innermost).  For a fixed
// value r of H's other axes (the REST) the steps only ever touch the 2^m contiguous entries H[r * 2^m + t]: a thread
// keeps them in registers, runs the m sum-outs there and writes the last step's 2^n entries (n = variables the steps'
// small SIDE operands add).  Intermediates between the steps never reach memory.
//
// Register tile of level j (its step's union): bit 0 = the variable it eliminates, then the head's later tile
// variables, then the variables added by earlier levels, then its own new ones -- so the output index of level j is
// its union index >> 1 and is exactly the input index of level j + 1.
#pragma once
#include <string>

#include "contract.hpp"

namespace bnpp {

constexpr int kChainMaxLevels = 4;
constexpr int kChainMaxSides = 2;       // operands of a level besides the head (steps of up to three operands)
constexpr int kChainMaxAdd = 2;         // variables one level may add
constexpr int kChainTile = 16;          // doubles of a level's input or output tile
constexpr int kChainMaxUBits = 5;       // union bits of a level: log2(2 * kChainTile)
constexpr int kChainMaxFields = 16;
constexpr uint32_t kChainDefaultDepth = 4;  // levels of a window unless bnpp_tuning_set("chain_depth") says otherwise

// rest items a CTA takes per chunk: two per thread when the head tile is 4 doubles, one for 8 or 16 (at most 16 doubles
// of head in flight per thread)
__host__ __device__ constexpr uint32_t chain_chunk_items(int m) { return (m == 2 ? 2u : 1u) * kBlock; }

struct ChainSide {
    const double *p;
    uint32_t us[kChainMaxUBits];        // stride per union bit (0: the operand does not have that variable)
    uint8_t nf;
    Field f[kChainMaxFields];           // rest index -> offset
};

struct ChainLevel {
    uint8_t k;                          // sides (0 .. kChainMaxSides), in the step's operand order (the head is last)
    ChainSide s[kChainMaxSides];
};

struct ChainParams {
    const double *head;
    double *out;
    uint32_t n_items;                   // rest items = head entries >> m
    uint8_t onf;
    Field of[kChainMaxFields];          // rest index -> output offset
    uint32_t os[4];                     // output stride of new variable i, in order of addition (2^4 = kChainTile)
    ChainLevel lv[kChainMaxLevels];
};

// the kernel for m levels adding add[j] variables at level j; nullptr when the shape has no instantiation
const void *chain_kernel(int m, const int *add);
// one launch of a window's kernel `fn` on the context's stream; bnpp_last_launch reports it as `name`
int chain_launch(bnpp_ctx *ctx, const void *fn, unsigned grid, const ChainParams &p, const std::string &name);
// blocks per SM the kernel reaches with kBlock threads (0 on error)
int chain_occupancy(const void *fn);
std::string chain_name(int m, const int *add);

}  // namespace bnpp
