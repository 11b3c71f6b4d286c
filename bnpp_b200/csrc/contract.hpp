// A fully resolved launch of the contraction engine: kernel variant, grid and parameter block.
// Planning (axis analysis, iteration order, class selection) is done once; replaying a
// descriptor only patches the operand / output pointers -- what a VE plan does per query.
#pragma once
#include <string>

#include "common.cuh"

namespace bnpp {

constexpr int kMaxF = 24;
struct Field {
    uint32_t mask, mul, sh;
};

struct ParamsHead {
    const double *in[kMaxK];
    double *out;
    double *partials;
    unsigned int *ticket;
    double *z;
    unsigned int *status;
    uint64_t n_items;           // output entries / V
    uint32_t cx;                // cardinality of the eliminated variable (1 = none)
    uint32_t sx[kMaxK];         // operand stride of the eliminated variable
    uint32_t sl[kMaxK];         // operand stride between the V entries of an item
    uint32_t sol;               // output stride between the V entries of an item
    uint8_t cls[kMaxK];
    uint8_t out_vec;            // 16-byte store allowed
    uint8_t *arg;               // max-product steps: the first maximising x per output entry, at the output's index
};

// Mixed-radix iteration space: digits by multiply-high division, outermost axis first.
struct ParamsMR {
    ParamsHead h;
    uint32_t R;
    FastDiv div[kMaxR];
    uint32_t so[kMaxR];         // output stride per axis (per item on the innermost axis)
    uint32_t s[kMaxK][kMaxR];   // operand stride per axis
};

// Power-of-two iteration space: off = sum_f ((item >> sh) & mask) * mul, fields merged PER
// OPERAND, so an operand laid out like the output costs one field no matter how
// scattered the other operands' axes are.
struct ParamsP2 {
    ParamsHead h;
    uint8_t nf[kMaxK + 1];      // [K] is the output
    Field f[kMaxK + 1][kMaxF];
};

// One operand whose fastest axes are slow axes of the output ("transposed" layout) is not
// gathered from global memory lane by lane: each CTA chunk first copies the tile of it that
// the chunk needs into shared memory, reading along the operand's OWN fastest axes.
//   slot -> operand offset : sum_f ((slot  >> sh) & mask) * mul   over lf   (tile load)
//   item -> slot           : sum_f ((local >> sh) & mask) * mul   over cf   (consumption)
constexpr uint32_t kStagedMaxStages = 3;
constexpr uint32_t kStagedSmemBudget = 110u * 1024u;      // contract_staged_tma: two CTAs per SM
struct StageInfo {
    int32_t sk;                 // staged operand
    uint32_t tile;              // tile entries (power of two, <= 4096)
    uint32_t slot_j, slot_x;    // slot stride of the V bit and of the eliminated variable (0 = independent)
    uint32_t swz;               // bank swizzle: phys = slot ^ (((slot >> swz) & 15) << 1); the lanes differ in slot bits >= swz
    uint32_t pair;              // tile copies move 16 bytes (slots 2m, 2m+1 are neighbours in the operand)
    uint8_t nlf, ncf;
    Field lf[12], cf[12];
};
struct ParamsP2S {
    ParamsP2 b;
    StageInfo st;
};

// The same tiling with the tiles brought in by the TMA engine (contract_staged_tma).  Ranked by an operand's own
// strides, slots 0 .. 2^rbits - 1 of its tile are ONE contiguous run of it, so a tile is tile >> rbits bulk copies;
// a run sits at (its run position) * (2^rbits + 2) doubles of the stage: with the 16-byte pad and the lane-driven run
// bits lowest in the run position, the lanes of a warp that walk over runs meet two to a bank at worst.
// Any operand whose runs are 16-byte aligned and at least 64 bytes long can come this way -- the transposed one
// must, the others do when the ring of stages fits; the rest is loaded into registers chunk by chunk.
constexpr int kTmaMaxK = 3;
struct TmaOperand {
    uint32_t tile, rbits;       // slots; log2 of the run length
    uint32_t off;               // where the padded tile starts inside a stage (doubles, even)
    uint32_t dj, dx;            // padded-tile distance of the V bit and of the eliminated variable (0 = independent)
    uint8_t nlf, ncf;
    uint8_t nrb, rpos[12];      // run r of the tile sits at run position sum_i bit_i(r) << rpos[i]: the run bits the LANES drive first
    Field lf[12], cf[12];       // lf[0] is the run itself; lf[1..] place run r inside the operand
};
struct ParamsP2T {
    ParamsP2 b;
    uint32_t mask;              // operands that come through shared memory
    uint32_t stages, stage_doubles, stage_bytes;     // ring depth (2..3); doubles per stage; bytes the copies of one stage move
    TmaOperand t[kTmaMaxK];
};

// Multi-valued elimination (cardinality of the eliminated variable > 2), table driven.  A CTA owns TILES of T
// consecutive output entries = [g digits of the split axis] x [all inner axes]; the E = T * cx union entries of a
// tile are enumerated lane by lane in the order that is contiguous in the large operands (the eliminated variable
// fastest when it is their stride-1 axis), their products go to a shared-memory stage with an odd row pitch, and
// one thread per output entry adds its row up in the reference's order.  What depends on the position INSIDE a
// tile is the same for every tile and comes from a table built once by the plan (device copy `tab`, staged into
// shared memory by one bulk copy per CTA): per entry the operand offsets and the stage slot.  What depends on the
// tile is a mixed-radix decomposition of the tile index over the outer axes, done by K+1 threads per tile.
struct ParamsMV {
    ParamsHead h;               // in / out / z / partials / ticket / status, cx; n_items = output entries
    const uint32_t *tab;        // [E][KP] words: operand offsets..., (stage slot | tile-local output index << 16) in the last word
    uint32_t E, T, cxp;         // union entries and output entries of a full tile, row pitch of the stage (odd)
    uint32_t inner;             // output entries per digit of the split axis
    uint32_t g, ext_split, n_split;   // split axis: digits per tile, extent, tiles along it
    uint32_t n_tiles, R;        // R outer axes (outside the split axis), outermost first
    FastDiv dsplit;             // tile -> (outer index, chunk of the split axis); valid when n_split >= 2
    FastDiv div[kMaxR];
    uint32_t s_split[kMaxK];    // operand stride of the split axis
    uint32_t s[kMaxK][kMaxR];   // operand stride per outer axis
};

// Multi-valued elimination, TMA-staged (contract_mvt.cu): per tile every operand is ONE contiguous range brought
// into shared memory by a bulk copy; thread j owns output entry j of the tile.
constexpr int kMvtMaxStages = 6;
struct ParamsMVT {
    ParamsHead h;               // in / out / z / partials / ticket / status, cx, sx; n_items = output entries
    const uint32_t *rowtab;     // [T][K]: offset of output entry j's row inside operand k's range
    uint32_t T, inner;          // output entries per tile, output entries per digit of the split axis
    uint32_t g, ext_split, n_split;
    uint32_t n_tiles, R;
    uint32_t stages, stage_doubles, rowtab_bytes;
    uint32_t range[kMaxK];      // doubles of operand k one tile touches (a contiguous range)
    uint32_t soff[kMaxK];       // where operand k's range sits inside a stage (doubles, even)
    FastDiv dsplit;
    FastDiv div[kMaxR];
    uint32_t so[kMaxR];         // output stride per outer axis (the plan may walk the outer axes in another order)
    uint32_t s_split[kMaxK];
    uint32_t s[kMaxK][kMaxR];
};

struct LaunchDesc {
    const void *fn = nullptr;
    unsigned grid = 0;
    bool p2 = false;
    bool staged = false;
    bool mv = false;            // contract_mv: params in mvp, dynamic shared memory `smem`, device table `mv_tab`
    bool mvt = false;           // contract_mvt: params in mvtp, same ownership of `mv_tab`
    bool tma = false;           // contract_staged_tma: params in p2t, dynamic shared memory `smem`
    int k = 0;
    unsigned smem = 0;
    uint32_t *mv_tab = nullptr; // owned: freed by contract_release (stream-ordered)
    ParamsP2S p2p;              // .b is the plain power-of-two block
    ParamsP2T p2t;
    ParamsMR mrp;
    ParamsMV mvp;
    ParamsMVT mvtp;
    // pieces of the printable name (formatted lazily: a VE query launches hundreds of these)
    const char *variant = "";
    int C = 0, V = 0, U = 0;
    bool div = false, generic = false;
    bool max = false;           // max-product step: contract_canon_max / contract_generic_max
    uint32_t R = 0;
    std::string name();
    ParamsHead &head() { return tma ? p2t.b.h : (mvt ? mvtp.h : (mv ? mvp.h : (p2 ? p2p.b.h : mrp.h))); }
    void *params() { return tma ? static_cast<void *>(&p2t) : mvt ? static_cast<void *>(&mvtp) : mv ? static_cast<void *>(&mvp) : (p2 ? (staged ? static_cast<void *>(&p2p) : static_cast<void *>(&p2p.b)) : static_cast<void *>(&mrp)); }
};

// max_mode: out[o] = max_x prod_k F_k[pi_k(o, x)] and arg_dev[o] = the first x attaining it (no Z); elim_var must be
// >= 0 with at most 255 values.  The step takes contract_canon<MAX> where the sum-mode plan would take contract_canon,
// else contract_generic<MAX>.  arg_dev is fixed at planning time: contract_launch does not patch it.
int contract_plan(bnpp_ctx *ctx, int k, const bnpp_operand *ops, const bnpp_scope *out_scope, int64_t elim_var,
                  int divide, double *out_dev, double *z_dev, LaunchDesc *desc, bool max_mode = false,
                  uint8_t *arg_dev = nullptr);
// in / out / z replace the pointers the descriptor was planned with; they must be at least as
// aligned (a descriptor planned for 32-byte aligned operands may use 256-bit loads)
int contract_launch(bnpp_ctx *ctx, LaunchDesc &desc, const double *const *in, double *out, double *z);
// frees what a descriptor owns on the device (the table of a contract_mv launch); stream-ordered, idempotent
void contract_release(bnpp_ctx *ctx, LaunchDesc &desc);

}  // namespace bnpp
