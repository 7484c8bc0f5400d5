// Tuning / debugging switches of libibo_b200 and the scoring paths a caller can force (host-only header: shared by the CUDA
// sources and the host DIRECT driver).
#pragma once

namespace ibo {

// Tuning / debugging switches.  Each has a default, may be preset from the environment variable IBO_<NAME> when the library
// is loaded, and is read and written through the C ABI (ibo_set_option / ibo_get_option) -- nothing in a launch path calls getenv.
enum {
    OPT_INT8 = 0,        // 1 (default): wide batches take the INT8 tensor-core path; 0: FP64 DMMA everywhere
    OPT_I8_PIPE,         // 1: K1 of chunk c+1 on a second (low-priority) stream under K2 of chunk c
    OPT_CHUNK_TILES,     // candidate tiles per chunk (0: 2 x SMs)
    OPT_NARROW_MAX,      // batches up to this many candidates use K2's latency shapes
    OPT_NARROW_MT,       // force the latency shape (0: cost model)
    OPT_K2_DEEP,         // -1 auto, 0 never, 1 always: deep-pipeline variant of the latency shapes
    OPT_PDL,             // programmatic dependent launch for small batches
    OPT_KSTAR_DIRECT,    // 1: K1 from direct differences instead of the DMMA expansion
    OPT_DEBUG_PLAN,      // print the latency-shape plan and the instance of every FP64 K2 launch
    OPT_TINY,            // -1 auto, 0 never, 1 force: fused small-model kernel
    OPT_DIRECT_TIMING,   // print the host/GPU split of a DIRECT query
    OPT_SHARD_MIN,       // sharded DIRECT: batches below this many points stay on every rank (0: 64 x ranks)
    OPT_I8_GUARD,        // 1 (default): candidates with sigma^2 < 2^-10 on the INT8 path are re-scored by the DMMA kernels
    OPT_I8_MIN_BATCH,    // batches of at least this many candidates (and at most narrow_max) also take the INT8 path (-1: measured break-even rule, 0: only wide batches)
    OPT_I8_RB_PER_CTA,   // row-blocks a CTA of the INT8 K2 sweeps (G = nb / this many CTAs share a candidate tile); 0: four groups whatever the size
    OPT_CHOL_PAIR,       // model build: block columns in pairs (256-deep trailing updates); -1 = from 48 block columns on, 0 / 1 forced
    OPT_TINY_SERVER,     // DIRECT on a one-row-block model: resident kernel fed through a mailbox in mapped host memory (1) or one launch per batch (0)
    OPT_COUNT
};
long get_option(int id);

// A scoring path a caller imposes on a batch whatever its size (score.cu, plan_score): the guard pass re-scores its candidates with
// K2's throughput shape, and a sharded DIRECT slice takes the INT8 path when the whole batch does.
enum class ScoreForce { None, Fp64Wide, I8 };

}  // namespace ibo
