// volume.cuh -- host-side state of one ScalableTSDFVolume replacement (see volume.cu).
#pragma once
#include <vector>

#include "hash_table.cuh"

namespace otslam {

constexpr int kMaxBatch = 32;   // frames fused per block residency (one bit each in the entry mask)
// integration kernel's brick cull (tests/cull_ref.py models it): max-depth tile edge in pixels, and the most tiles one
// (brick, frame) test reads; a footprint over more tiles is not tested.  Chosen by tools/study_culling_bricks.py.
constexpr int kCullTile = 4;
constexpr int kCullMaxTiles = 36;

// per-frame constants consumed by the allocation (FP64 pose) and integration (FP32 extrinsic) kernels
struct FrameDev {
    float E[12];      // rows 0..2 of extrinsic.cast<float>()           (SURVEY A.4)
    float es[3];      // (E * voxel_length).col(2): the per-z increment  (SURVEY A.4)
    int32_t key_off;  // multi-object arenas: x-key offset of the frame's object (0 for ordinary volumes)
    double pose[12];  // rows 0..2 of camera_pose = extrinsic.inverse()  (SURVEY A.3)
};
static_assert(sizeof(FrameDev) == 160, "FrameDev layout");

constexpr int kNB = 3;          // batch buffers: allocation runs up to two batches ahead of integration
// device counters: [0] pool slots handed out; per batch buffer b: [2+b] work-list length, [5+b] flags
enum CounterIdx { kPoolCount = 0, kListCount = 2, kFlags = 5, kNumCounters = 8 };
enum Flags { kFlagHashFull = 1, kFlagKeyRange = 2, kFlagBoxTooLarge = 4 };

// extraction results (extract.cu): built in a local and moved into the volume only after the stream has synchronised, so
// a failed extraction leaves an empty result
struct MeshResult {
    int64_t nv = 0, nf = 0;
    DevBuf<double> verts;     // [nv][3]
    DevBuf<double> colors;    // [nv][3]
    DevBuf<double> normals;   // [nv][3]
    DevBuf<int32_t> faces;    // [nf][3]
    DevBuf<int32_t> ekeys;    // [nv][4]
};
struct PointsResult {
    int64_t n = 0;
    DevBuf<double> pts;       // [n][3]
    DevBuf<double> cols;      // [n][3]
    DevBuf<int32_t> ekeys;    // [n][4]
};
// halo pieces packed by otslam_volume_halo_pack: grouped by destination rank, (key, kind) order inside a group
struct HaloPieces {
    int64_t n = 0;
    DevBuf<int32_t> keys;     // [n][4]
    DevBuf<uint4> planes;     // [n][256]
    std::vector<int64_t> counts;   // pieces per destination rank
};

// block hash (hash_table.cuh): the entry index is the handle used by the per-batch work list.  Built whole or not at all
// (volume.cu: new_hash).
struct BlockHash {
    uint32_t cap = 0;
    DeviceArray<uint64_t> keys;
    DeviceArray<int32_t> vals;     // entry -> pool slot
    // kNB-buffered per batch: allocation of batches b+1, b+2 runs on pre_stream while batch b integrates
    DeviceArray<uint32_t> masks[kNB];   // entry -> bit f set when frame f of the batch touches it
    DeviceArray<int32_t> list[kNB];     // entries touched by the batch (each once)
    DeviceArray<int32_t> order[kNB];    // the same entries, most-frames-first (launch order of the integration CTAs)
    DeviceArray<uint32_t> lmask[kNB];   // their frame masks in that order (the hash-side masks are cleared when this is built)
};

}  // namespace otslam

struct otslam_volume {
    int device = 0;
    double voxel_length = 0, sdf_trunc = 0, unit_length = 0;
    int color_type = OTSLAM_COLOR_RGB8;
    otslam::SlabSpec slab{0, 8, 1, 0, 1};
    otslam::Stream main_stream, copy_stream, pre_stream;
    cudaStream_t stream = nullptr;         // main_stream, or the caller's (otslam_volume_set_stream)
    int batch = otslam::kMaxBatch;
    int zsplit = 0;                // CTAs per block along z in the integration kernel: 0 = default (2), 1, 2, 4, 8
    int n_objects = 0;             // > 0: multi-object arena (object id in the block key), see common.cuh
    int sel_obj = -1;              // arena: object that extraction / export / stats address (-1 = none selected)
    int64_t obj_frames[otslam::kMaxObjects] = {};   // frames integrated per object (the 65535 limit is per voxel)
    int64_t frames_integrated = 0;

    otslam::BlockHash hash;        // volume_hash() below

    // block pool: chunks of kChunkBlocks blocks, 64 KiB per block
    std::vector<otslam::DeviceArray<uint4>> chunks;
    otslam::DeviceArray<uint4*> d_chunks;   // [kMaxChunks]
    int64_t n_blocks = 0;          // host mirror of the pool counter

    otslam::DeviceArray<int> d_counters;
    otslam::PinnedArray<int> h_counters;     // [kNB][kNumCounters]
    std::vector<uint4*> h_chunk_table;   // never reallocates (reserved to kMaxChunks): async copies read from it
    otslam::Event ev_pre_done[otslam::kNB], ev_k4_done[otslam::kNB], ev_main;

    // frame staging (kNB buffers)
    otslam::DeviceArray<uint8_t> d_raw_depth[otslam::kNB];   // u16 or f32 frames as uploaded
    otslam::DeviceArray<uint8_t> d_raw_rgb[otslam::kNB];
    otslam::DeviceArray<uint2> d_packed[otslam::kNB];
    otslam::DeviceArray<float> d_tiles[otslam::kNB];        // max-depth tiles of the packed frames (integration kernel's brick cull)
    bool cull = true;                      // OTSLAM_K4_CULL=0 turns the brick cull off (results are the same)
    size_t packed_px = 0;                  // image size of d_packed's zero sentinels
    otslam::Event ev_copied[otslam::kNB], ev_raw_free[otslam::kNB];
    otslam::DeviceArray<otslam::FrameDev> d_frames[otslam::kNB];   // [kMaxBatch]
    otslam::PinnedArray<otslam::FrameDev> h_frames;               // [kNB][kMaxBatch]

    // depth->camera-distance multiplier image, cached per intrinsics (SURVEY A.2)
    otslam::DeviceArray<float> d_mult;
    int mult_w = 0, mult_h = 0;
    double mult_intr[4] = {0, 0, 0, 0};

    // optional per-kernel timing (otslam_volume_profile)
    bool profiling = false;
    double prof_ms[4] = {0, 0, 0, 0};
    int64_t prof_launches[4] = {0, 0, 0, 0};
    std::vector<otslam::Event> prof_events;        // pairs, recycled
    std::vector<int> prof_pending;                 // kernel id per recorded pair
    size_t prof_used = 0;

    otslam::MeshResult mesh;
    otslam::PointsResult points;

    // device-resident list of the allocated blocks sorted by key (extraction order, export, halo selection); rebuilt
    // when `epoch` (bumped by integrate / reset / halo import) has moved past `sorted_epoch`
    uint64_t epoch = 1, sorted_epoch = 0;
    otslam::DevBuf<uint64_t> sorted_keys;
    otslam::DevBuf<int32_t> sorted_slots;
    int64_t n_sorted = 0;

    otslam::HaloPieces halo;

    otslam::Event ev_ext;                // otslam_volume_wait_stream

    ~otslam_volume();                    // drains the streams before the members release their memory
};

namespace otslam {
// implemented in volume.cu, used by extract.cu: the allocated blocks sorted by key, in HBM (valid until the volume changes)
int volume_sorted_blocks_device(otslam_volume* v, const uint64_t** d_keys, const int32_t** d_slots, int* n);
// the same restricted to the selected object of a multi-object arena (x_off = the object's x-key offset; 0 otherwise)
int volume_selected_blocks_device(otslam_volume* v, const uint64_t** d_keys, const int32_t** d_slots, int* n, int* x_off);
// the same downloaded to the host (export_blocks)
int volume_sorted_blocks(otslam_volume* v, std::vector<uint64_t>& keys, std::vector<int32_t>& slots);
// the volume's block hash as the kernels take it
inline HashTable volume_hash(const otslam_volume* v) { return {v->hash.keys.p, v->hash.vals.p, v->hash.cap - 1}; }
// volume.cu, used by checkpoint.cu: grow the block hash until it holds n_entries (drains both streams first when it must
// grow); pool chunks for blocks_needed slots
int reserve_hash(otslam_volume* v, int64_t n_entries);
int ensure_pool(otslam_volume* v, int64_t blocks_needed);
}
