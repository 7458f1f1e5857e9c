// ptcore.cu — the B200 path-tracing core: host side of the wavefront (csrc/pt_wavefront.cuh holds the kernels) and the
// C ABI of include/ptcore.h.
//
// Replaces the body of render_scene (src/renderer.rs:87-106 of the reference) and everything trace_ray
// (renderer.rs:19-65) calls.  One iteration of the wavefront = k_extend_pre, then (k_traverse, k_extend_post) once per
// mesh object a ray can meet, then k_shade (which also regenerates paths).  Every launch is `segments` blocks of 256
// threads, one block per pool segment, all sizes read on the device, and block b of a launch waits for block b of the
// launch before it, not for the whole launch (pt_wavefront.cuh: stage_begin) — the host enqueues iterations without
// synchronising and reads the state of the render from a word the device writes into mapped host memory.
//
// There is no CPU fallback in this library: without a CUDA device commit / render / intersect return PTC_E_CUDA.
#include <cuda_runtime.h>
#include <dlfcn.h>
#include <nccl.h>  // types and enums only: the library is bound at run time (see NcclApi)

#include <algorithm>
#include <chrono>
#include <cmath>
#include <condition_variable>
#include <exception>
#include <memory>
#include <mutex>
#include <thread>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <deque>
#include <functional>
#include <string>
#include <vector>

#include <cub/device/device_select.cuh>

#include "../../include/ptcore.h"
#include "pt_build_dev.h"
#include "pt_scene_host.h"
#include "pt_wavefront.cuh"
#include "pt_denoise.cuh"

using namespace pt;
using namespace ptw;

namespace {
constexpr uint32_t kTravCounters = 1u << 16;  // hand-out counters of split traversal launches, one per launch of a render

thread_local std::string g_err;

struct CudaError : std::runtime_error {
  using std::runtime_error::runtime_error;
};
#define CK(call)                                                                                      \
  do {                                                                                                \
    cudaError_t e_ = (call);                                                                          \
    if (e_ != cudaSuccess)                                                                            \
      throw CudaError(std::string(#call) + ": " + cudaGetErrorString(e_) + " (" __FILE__ ":" + std::to_string(__LINE__) + ")"); \
  } while (0)

template <typename T>
struct DevBuf {
  T *p = nullptr;
  size_t n = 0;
  void alloc(size_t count) {
    release();
    if (count == 0) count = 1;
    CK(cudaMalloc(&p, count * sizeof(T)));
    n = count;
  }
  void upload(const T *src, size_t count) {
    alloc(count);
    if (count) CK(cudaMemcpy(p, src, count * sizeof(T), cudaMemcpyHostToDevice));
  }
  void release() {
    if (p) cudaFree(p);
    p = nullptr;
    n = 0;
  }
  ~DevBuf() { release(); }
  DevBuf() = default;
  DevBuf(const DevBuf &) = delete;
  DevBuf &operator=(const DevBuf &) = delete;
};

// Path-state + task-queue storage for `segments` x `cap` slots.
struct Workspace {
  uint32_t segments = 0, cap = 0;
  int rounds = 0;
  DevBuf<float4> ray_o, ray_d, beta, hit0, hit1;
  DevBuf<float4> ray_o2, ray_d2, beta2;  // second set of ray arrays (renders only): k_shade reads one set, writes the other
  DevBuf<float> aux, aux2;               // PTC_FLAG_NEE only (allocated at the first such render)
  DevBuf<float> tau, tau2;               // motion renders only: the shutter time of every ray of the two sets (MotionTables)
  DevBuf<uint32_t> cnt;
  DevBuf<uint32_t> seg_flags;      // [3 * segments]: SegRange::flags
  DevBuf<uint32_t> trav_counters;  // [kTravCounters]: SegRange::trav_counter of the render's split traversal launches
  DevBuf<uint2> tq_ray[2];
  DevBuf<float4> tq_o[2], tq_d[2];
  DevBuf<unsigned long long> tq_res[2];
  DevBuf<uint32_t> tq_cnt;
  DevBuf<int2> ids;

  size_t slots() const { return (size_t)segments * cap; }
  // grow-only in cap; segments and rounds are fixed per scene / device
  void ensure(uint32_t seg, uint32_t want_cap, int mesh_rounds, bool want_ids, bool want_pingpong) {
    if (seg == segments && want_cap <= cap && mesh_rounds == rounds && (!want_ids || ids.n >= slots()) &&
        (!want_pingpong || ray_o2.n >= slots()))
      return;
    segments = seg;
    cap = std::max(cap, want_cap);
    rounds = mesh_rounds;
    const size_t n = slots();
    ray_o.alloc(n), ray_d.alloc(n), beta.alloc(n), hit0.alloc(n), hit1.alloc(n);
    cnt.alloc(segments);
    seg_flags.alloc(3 * (size_t)segments);
    trav_counters.alloc(kTravCounters);
    if (rounds > 0) {
      for (int k = 0; k < 2; k++) tq_ray[k].alloc(n), tq_o[k].alloc(n), tq_d[k].alloc(n), tq_res[k].alloc(n);
      tq_cnt.alloc((size_t)(rounds + 1) * segments);
    }
    if (want_ids) ids.alloc(n);
    if (want_pingpong) ray_o2.alloc(n), ray_d2.alloc(n), beta2.alloc(n);
  }
  // flip = 0: the stages read set 1 and k_shade writes set 2; flip = 1: the other way round
  void ensure_aux() {
    if (aux.n < slots()) aux.alloc(slots()), aux2.alloc(slots());
  }
  void ensure_tau() {
    if (tau.n < slots()) tau.alloc(slots()), tau2.alloc(slots());
  }
  // the shutter times that go with buffers(flip): the stages read `tau`, k_shade writes `ntau`
  MotionTables motion(int flip, const float4 *disp, const DCamera *end_cams) const {
    if (flip == 0) return MotionTables{disp, end_cams, tau.p, tau2.p};
    return MotionTables{disp, end_cams, tau2.p, tau.p};
  }
  Buffers buffers(int flip = 0) const {
    if (flip == 0) return Buffers{ray_o.p, ray_d.p, beta.p, hit0.p, hit1.p, cnt.p, cap, ray_o2.p, ray_d2.p, beta2.p, aux.p, aux2.p};
    return Buffers{ray_o2.p, ray_d2.p, beta2.p, hit0.p, hit1.p, cnt.p, cap, ray_o.p, ray_d.p, beta.p, aux2.p, aux.p};
  }
  TaskQ taskq() const {
    TaskQ q;
    for (int k = 0; k < 2; k++) q.ray[k] = tq_ray[k].p, q.o[k] = tq_o[k].p, q.d[k] = tq_d[k].p, q.res[k] = tq_res[k].p;
    q.cnt = rounds > 0 ? tq_cnt.p : nullptr;
    return q;
  }
};

}  // namespace

// ------------------------------------------------------------------------------------------------------------
struct ptc_scene {
  HostScene hs;
  bool committed = false;
  int device = -1;
  int sm_count = 0;
  DevBuf<DObject> d_objects;
  DevBuf<DMaterial> d_materials;
  DevBuf<DMesh> d_meshes;
  DevBuf<float> d_sky;
  DevBuf<DLight> d_lights;
  DevBuf<float> d_sky_dist;
  // PTC_FLAG_NEE_EMITTERS (HostScene::build_emitters): the object table with these light ids, the light list, its tables
  DevBuf<DObject> d_objects_em;
  DevBuf<DLight> d_lights_em;
  DevBuf<float> d_em_sel_cdf, d_em_ent_cdf;
  DevBuf<float4> d_em_ent;
  std::vector<std::unique_ptr<DevBuf<float4>>> mesh_bufs;
  std::vector<DevMeshBuffers> dev_built;  // per mesh: device arrays left behind by the device-side builder (adopted by upload_scene)
  DScene ds;
  DScene ds_em;      // ds with d_objects_em and d_lights_em: what every launch of a PTC_FLAG_NEE_EMITTERS render sees
  EmitterTables et;  // the tables of ds_em's lights
  int mesh_objects = 0;  // mesh entries in object_list = extend rounds needed

  int64_t last_pool_slots = 0;  // path-pool slots of the last render (ptc_scene_last_pool_slots)
  uint64_t pool_budget_bytes = 0;  // what the default pool may occupy: a quarter of the memory free at the first render, at most 48 GiB
  Workspace ws;       // render
  Workspace ws_hook;  // ptc_intersect (kept apart so a parity call never disturbs a render's pool)
  DevBuf<long long> film_sum;            // the fixed-point film of the render in flight (pt_wavefront.cuh: Film), grow-only
  DevBuf<unsigned long long> film_flags;
  char *h_film = nullptr;  // pinned staging for an image's way to the caller's (pageable) buffer, grow-only
  size_t h_film_bytes = 0;
  DevBuf<float> w_film_out;  // the resolved images (resolve_film_to_host) and ptc_resolve_u32's input, grow-only
  DevBuf<uint32_t> w_packed;
  // ptc_render_adaptive, grow-only: the film snapshot of the last decision, the needs-more byte map, the keep flag of
  // each list entry, the active list and the next one, every pixel's final count, the compaction's count and scratch
  DevBuf<float> w_adapt_vp;
  DevBuf<uint8_t> w_adapt_needs, w_adapt_keep;
  DevBuf<uint32_t> w_adapt_list[2];
  DevBuf<int32_t> w_adapt_spp;
  DevBuf<uint32_t> w_adapt_n;
  DevBuf<uint8_t> w_adapt_tmp;
  // ptc_render_progressive: two preview slots (pass j resolves into slot j % 2; the rgb image only when the caller wants
  // it), grow-only; the pinned buffer the calling thread shows previews from, and the stream it copies them on
  DevBuf<uint32_t> w_prog_packed[2];
  DevBuf<float> w_prog_rgb[2];
  uint32_t *h_preview = nullptr;
  size_t h_preview_px = 0;
  cudaStream_t preview_stream = nullptr;
  cudaEvent_t ev_prog_slot[2] = {nullptr, nullptr};  // recorded once slot j % 2 holds preview j
  cudaEvent_t ev_prog_begin = nullptr;                // render_ms: from here to the last slot event
  // ptc_render_denoised / ptc_denoise_image, grow-only: the fp32 film sums after the first half of the samples, one
  // sample's camera rays (origins, then directions), the feature sums (then means), the variance, the denoised image,
  // the filter's ping-pong input and its guides; the feature pass's control block; render_ms brackets
  DevBuf<float> w_dn_half, w_dn_rays, w_dn_albedo, w_dn_normal, w_dn_var, w_dn_out;
  DevBuf<float> w_dn_tau;  // a motion render's feature pass: the shutter time of every camera ray
  DevBuf<float4> w_dn_xv[2], w_dn_ga, w_dn_gn;
  DevBuf<Ctl> w_dn_ctl;
  cudaEvent_t ev_dn_begin = nullptr, ev_dn_end = nullptr;
  // ptc_render_batch, grow-only: the cameras and seeds of the views (pt_wavefront.cuh: BatchTables)
  DevBuf<DCamera> d_batch_cams;
  DevBuf<uint64_t> d_batch_seeds;
  // ptc_scene_set_lens: the lenses as set (empty = pinhole), and the (R, F) table of the render in flight, grow-only
  // (pt_wavefront.cuh: LensTables)
  std::vector<ptc_lens> lens;
  DevBuf<float2> d_lens;
  // ptc_scene_set_object_motion / ptc_scene_set_camera_motion: D per object as set (missing entries are 0) and the end
  // cameras (empty = static); the tables of the render in flight, grow-only (pt_wavefront.cuh: MotionTables)
  std::vector<float4> motion;
  std::vector<ptc_camera> end_cams;
  DevBuf<float4> d_motion_disp;
  DevBuf<DCamera> d_motion_cams;
  DevBuf<Ctl> d_ctl;
  Ctl *h_ctl = nullptr;  // pinned ring
  uint32_t *h_progress = nullptr;  // pinned + mapped: the word k_extend_pre reports the state of the render in
  static constexpr int kRing = 4;
  cudaEvent_t ring_ev[kRing] = {nullptr, nullptr, nullptr, nullptr};
  cudaEvent_t ev_begin = nullptr, ev_end = nullptr;  // render_ms brackets, created once (ensure_ctl)
  cudaEvent_t ev_adapt_begin = nullptr, ev_adapt_end = nullptr;  // ... of ptc_render_adaptive, around all its passes
  cudaStream_t own_stream = nullptr;
  std::vector<cudaEvent_t> timing_events;

  uint32_t segments() const { return (uint32_t)(sm_count * kSegPerSM); }
  Film film() const { return Film{film_sum.p, film_flags.p}; }

  ~ptc_scene() {
    if (device >= 0) cudaSetDevice(device);
    for (DevMeshBuffers &b : dev_built) {  // built but never adopted (commit failed half-way)
      if (b.device >= 0) cudaSetDevice(b.device);
      if (b.nodes) cudaFree(b.nodes);
      if (b.tris) cudaFree(b.tris);
      if (b.normals) cudaFree(b.normals);
    }
    if (device >= 0) cudaSetDevice(device);
    if (h_ctl) cudaFreeHost(h_ctl);
    if (h_progress) cudaFreeHost(h_progress);
    if (h_film) cudaFreeHost(h_film);
    for (auto &e : ring_ev)
      if (e) cudaEventDestroy(e);
    if (ev_begin) cudaEventDestroy(ev_begin);
    if (ev_end) cudaEventDestroy(ev_end);
    if (ev_adapt_begin) cudaEventDestroy(ev_adapt_begin);
    if (ev_adapt_end) cudaEventDestroy(ev_adapt_end);
    if (h_preview) cudaFreeHost(h_preview);
    for (auto &e : ev_prog_slot)
      if (e) cudaEventDestroy(e);
    if (ev_prog_begin) cudaEventDestroy(ev_prog_begin);
    if (ev_dn_begin) cudaEventDestroy(ev_dn_begin);
    if (ev_dn_end) cudaEventDestroy(ev_dn_end);
    if (preview_stream) cudaStreamDestroy(preview_stream);
    for (auto &e : timing_events) cudaEventDestroy(e);
    if (own_stream) cudaStreamDestroy(own_stream);
  }
};

namespace {

constexpr int64_t kDeviceRefMinTriangles = 1 << 17;  // ptc_scene_commit: from this size on the reference BVH is restated on the device

constexpr int64_t kHeavyMeshTriangles = 1 << 19;  // from this many mesh triangles on, k_traverse hands its tasks out in parts (measured:
                                                  // C5, 2 M triangles, -7 %; the 125 k-triangle teapot +5 %; profiles/r2_ab_travparts.jsonl)
constexpr int kTravParts = 4;

enum Stage { ST_PRE = 0, ST_TRAVERSE, ST_POST, ST_SHADE, ST_COUNT };

// One stage launch of the render loop: `segments` blocks of kBlock threads, optionally as a programmatic dependent launch
// (pt_wavefront.cuh: pdl_prologue).
template <typename... KArgs, typename... Args>
void launch_stage(bool pdl, cudaStream_t stream, uint32_t segments, void (*kernel)(KArgs...), Args &&...args) {
  cudaLaunchAttribute attr;
  attr.id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr.val.programmaticStreamSerializationAllowed = 1;
  cudaLaunchConfig_t cfg;
  memset(&cfg, 0, sizeof(cfg));
  cfg.gridDim = dim3(segments), cfg.blockDim = dim3(kBlock), cfg.dynamicSmemBytes = 0, cfg.stream = stream;
  cfg.attrs = pdl ? &attr : nullptr, cfg.numAttrs = pdl ? 1 : 0;
  CK(cudaLaunchKernelEx(&cfg, kernel, std::forward<Args>(args)...));
}

// k_traverse's `refill_lanes` argument.  PTC_REFILL: idle lanes that trigger a task fetch; PTC_STEAL=0: in-warp work
// stealing off (both read per call, for A/B measurements and tests)
uint32_t traverse_refill_arg() {
  const char *r = getenv("PTC_REFILL"), *st = getenv("PTC_STEAL");
  return (r ? (uint32_t)atoi(r) : kRefillLanes) | ((st && atoi(st) == 0) ? kNoSteal : 0u);
}

// One extend pass over ALL segments on one stream (ptc_intersect) = pre, then (traverse, post) once per mesh object a ray
// can meet.  Returns the number of launches.
// mt.tau != nullptr: the rays at their shutter times, through the motion twins of pre and post.
int launch_extend(cudaStream_t stream, uint32_t segments, int rounds, Ctl *ctl, const DScene &ds, const ExtendOut &eo, const TaskQ &tq,
                  float t_min, float t_max, bool counters, const MotionTables &mt = MotionTables{}) {
  const SegRange sr{0u, segments, 0u, 0u, 1u};
  if (mt.tau) k_extend_pre_motion<<<segments, kBlock, 0, stream>>>(ctl, sr, ds, eo, tq, t_min, t_max, nullptr, 0u, mt);
  else k_extend_pre<<<segments, kBlock, 0, stream>>>(ctl, sr, ds, eo, tq, t_min, t_max, nullptr, 0u);
  for (int r = 0; r < rounds; r++) {
    const SegRange tsr{0u, segments, 0u, (uint32_t)r, 1u};
    if (counters) k_traverse<true><<<segments, kBlock, 0, stream>>>(ctl, tsr, ds, tq, r, t_min, eo.b.cap, traverse_refill_arg());
    else k_traverse<false><<<segments, kBlock, 0, stream>>>(ctl, tsr, ds, tq, r, t_min, eo.b.cap, traverse_refill_arg());
    if (mt.tau) k_extend_post_motion<<<segments, kBlock, 0, stream>>>(ctl, sr, ds, eo, tq, r, t_min, t_max, mt);
    else k_extend_post<<<segments, kBlock, 0, stream>>>(ctl, sr, ds, eo, tq, r, t_min, t_max);
  }
  return 1 + 2 * rounds;
}

// n rays (device arrays of n x 3 floats) laid out like a render's pool in the hook workspace (segment b = slots
// [b * cap, ...), ray i in slot i) and run through the render's extend kernels: the hit records are left in ws_hook's
// hit0 / hit1 / ids.  ptc_intersect's rays and ptc_render_denoised's feature rays.  `before` / `after`, if given, are
// recorded around the extend launches.  `d_tau` (n floats) and `disp` (the object displacements, device), if given: the
// rays at their shutter times (ray i is in slot i, so d_tau is the time table as it stands).  Returns the number of
// extend launches.
int extend_hook_rays(ptc_scene *s, const float *d_o, const float *d_d, uint32_t n, float t_min, float t_max, Ctl *ctl, bool counters,
                     cudaStream_t st, cudaEvent_t before = nullptr, cudaEvent_t after = nullptr, const DScene *ds = nullptr,
                     const float *d_tau = nullptr, const float4 *disp = nullptr) {
  const uint32_t segments = s->segments();
  const uint32_t cap = (uint32_t)(((uint64_t)n + segments - 1) / segments + kBlock - 1) / kBlock * kBlock;
  s->ws_hook.ensure(segments, cap, s->mesh_objects, true, false);
  Buffers b = s->ws_hook.buffers();
  b.cap = cap;
  const TaskQ tq = s->ws_hook.taskq();
  k_fill_counts<<<(segments + 255) / 256, 256, 0, st>>>(b.cnt, segments, cap, n);
  k_pack_rays<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(d_o, d_d, (size_t)n, b.ray_o, b.ray_d);
  const ExtendOut eo{b, s->ws_hook.ids.p};
  if (before) CK(cudaEventRecord(before, st));
  const MotionTables mt = d_tau ? MotionTables{disp, nullptr, d_tau, nullptr} : MotionTables{};
  const int launches = launch_extend(st, segments, s->mesh_objects, ctl, ds ? *ds : s->ds, eo, tq, t_min, t_max, counters, mt);
  CK(cudaGetLastError());
  if (after) CK(cudaEventRecord(after, st));
  return launches;
}

void require_committed(const ptc_scene *s) {
  if (!s) throw std::invalid_argument("null scene");
  if (!s->committed) throw std::logic_error("scene not committed (call ptc_scene_commit first)");
}

// What every render entry point checks of its arguments; `has_output`: the caller passed the output(s) it needs.  The
// scene's state is checked apart (ptc_render_adaptive checks it after its own arguments).
void check_render_args(const ptc_camera *cam, const ptc_render_settings *st, bool has_output) {
  if (!cam || !st || !has_output) throw std::invalid_argument("null argument");
  if (st->width <= 0 || st->height <= 0 || st->spp <= 0) throw std::invalid_argument("bad render settings");
  if ((int64_t)st->width * st->height > (int64_t)0x3fffffff) throw std::invalid_argument("image too large");
  if ((st->flags & PTC_FLAG_NEE_SKY) && !(st->flags & PTC_FLAG_NEE)) throw std::invalid_argument("PTC_FLAG_NEE_SKY needs PTC_FLAG_NEE");
  if ((st->flags & PTC_FLAG_NEE_EMITTERS) && !(st->flags & PTC_FLAG_NEE)) throw std::invalid_argument("PTC_FLAG_NEE_EMITTERS needs PTC_FLAG_NEE");
}

// The samples [begin, end) a call renders: sample_begin = sample_end = 0 means [0, spp)
void sample_range(const ptc_render_settings *st, int &begin, int &end) {
  begin = st->sample_begin, end = st->sample_end;
  if (begin == 0 && end == 0) end = st->spp;
  if (begin < 0 || end < begin) throw std::invalid_argument("bad sample range");
}

// The scene's fixed-point film for n_px pixels: grow-only, and cleared on `stream` before every render that starts it
void ensure_film(ptc_scene *s, size_t n_px) {
  if (s->film_sum.n < n_px * 3) s->film_sum.alloc(n_px * 3);
  if (s->film_flags.n < n_px) s->film_flags.alloc(n_px);
}
void clear_film(ptc_scene *s, size_t n_px, cudaStream_t stream) {
  CK(cudaMemsetAsync(s->film_sum.p, 0, n_px * 3 * sizeof(long long), stream));
  CK(cudaMemsetAsync(s->film_flags.p, 0, n_px * sizeof(unsigned long long), stream));
}

void ensure_ctl(ptc_scene *s) {
  if (s->h_ctl) return;
  s->d_ctl.alloc(1);
  CK(cudaMallocHost(&s->h_ctl, sizeof(Ctl) * ptc_scene::kRing));
  CK(cudaHostAlloc(&s->h_progress, 64, cudaHostAllocMapped | cudaHostAllocPortable));
  for (auto &e : s->ring_ev) CK(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
  CK(cudaEventCreate(&s->ev_begin));
  CK(cudaEventCreate(&s->ev_end));
  CK(cudaEventCreate(&s->ev_adapt_begin));
  CK(cudaEventCreate(&s->ev_adapt_end));
}

// What one call of render_accumulate renders besides its settings.  Default: the tiles of the settings into a cleared
// film.  ptc_render_adaptive's passes add samples to the film as it stands, the later ones for a list of pixels only.
// ptc_render_batch renders the tiles of `views` cameras into one film of views x W x H pixels, view-major.
struct Pass {
  bool clear_film = true;
  const uint32_t *pixels = nullptr;  // device, ascending; nullptr: the tiles of tile_mod / tile_rem
  uint32_t n_pixels = 0;
  uint32_t views = 0;                // > 0: a batch (tile_mod = 0); its cameras and seeds, device tables of `views` entries
  const DCamera *cams = nullptr;
  const uint64_t *seeds = nullptr;
  const float2 *lens = nullptr;      // device, (R, F) per view (one for a single camera); nullptr: pinhole, today's kernels
  // motion blur: the motion twins run, with the displacement table (device, one per object) and the end cameras (device,
  // one per view; nullptr: a static camera).  false: no object moves and every end camera is its start camera, today's kernels
  bool motion = false;
  const float4 *disp = nullptr;
  const DCamera *end_cams = nullptr;
};

// The end camera a single-camera call uses: end_cams[0] of ptc_scene_set_camera_motion, nullptr for a static camera.
// Checked before the scene's state.
const ptc_camera *single_end_cam(const ptc_scene *s) {
  if (s->end_cams.size() > 1)
    throw std::invalid_argument("a single-camera call uses one end camera: ptc_scene_set_camera_motion was given n > 1");
  return s->end_cams.empty() ? nullptr : &s->end_cams[0];
}

// What one call moves, from the motion state of handle `s` (the primary handle of a ptc_multi): D per object, and an end
// camera per view where the views' end cameras are not all equal to their start cameras bit for bit (ends[k % ends.size()]
// goes with view k: one end camera for all views, or one each).
struct MotionCall {
  std::vector<float4> disp;
  std::vector<DCamera> end_cams;  // empty: no camera moves
  bool objects = false;
  bool any() const { return objects || !end_cams.empty(); }
};
MotionCall motion_call(const ptc_scene *s, const ptc_camera *cams, size_t views, const ptc_camera *ends, size_t n_ends) {
  MotionCall mc;
  const size_t n_obj = s->hs.objects.size();
  mc.disp.assign(std::max<size_t>(n_obj, 1), make_float4(0.0f, 0.0f, 0.0f, 0.0f));
  for (size_t k = 0; k < n_obj && k < s->motion.size(); k++) {
    mc.disp[k] = s->motion[k];
    mc.objects = mc.objects || motion_moves(s->motion[k]);
  }
  bool camera = false;
  for (size_t v = 0; v < views && n_ends > 0; v++) camera = camera || memcmp(&ends[v % n_ends], &cams[v], sizeof(ptc_camera)) != 0;
  if (camera) {
    mc.end_cams.resize(views);
    for (size_t v = 0; v < views; v++) memcpy(&mc.end_cams[v], &ends[v % n_ends], sizeof(DCamera));
  }
  return mc;
}
// Grow `d`'s motion tables to hold `mc` (ptc_multi allocates them before its threads start)
void ensure_motion(ptc_scene *d, const MotionCall &mc) {
  if (d->d_motion_disp.n < mc.disp.size()) d->d_motion_disp.alloc(mc.disp.size());
  if (d->d_motion_cams.n < mc.end_cams.size()) d->d_motion_cams.alloc(mc.end_cams.size());
}
// mc into the device tables of `d` (the scene a render runs on), one copy per table on `stream`, and into `pass`.  Nothing
// when nothing moves: the call runs today's kernels.
void upload_motion(ptc_scene *d, const MotionCall &mc, cudaStream_t stream, Pass &pass) {
  static_assert(sizeof(ptc_camera) == sizeof(DCamera), "ptc_camera and DCamera share one layout");
  if (!mc.any()) return;
  ensure_motion(d, mc);
  // (from pageable memory: the call returns once the source has been read)
  CK(cudaMemcpyAsync(d->d_motion_disp.p, mc.disp.data(), mc.disp.size() * sizeof(float4), cudaMemcpyHostToDevice, stream));
  if (!mc.end_cams.empty())
    CK(cudaMemcpyAsync(d->d_motion_cams.p, mc.end_cams.data(), mc.end_cams.size() * sizeof(DCamera), cudaMemcpyHostToDevice, stream));
  pass.motion = true;
  pass.disp = d->d_motion_disp.p;
  pass.end_cams = mc.end_cams.empty() ? nullptr : d->d_motion_cams.p;
}
// the motion of a single-camera call of `s` (end camera from single_end_cam)
MotionCall single_motion(const ptc_scene *s, const ptc_camera *cam, const ptc_camera *end) {
  return motion_call(s, cam, 1, end, end ? 1 : 0);
}

// The lens a single-camera call uses: lenses[0] of ptc_scene_set_lens, nullptr for a pinhole or a zero aperture (the call
// then runs exactly the kernels it runs without a lens).  Checked before the scene's state.
const ptc_lens *single_lens(const ptc_scene *s) {
  if (s->lens.size() > 1) throw std::invalid_argument("a single-camera call uses one lens: ptc_scene_set_lens was given n > 1");
  return !s->lens.empty() && s->lens[0].aperture_radius > 0.0f ? &s->lens[0] : nullptr;
}

// n lenses into the device table of `d` (the scene a render runs on), one copy on `stream`; nullptr when none has an
// aperture.  The table grows only, and is allocated before the copy (ptc_multi allocates it before its threads start).
const float2 *upload_lens(ptc_scene *d, const ptc_lens *l, size_t n, cudaStream_t stream) {
  static_assert(sizeof(ptc_lens) == sizeof(float2), "ptc_lens and float2 share one layout");
  bool any = false;
  for (size_t k = 0; k < n; k++) any = any || l[k].aperture_radius > 0.0f;
  if (!any) return nullptr;
  if (d->d_lens.n < n) d->d_lens.alloc(n);
  // (from pageable memory: the call returns once the source has been read)
  CK(cudaMemcpyAsync(d->d_lens.p, l, n * sizeof(float2), cudaMemcpyHostToDevice, stream));
  return d->d_lens.p;
}

// k_shade_lens<mode, Src>: 0 plain, 1 NEE, 2 NEE + sky, 3 NEE + emitters, 4 NEE + sky + emitters
using ShadeLensKernel = void (*)(Ctl *, SegRange, DScene, RenderParams, Buffers, Film, BatchTables, EmitterTables, LensTables);
template <int Src>
ShadeLensKernel shade_lens_kernel(int mode) {
  switch (mode) {
    case 0: return k_shade_lens<0, Src>;
    case 1: return k_shade_lens<1, Src>;
    case 2: return k_shade_lens<2, Src>;
    case 3: return k_shade_lens<3, Src>;
    default: return k_shade_lens<4, Src>;
  }
}

// k_shade_motion<mode, Src>, the same modes
using ShadeMotionKernel = void (*)(Ctl *, SegRange, DScene, RenderParams, Buffers, Film, BatchTables, EmitterTables, LensTables, MotionTables);
template <int Src>
ShadeMotionKernel shade_motion_kernel(int mode) {
  switch (mode) {
    case 0: return k_shade_motion<0, Src>;
    case 1: return k_shade_motion<1, Src>;
    case 2: return k_shade_motion<2, Src>;
    case 3: return k_shade_motion<3, Src>;
    default: return k_shade_motion<4, Src>;
  }
}

// the wavefront loop; renders into the scene's fixed-point film and then adds its fp32 image into d_accum on `stream`
// (d_accum == nullptr: the caller takes the fixed-point film itself).  The caller has checked the scene's state and
// check_render_args.
void render_accumulate(ptc_scene *s, const ptc_camera *cam, const ptc_render_settings *st, float *d_accum,
                       cudaStream_t stream, ptc_stats *stats, const Pass &pass = Pass()) {
  CK(cudaSetDevice(s->device));
  int s_begin, s_end;
  sample_range(st, s_begin, s_end);
  const int tile_mod = st->tile_mod > 0 ? st->tile_mod : 1;
  const int tile_rem = st->tile_mod > 0 ? st->tile_rem : 0;
  if (tile_rem < 0 || tile_rem >= tile_mod) throw std::invalid_argument("tile_rem out of range");
  const bool nee = (st->flags & PTC_FLAG_NEE) != 0;
  // the sky joins the sampled lights only where there is a sky distribution; elsewhere the flag changes nothing
  const bool nee_sky = nee && (st->flags & PTC_FLAG_NEE_SKY) != 0 && s->ds.sky_dist != nullptr;
  // emissive meshes and cubes join the sampled lights: every launch sees the object table that carries their light ids
  const bool nee_em = nee && (st->flags & PTC_FLAG_NEE_EMITTERS) != 0;
  const DScene &ds = nee_em ? s->ds_em : s->ds;
  const int tiles_x = (st->width + 31) / 32, n_tiles = tiles_x * ((st->height + 31) / 32);
  const uint32_t views = std::max<uint32_t>(pass.views, 1u);  // a batch's tile grids are stacked (the caller checked the size)
  const int n_my_tiles = (tile_rem < n_tiles ? (n_tiles - tile_rem + tile_mod - 1) / tile_mod : 0) * (int)views;
  // paths this call starts (its tiles x its samples; border tiles padded to 32 x 32 like the path index space; a pixel
  // list padded to 32 entries)
  const uint64_t list_padded = ((uint64_t)pass.n_pixels + 31u) & ~31ull;
  const uint64_t want_paths = (pass.pixels ? list_padded : (uint64_t)n_my_tiles * 1024ull) * (uint64_t)(s_end - s_begin);
  uint64_t pool;
  if (st->pool_paths > 0) {
    pool = (uint64_t)st->pool_paths;
  } else {
    // Default pool.  Measured on C2 (profiles/r2_pool_sweep.jsonl, tools/pool_share_probe.py): fastest when the WHOLE job is
    // in flight at once (as many iterations as the depth limit, all of them as full as they can be: 41.6 ms against
    // 43.2 ms at 48 Mi slots), next best with many fills of a large pool, worst when a second, ragged fill trails the
    // first (46.6 ms at 0.8 x the job).  So: the job itself if that fits a quarter of the free memory (and 48 GiB),
    // else 48 Mi slots, and never between one and 2.5 fills.
    const uint64_t per_slot = 128ull + (s->mesh_objects > 0 ? 96ull : 0ull) + (nee ? 8ull : 0ull) + (pass.motion ? 8ull : 0ull);
    if (s->pool_budget_bytes == 0) {
      // asked once per scene: cudaMemGetInfo contends with NVML pollers (nvidia-smi -lms) for tens of milliseconds
      size_t free_b = 0, total_b = 0;
      CK(cudaMemGetInfo(&free_b, &total_b));
      s->pool_budget_bytes = std::max<uint64_t>(std::min<uint64_t>((uint64_t)free_b / 4, 48ull << 30), 1ull << 24);
    }
    const uint64_t budget = s->pool_budget_bytes / per_slot;
    const uint64_t want_slots = nee ? 2 * want_paths : want_paths;  // with NEE paths may fill half a segment only
    if (want_slots <= budget) {
      pool = std::max<uint64_t>(want_slots, 1u << 16);
    } else {
      pool = std::min<uint64_t>(budget, 48ull << 20);
      if (want_slots < 5 * pool / 2) pool = (want_slots + 2) / 3;
    }
  }
  const uint32_t segments = s->segments();
  uint64_t cap64 = (pool + segments - 1) / segments;
  cap64 = std::max<uint64_t>((cap64 + kBlock - 1) / kBlock * kBlock, kBlock);
  if (cap64 * segments > 0x7fffffffull) throw std::invalid_argument("pool_paths too large");
  ensure_ctl(s);
  s->ws.ensure(segments, (uint32_t)cap64, s->mesh_objects, false, true);
  if (nee) s->ws.ensure_aux();
  if (pass.motion) s->ws.ensure_tau();
  s->last_pool_slots = (int64_t)cap64 * segments;
  Buffers bufs[2] = {s->ws.buffers(0), s->ws.buffers(1)};
  bufs[0].cap = bufs[1].cap = (uint32_t)cap64;  // a pool smaller than the allocation simply uses a smaller segment stride
  const TaskQ tq = s->ws.taskq();

  RenderParams rp;
  memcpy(&rp.cam, cam, sizeof(DCamera));
  rp.width = st->width, rp.height = st->height;
  rp.max_depth = st->max_depth;
  rp.sample_begin = s_begin, rp.n_samples = s_end - s_begin;
  rp.tiles_x = tiles_x;
  rp.n_my_tiles = n_my_tiles;
  rp.tile_mod = tile_mod, rp.tile_rem = tile_rem;
  rp.seed = st->seed;
  rp.pixel_list = pass.pixels, rp.n_list = pass.n_pixels;
  {  // odd multiplier coprime with the number of 32-pixel rows (= n_my_tiles * 32, or padded list entries / 32): a bijection
     // on row indices
    auto gcd = [](uint64_t a, uint64_t b) {
      while (b) {
        const uint64_t t = a % b;
        a = b;
        b = t;
      }
      return a;
    };
    const uint64_t rows = pass.pixels ? std::max<uint64_t>(list_padded / 32u, 1u) : (uint64_t)std::max(rp.n_my_tiles, 1) * 32ull;
    uint64_t m = (0x9E3779B1ull % rows) | 1ull;
    while (gcd(m, rows) != 1) m += 2;
    rp.row_mult = (uint32_t)m;
  }

  // valid pixels of this rank (for the paths statistic)
  uint64_t my_pixels = pass.pixels ? pass.n_pixels : 0;
  for (int t = tile_rem; !pass.pixels && t < n_tiles; t += tile_mod) {
    const int tx = t % rp.tiles_x, ty = t / rp.tiles_x;
    const int w = std::min(32, st->width - tx * 32), h = std::min(32, st->height - ty * 32);
    my_pixels += (uint64_t)w * h;
  }
  my_pixels *= views;

  Ctl init;
  memset(&init, 0, sizeof(init));
  init.total_paths = rp.max_depth > 0 ? want_paths : 0ull;
  init.n_active = init.total_paths != 0ull ? segments : 0u;  // every segment reports once when it is empty for good (stage_shade)
  // Does the initial fill reserve every path?  Each segment's first reservation takes min(room, share) paths (stage_shade:
  // room = cap, cap / 2 with NEE; share = its fair share of the job in whole rows) unless the supply is already out.
  const uint64_t fill_share = ((init.total_paths + segments - 1) / segments + 31ull) & ~31ull;
  const bool job_in_first_fill = (uint64_t)segments * std::min<uint64_t>(nee ? cap64 / 2 : cap64, fill_share) >= init.total_paths;
  const size_t n_px = (size_t)st->width * st->height * views;
  ensure_film(s, n_px);
  const Film film = s->film();
  if (pass.clear_film) clear_film(s, n_px, stream);
  CK(cudaMemcpyAsync(s->d_ctl.p, &init, sizeof(Ctl), cudaMemcpyHostToDevice, stream));
  CK(cudaMemsetAsync(bufs[0].cnt, 0, segments * sizeof(uint32_t), stream));
  CK(cudaMemsetAsync(s->ws.seg_flags.p, 0, 3 * (size_t)segments * sizeof(uint32_t), stream));

  const bool counters = (st->flags & PTC_FLAG_COUNTERS) != 0;
  const bool timing = (st->flags & PTC_FLAG_TIMING) != 0;
  const int rounds = s->mesh_objects;

  const cudaEvent_t ev_begin = s->ev_begin, ev_end = s->ev_end;  // owned by the scene: nothing to leak if a launch throws
  size_t tev_used = 0;
  auto tev = [&]() -> cudaEvent_t {
    if (tev_used == s->timing_events.size()) {
      cudaEvent_t e;
      CK(cudaEventCreate(&e));
      s->timing_events.push_back(e);
    }
    return s->timing_events[tev_used++];
  };
  std::vector<int> mark_stage;
  const auto mark = [&](int stage) {
    CK(cudaEventRecord(tev(), stream));
    mark_stage.push_back(stage);
  };

  CK(cudaEventRecord(ev_begin, stream));
  uint64_t launches = 0;
  const uint32_t refill = traverse_refill_arg();
  auto is_done = [](const Ctl &c) { return c.n_active == 0 && c.sync_timeouts == 0 && c.next_path >= c.total_paths; };
  // programmatic dependent launches, unless the per-stage events are wanted (they would sit between the launches) or
  // PTC_PDL=0
  static const bool pdl_on = getenv("PTC_PDL") ? atoi(getenv("PTC_PDL")) != 0 : true;
  const bool pdl = pdl_on && !timing;
  if (init.total_paths != 0) {
    // Every launch gets a number; a block waits for ITS segment to have been finished by launch number - 1 instead of for
    // the whole launch (pt_wavefront.cuh: stage_begin).  PTC_DATAFLOW=0: whole launches, as in round 1.
    const bool dataflow = getenv("PTC_DATAFLOW") ? atoi(getenv("PTC_DATAFLOW")) != 0 : true;
    uint32_t stage_id = 0;
    auto seg_range = [&](uint32_t trav_seq_, uint32_t trav_parts_) {
      // (the first launch follows the host's memsets: it waits for the stream, not for a flag)
      SegRange r{0u, segments, 0u, trav_seq_, trav_parts_, s->ws.seg_flags.p, ++stage_id, (dataflow && stage_id > 1u) ? 1u : 0u, nullptr};
      if (trav_parts_ > 1u) r.trav_counter = s->ws.trav_counters.p + trav_seq_;
      return r;
    };
    // k_traverse cuts the task lists into parts handed out dynamically while a scene with a heavy mesh is in the bulk of
    // its render (pt_wavefront.cuh: k_traverse); in the drain the lists are too short for that.  PTC_TRAV_PARTS overrides.
    int64_t mesh_tris = 0;
    for (const auto &mb : s->hs.meshes) mesh_tris += mb->n;
    const char *tp_env = getenv("PTC_TRAV_PARTS");
    const uint32_t trav_parts_bulk = tp_env ? (uint32_t)std::max(1, atoi(tp_env)) : (mesh_tris >= kHeavyMeshTriangles ? (uint32_t)kTravParts : 1u);
    if (trav_parts_bulk > 1u) CK(cudaMemsetAsync(s->ws.trav_counters.p, 0, kTravCounters * sizeof(uint32_t), stream));  // before any launch
    uint32_t trav_seq = 0;
    bool draining = false;  // the progress word (or a snapshot) has shown the path supply exhausted
    int flip = 0;  // the ray set the extend stages read
    // How the host learns that the render is over.  Default: k_extend_pre writes one word into mapped host memory
    // (pt_wavefront.cuh) and the host polls it — nothing sits between the launches, and the host stays at most a few
    // iterations ahead of the device.  PTC_PROGRESS=0: round 1's way, a copy of the control block + an event in the stream
    // (every iteration of the drain: the copy engine's turn and a launch that cannot overlap cost ~7 us of each ~55 us).
    const bool progress_on = getenv("PTC_PROGRESS") ? atoi(getenv("PTC_PROGRESS")) != 0 : true;
    uint32_t *d_progress = nullptr;
    if (progress_on) {
      CK(cudaHostGetDevicePointer((void **)&d_progress, s->h_progress, 0));
      *(volatile uint32_t *)s->h_progress = 0u;
    }
    uint64_t it = 0;
    auto run_extend = [&]() {
      const ExtendOut eo{bufs[flip], nullptr};
      if (timing) mark(ST_PRE);
      if (pass.motion)
        launch_stage(pdl, stream, segments, k_extend_pre_motion, s->d_ctl.p, seg_range(0u, 1u), ds, eo, tq, kEps, INFINITY,
                     (volatile uint32_t *)d_progress, (uint32_t)(it + 1), s->ws.motion(flip, pass.disp, pass.end_cams));
      else
        launch_stage(pdl, stream, segments, k_extend_pre, s->d_ctl.p, seg_range(0u, 1u), ds, eo, tq, kEps, INFINITY,
                     (volatile uint32_t *)d_progress, (uint32_t)(it + 1));  // renderer.rs:24
      for (int r = 0; r < rounds; r++) {
        if (timing) mark(ST_TRAVERSE);
        // (a split launch needs a hand-out counter of its own; a render with more launches than counters goes on unsplit)
        const SegRange tsr = seg_range(trav_seq, (draining || trav_seq >= kTravCounters) ? 1u : trav_parts_bulk);
        trav_seq++;
        if (counters) launch_stage(pdl, stream, segments, k_traverse<true>, s->d_ctl.p, tsr, ds, tq, r, kEps, eo.b.cap, refill);
        else launch_stage(pdl, stream, segments, k_traverse<false>, s->d_ctl.p, tsr, ds, tq, r, kEps, eo.b.cap, refill);
        if (timing) mark(ST_POST);
        if (pass.motion)
          launch_stage(pdl, stream, segments, k_extend_post_motion, s->d_ctl.p, seg_range(0u, 1u), ds, eo, tq, r, kEps, INFINITY,
                       s->ws.motion(flip, pass.disp, pass.end_cams));
        else
          launch_stage(pdl, stream, segments, k_extend_post, s->d_ctl.p, seg_range(0u, 1u), ds, eo, tq, r, kEps, INFINITY);
      }
      launches += 1 + 2 * (uint64_t)rounds;
    };
    auto run_shade = [&]() {  // reads set `flip`, writes the other one, which the next extend then reads
      if (timing) mark(ST_SHADE);
      const SegRange ssr = seg_range(0u, 1u);
      const int mode = nee_sky ? 2 : (nee ? 1 : 0);
      if (pass.motion) {
        const BatchTables bt = pass.views > 0 ? BatchTables{pass.cams, pass.seeds, (uint32_t)st->width * (uint32_t)st->height, (uint32_t)n_tiles}
                                              : BatchTables{};
        const int mmode = nee_em ? (nee_sky ? 4 : 3) : mode;
        auto *kernel = pass.views > 0 ? shade_motion_kernel<kSrcBatch>(mmode)
                       : pass.pixels  ? shade_motion_kernel<kSrcList>(mmode)
                                      : shade_motion_kernel<kSrcTiles>(mmode);
        launch_stage(pdl, stream, segments, kernel, s->d_ctl.p, ssr, ds, rp, bufs[flip], film, bt, nee_em ? s->et : EmitterTables{},
                     LensTables{pass.lens}, s->ws.motion(flip, pass.disp, pass.end_cams));
      } else if (pass.lens) {
        const BatchTables bt = pass.views > 0 ? BatchTables{pass.cams, pass.seeds, (uint32_t)st->width * (uint32_t)st->height, (uint32_t)n_tiles}
                                              : BatchTables{};
        const int lmode = nee_em ? (nee_sky ? 4 : 3) : mode;
        auto *kernel = pass.views > 0 ? shade_lens_kernel<kSrcBatch>(lmode)
                       : pass.pixels  ? shade_lens_kernel<kSrcList>(lmode)
                                      : shade_lens_kernel<kSrcTiles>(lmode);
        launch_stage(pdl, stream, segments, kernel, s->d_ctl.p, ssr, ds, rp, bufs[flip], film, bt, nee_em ? s->et : EmitterTables{},
                     LensTables{pass.lens});
      } else if (nee_em) {
        const BatchTables bt = pass.views > 0 ? BatchTables{pass.cams, pass.seeds, (uint32_t)st->width * (uint32_t)st->height, (uint32_t)n_tiles}
                                              : BatchTables{};
        auto *kernel = pass.views > 0 ? (nee_sky ? k_shade_em<4, kSrcBatch> : k_shade_em<3, kSrcBatch>)
                       : pass.pixels  ? (nee_sky ? k_shade_em<4, kSrcList> : k_shade_em<3, kSrcList>)
                                      : (nee_sky ? k_shade_em<4, kSrcTiles> : k_shade_em<3, kSrcTiles>);
        launch_stage(pdl, stream, segments, kernel, s->d_ctl.p, ssr, ds, rp, bufs[flip], film, bt, s->et);
      } else if (pass.views > 0) {
        const BatchTables bt{pass.cams, pass.seeds, (uint32_t)st->width * (uint32_t)st->height, (uint32_t)n_tiles};
        auto *kernel = mode == 2 ? k_shade_batch<2> : mode == 1 ? k_shade_batch<1> : k_shade_batch<0>;
        launch_stage(pdl, stream, segments, kernel, s->d_ctl.p, ssr, s->ds, rp, bufs[flip], film, bt);
      } else {
        auto *kernel = pass.pixels ? (mode == 2 ? k_shade<2, true> : mode == 1 ? k_shade<1, true> : k_shade<0, true>)
                                   : (mode == 2 ? k_shade<2> : mode == 1 ? k_shade<1> : k_shade<0>);
        launch_stage(pdl, stream, segments, kernel, s->d_ctl.p, ssr, s->ds, rp, bufs[flip], film);
      }
      launches += 1;
      flip ^= 1;
    };
    run_shade();  // initial fill: a shade pass over empty segments is pure regeneration
    bool finished = false;
    uint64_t last_iteration = ~0ull;
    if (progress_on) {
      const volatile uint32_t *prog = s->h_progress;
      while (!finished) {
        run_extend();
        run_shade();
        it++;
        // the extend of iteration k reports what the shade of iteration k - 1 left: nothing alive and nothing to start
        // means every launch from k on is empty.  Ahead of the device by kAhead iterations at most (4 launches of ~2.5 us
        // each against >= 45 us per iteration: two would do), so that few empty launches trail the render.
        // And once the supply is known to be exhausted the end is known too.  When the initial fill reserved every path,
        // a path started by the shade of iteration k - 1 at the latest has its last segment in iteration k - 1 +
        // max_depth (the whole job in flight at once: exactly max_depth iterations, no trailing launch at all).
        // Otherwise segment 0's report says nothing about the others: segments run ahead of each other, and another one
        // may have reserved the last paths in a later shade.  Every shade it can have run has been enqueued, though, so
        // the paths end by iteration it + max_depth.
        const uint64_t kAhead = getenv("PTC_AHEAD") ? (uint64_t)std::max(1, atoi(getenv("PTC_AHEAD"))) : 3u;
        for (uint32_t spins = 0;; spins++) {
          const uint32_t w = *prog;
          if ((w & 3u) == 3u) {
            finished = true;
            break;
          }
          if ((w & 2u) && !draining) {
            draining = true;
            last_iteration = (job_in_first_fill ? (uint64_t)(w >> 2) - 1u : it) + (uint64_t)rp.max_depth + (nee ? 1u : 0u);  // + the last hit's shadow ray
          }
          if (it >= last_iteration) {
            finished = true;
            break;
          }
          if (it < kAhead + (uint64_t)(w >> 2)) break;
          if ((spins & 0x3ffu) == 0x3ffu) {  // a device fault must not leave the host spinning
            const cudaError_t e = cudaStreamQuery(stream);
            if (e != cudaSuccess && e != cudaErrorNotReady) CK(e);
          }
        }
      }
    } else {
      std::deque<int> pending;
      int ring_next = 0;
      int check_every = 4;  // 1 once a snapshot shows the path supply exhausted: the drain's launches are cheap, running ahead of
                            // the device by up to kRing x 4 empty iterations at the end of every render is not
      while (!finished) {
        run_extend();
        run_shade();
        it++;
        if (it % check_every == 0) {
          // snapshot the control block; consume finished snapshots without stalling the launch queue.  The host only
          // blocks when the ring is full.
          const int k = ring_next;
          ring_next = (ring_next + 1) % ptc_scene::kRing;
          CK(cudaMemcpyAsync(&s->h_ctl[k], s->d_ctl.p, sizeof(Ctl), cudaMemcpyDeviceToHost, stream));
          CK(cudaEventRecord(s->ring_ev[k], stream));
          pending.push_back(k);
          while (!pending.empty()) {
            const int o = pending.front();
            const bool must_wait = (int)pending.size() >= ptc_scene::kRing;
            if (!must_wait && cudaEventQuery(s->ring_ev[o]) == cudaErrorNotReady) {
              cudaGetLastError();
              break;
            }
            CK(cudaEventSynchronize(s->ring_ev[o]));
            pending.pop_front();
            if (is_done(s->h_ctl[o])) {
              finished = true;
              break;
            }
            if (s->h_ctl[o].next_path >= s->h_ctl[o].total_paths) check_every = 1, draining = true;
          }
        }
      }
    }
  }
  CK(cudaGetLastError());
  if (d_accum) {
    k_film_to_accum<<<(unsigned)((n_px * 3 + 255) / 256), 256, 0, stream>>>(film, n_px, d_accum);
    launches += 1;
  }
  CK(cudaGetLastError());
  CK(cudaEventRecord(ev_end, stream));
  CK(cudaMemcpyAsync(&s->h_ctl[0], s->d_ctl.p, sizeof(Ctl), cudaMemcpyDeviceToHost, stream));
  CK(cudaStreamSynchronize(stream));
  const Ctl fin = s->h_ctl[0];
  if (!is_done(fin)) throw std::runtime_error("wavefront loop ended before all paths terminated");
  if (stats) {
    memset(stats, 0, sizeof(*stats));
    stats->paths = rp.max_depth > 0 ? my_pixels * (uint64_t)rp.n_samples : 0;
    stats->rays = fin.rays;
    stats->iterations = fin.iterations[0];  // the last iteration any segment had a ray in
    stats->kernel_launches = launches;
    float ms = 0.0f;
    CK(cudaEventElapsedTime(&ms, ev_begin, ev_end));
    stats->render_ms = ms;
    if (timing) {
      // every mark opens a stage that lasts until the next mark (the last one until the end-of-render event)
      double per[ST_COUNT] = {0, 0, 0, 0};
      uint64_t n_ext = 0;
      // PTC_TRACE_STAGES=<file>: every launch's stage number and milliseconds, in launch order (tools/drain_trace.py)
      const char *trace_path = getenv("PTC_TRACE_STAGES");
      FILE *trace = trace_path ? fopen(trace_path, "w") : nullptr;
      for (size_t k = 0; k < tev_used; k++) {
        float a = 0.0f;
        CK(cudaEventElapsedTime(&a, s->timing_events[k], k + 1 < tev_used ? s->timing_events[k + 1] : ev_end));
        if (trace) fprintf(trace, "%d %.6f\n", mark_stage[k], a);
        per[mark_stage[k]] += a;
        if (mark_stage[k] == ST_PRE) n_ext++;
      }
      if (trace) fclose(trace);
      stats->pre_ms = per[ST_PRE];
      stats->traverse_ms = per[ST_TRAVERSE];
      stats->post_ms = per[ST_POST];
      stats->extend_ms = per[ST_PRE] + per[ST_TRAVERSE] + per[ST_POST];
      stats->shade_ms = per[ST_SHADE];
      stats->regen_ms = 0.0;  // regeneration is part of k_shade
      stats->extend_launches = n_ext;
    }
    stats->nodes_visited = fin.nodes;
    stats->tris_tested = fin.tris;
    stats->mesh_rays = fin.mesh_rays;
  }
}

// One pass of a render made of passes (ptc_render_adaptive, ptc_render_progressive): samples [first, last) of `pass`
// into the scene's film, its stats added to `total`.  render_ms is left alone: the caller brackets all its passes.
void render_pass(ptc_scene *s, const ptc_camera *cam, const ptc_render_settings *st, int first, int last, const Pass &pass,
                 cudaStream_t stream, ptc_stats &total) {
  ptc_render_settings ps = *st;
  ps.sample_begin = first, ps.sample_end = last;
  ptc_stats p;
  render_accumulate(s, cam, &ps, nullptr, stream, &p, pass);
  total.paths += p.paths, total.rays += p.rays, total.iterations += p.iterations, total.kernel_launches += p.kernel_launches;
  total.extend_ms += p.extend_ms, total.shade_ms += p.shade_ms, total.extend_launches += p.extend_launches;
  total.pre_ms += p.pre_ms, total.traverse_ms += p.traverse_ms, total.post_ms += p.post_ms;
  total.nodes_visited += p.nodes_visited, total.tris_tested += p.tris_tested, total.mesh_rays += p.mesh_rays;
}

int fail(int code, const std::string &msg) {
  g_err = msg;
  return code;
}

#define PTC_GUARD_BEGIN try {
#define PTC_GUARD_END                                   \
  }                                                     \
  catch (CudaError & e) { return fail(PTC_E_CUDA, e.what()); }             \
  catch (std::bad_alloc & e) { return fail(PTC_E_NOMEM, e.what()); }       \
  catch (std::logic_error & e) {                                           \
    return fail(dynamic_cast<std::invalid_argument *>(&e) ? PTC_E_INVALID : PTC_E_STATE, e.what()); \
  }                                                                        \
  catch (std::exception & e) { return fail(PTC_E_INVALID, e.what()); }

}  // namespace

// Device image -> caller's host buffer.  A copy straight into pageable memory runs at ~5 GB/s (C5's 99.5 MB film: 20 ms,
// as long as a quarter of the 8-GPU render); through a pinned staging buffer the PCIe leg runs at link speed and the
// host-side copy is split over a few threads.
void film_to_host(ptc_scene *s, const void *d_src, void *dst, size_t bytes, cudaStream_t stream) {
  if (bytes < ((size_t)8 << 20)) {
    CK(cudaMemcpyAsync(dst, d_src, bytes, cudaMemcpyDeviceToHost, stream));
    CK(cudaStreamSynchronize(stream));
    return;
  }
  if (s->h_film_bytes < bytes) {
    if (s->h_film) cudaFreeHost(s->h_film);
    s->h_film = nullptr, s->h_film_bytes = 0;
    CK(cudaMallocHost(&s->h_film, bytes));
    s->h_film_bytes = bytes;
  }
  CK(cudaMemcpyAsync(s->h_film, d_src, bytes, cudaMemcpyDeviceToHost, stream));
  CK(cudaStreamSynchronize(stream));
  const int nt = (int)std::min<size_t>(8, std::max<size_t>(1, std::thread::hardware_concurrency()));
  std::vector<std::thread> th;
  const size_t per = (bytes + (size_t)nt - 1) / (size_t)nt;
  for (int t = 0; t < nt; t++) {
    const size_t a = (size_t)t * per, b = std::min(bytes, a + per);
    if (a >= b) break;
    th.emplace_back([=] { memcpy(static_cast<char *>(dst) + a, s->h_film + a, b - a); });
  }
  for (auto &t : th) t.join();
}

// The scene's film -> the caller's host images, the one way every render that returns an image ends: k_resolve_film
// into the staging buffers, then whichever of out_rgb (W*H*3 linear mean radiance) and out_u32 (W*H 0x00RRGGBB) is not
// nullptr to the host.  counts == nullptr: every pixel x scale, else x 1 / counts[p].  `resolved`, if given, is recorded
// once the resolve is done, before the copies.  Returns, with all the work queued on `stream` done (the event included,
// also when no image is asked for), the number of kernels launched.
int resolve_film_to_host(ptc_scene *s, size_t n_px, float scale, const int32_t *counts, float *out_rgb, uint32_t *out_u32,
                         cudaStream_t stream, cudaEvent_t resolved = nullptr) {
  if (out_rgb && s->w_film_out.n < n_px * 3) s->w_film_out.alloc(n_px * 3);
  if (out_u32 && s->w_packed.n < n_px) s->w_packed.alloc(n_px);
  const int launches = (out_rgb || out_u32) ? 1 : 0;
  if (launches) {
    k_resolve_film<<<(unsigned)((n_px + 255) / 256), 256, 0, stream>>>(s->film(), n_px, scale, counts, out_rgb ? s->w_film_out.p : nullptr,
                                                                       out_u32 ? s->w_packed.p : nullptr);
    CK(cudaGetLastError());
  }
  if (resolved) CK(cudaEventRecord(resolved, stream));
  if (out_u32) film_to_host(s, s->w_packed.p, out_u32, n_px * sizeof(uint32_t), stream);
  if (out_rgb) film_to_host(s, s->w_film_out.p, out_rgb, n_px * 3 * sizeof(float), stream);
  CK(cudaStreamSynchronize(stream));
  return launches;
}

// Device half of commit: upload the flattened scene `hs` (built) to `device` and fill s->ds.  `s` may be the handle that
// owns `hs` (ptc_scene_commit) or a replica that only holds device state (ptc_multi_create).
void upload_scene(ptc_scene *s, const HostScene &hs, int device) {
  CK(cudaSetDevice(device));
  s->device = device;
  cudaDeviceProp prop;
  CK(cudaGetDeviceProperties(&prop, device));
  s->sm_count = prop.multiProcessorCount;
  std::vector<DMesh> dm;
  for (size_t mi = 0; mi < hs.meshes.size(); mi++) {
    auto &m = hs.meshes[mi];
    auto nodes = std::make_unique<DevBuf<float4>>();
    auto tris = std::make_unique<DevBuf<float4>>();
    auto nrm = std::make_unique<DevBuf<float4>>();
    if (mi < s->dev_built.size() && s->dev_built[mi].device == device && s->dev_built[mi].nodes) {
      // the device-side builder left the arrays on this very device: adopt them instead of uploading the host copies
      DevMeshBuffers &b = s->dev_built[mi];
      nodes->p = static_cast<float4 *>(b.nodes), nodes->n = m->nodes.size() * 5;
      tris->p = static_cast<float4 *>(b.tris), tris->n = m->tri48.size() * 3;
      nrm->p = static_cast<float4 *>(b.normals), nrm->n = m->normals.size();
      b = DevMeshBuffers();
    } else {
      nodes->upload(reinterpret_cast<const float4 *>(m->nodes.data()), m->nodes.size() * 5);
      tris->upload(reinterpret_cast<const float4 *>(m->tri48.data()), m->tri48.size() * 3);
      nrm->upload(m->normals.data(), m->normals.size());
    }
    const DMesh d = make_dmesh(*m, nodes->p, tris->p, nrm->p);
    dm.push_back(d);
    s->mesh_bufs.push_back(std::move(nodes));
    s->mesh_bufs.push_back(std::move(tris));
    s->mesh_bufs.push_back(std::move(nrm));
  }
  s->d_objects.upload(hs.objects.data(), hs.objects.size());
  s->d_materials.upload(hs.materials.data(), hs.materials.size());
  s->d_meshes.upload(dm.data(), dm.size());
  if (!hs.sky.empty()) s->d_sky.upload(hs.sky.data(), hs.sky.size());
  s->ds.objects = s->d_objects.p;
  s->ds.materials = s->d_materials.p;
  s->ds.meshes = s->d_meshes.p;
  s->ds.sky = hs.sky.empty() ? nullptr : s->d_sky.p;
  s->d_lights.upload(hs.lights.data(), hs.lights.size());
  s->ds.lights = s->d_lights.p;
  if (!hs.sky_dist.empty()) s->d_sky_dist.upload(hs.sky_dist.data(), hs.sky_dist.size());
  s->ds.sky_dist = hs.sky_dist.empty() ? nullptr : s->d_sky_dist.p;
  s->ds.n_lights = (int32_t)hs.lights.size();
  s->ds.n_objects = (int32_t)hs.objects.size();
  s->ds.n_materials = (int32_t)hs.materials.size();
  s->ds.n_meshes = (int32_t)dm.size();
  s->ds.sky_w = hs.sky_w;
  s->ds.sky_h = hs.sky_h;
  s->d_objects_em.upload(hs.objects_em.data(), hs.objects_em.size());
  s->d_lights_em.upload(hs.lights_em.data(), hs.lights_em.size());
  s->d_em_sel_cdf.upload(hs.em_sel_cdf.data(), hs.em_sel_cdf.size());
  s->d_em_ent.upload(hs.em_ent.data(), hs.em_ent.size());
  s->d_em_ent_cdf.upload(hs.em_ent_cdf.data(), hs.em_ent_cdf.size());
  s->ds_em = s->ds;
  s->ds_em.objects = s->d_objects_em.p;
  s->ds_em.lights = s->d_lights_em.p;
  s->ds_em.n_lights = (int32_t)hs.lights_em.size();
  s->et = EmitterTables{s->d_em_sel_cdf.p, s->d_em_ent.p, s->d_em_ent_cdf.p};
  s->mesh_objects = 0;
  for (const DObject &o : hs.objects)
    if (o.type == OBJ_MESH) s->mesh_objects++;
  CK(cudaStreamCreateWithFlags(&s->own_stream, cudaStreamNonBlocking));
  s->committed = true;
}

// ---- in-process multi-GPU (ptc_multi_*): scene replicated per device, work sharded, the films reduced by NCCL ----
// NCCL is bound at run time: a process that also hosts PyTorch must end up with ONE libnccl (dlopen by soname returns
// the copy that is already loaded), and processes that never call ptc_multi_create never load it.
struct NcclApi {
  void *lib = nullptr;
  ncclResult_t (*GetVersion)(int *) = nullptr;
  ncclResult_t (*CommInitAll)(ncclComm_t *, int, const int *) = nullptr;
  ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
  ncclResult_t (*CommAbort)(ncclComm_t) = nullptr;
  ncclResult_t (*Reduce)(const void *, void *, size_t, ncclDataType_t, ncclRedOp_t, int, ncclComm_t, cudaStream_t) = nullptr;
  const char *(*GetErrorString)(ncclResult_t) = nullptr;
  void load() {
    if (lib) return;
    for (const char *name : {"libnccl.so.2", "libnccl.so"}) {
      lib = dlopen(name, RTLD_NOW | RTLD_LOCAL);
      if (lib) break;
    }
    if (!lib) throw std::runtime_error(std::string("NCCL not found: ") + dlerror());
    auto sym = [&](const char *n) {
      void *p = dlsym(lib, n);
      if (!p) throw std::runtime_error(std::string("NCCL symbol missing: ") + n);
      return p;
    };
    GetVersion = reinterpret_cast<decltype(GetVersion)>(sym("ncclGetVersion"));
    CommInitAll = reinterpret_cast<decltype(CommInitAll)>(sym("ncclCommInitAll"));
    CommDestroy = reinterpret_cast<decltype(CommDestroy)>(sym("ncclCommDestroy"));
    CommAbort = reinterpret_cast<decltype(CommAbort)>(sym("ncclCommAbort"));
    Reduce = reinterpret_cast<decltype(Reduce)>(sym("ncclReduce"));
    GetErrorString = reinterpret_cast<decltype(GetErrorString)>(sym("ncclGetErrorString"));
  }
  void check(ncclResult_t r, const char *what) const {
    if (r != ncclSuccess) throw CudaError(std::string(what) + ": " + (GetErrorString ? GetErrorString(r) : "NCCL error"));
  }
};

struct ptc_multi {
  ptc_scene *primary = nullptr;                     // devices[0]; not owned
  std::vector<std::unique_ptr<ptc_scene>> replicas;  // devices[1..]: device state only
  std::vector<ptc_scene *> scenes;
  std::vector<int> devices;
  std::vector<ncclComm_t> comms;  // empty for one device
  bool comms_dead = false;        // a failed render aborted the communicators: the next call creates new ones
  NcclApi nccl;
  void init_comms() {
    comms.assign(devices.size(), nullptr);
    nccl.check(nccl.CommInitAll(comms.data(), (int)devices.size(), devices.data()), "ncclCommInitAll");
    comms_dead = false;
  }
  void abort_comms() {  // unblocks every rank that waits inside the collective
    for (size_t i = 0; i < comms.size(); i++)
      if (comms[i]) nccl.CommAbort(comms[i]), comms[i] = nullptr;
    comms_dead = true;
  }
  ~ptc_multi() {
    for (size_t i = 0; i < comms.size(); i++) {
      cudaSetDevice(devices[i]);
      if (comms[i]) nccl.CommDestroy(comms[i]);
    }
  }
};

// =============================================================================================================
extern "C" {

const char *ptc_last_error(void) { return g_err.c_str(); }
int ptc_abi_version(void) { return PTC_ABI_VERSION; }
int ptc_device_count(void) {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess) {
    cudaGetLastError();
    return 0;
  }
  return n;
}

ptc_scene *ptc_scene_create(void) {
  try {
    return new ptc_scene();
  } catch (std::exception &e) {
    g_err = e.what();
    return nullptr;
  }
}
void ptc_scene_destroy(ptc_scene *s) { delete s; }

int ptc_scene_add_material(ptc_scene *s, const ptc_material *m) {
  PTC_GUARD_BEGIN
  if (!s || !m) throw std::invalid_argument("null argument");
  if (s->committed) throw std::logic_error("scene already committed");
  return s->hs.add_material(m);
  PTC_GUARD_END
}
int ptc_scene_add_sphere(ptc_scene *s, const float c[3], float radius, int material) {
  PTC_GUARD_BEGIN
  if (!s || !c) throw std::invalid_argument("null argument");
  if (s->committed) throw std::logic_error("scene already committed");
  return s->hs.add_sphere(c, radius, material);
  PTC_GUARD_END
}
int ptc_scene_add_plane(ptc_scene *s, const float p1[3], const float n[3], int material) {
  PTC_GUARD_BEGIN
  if (!s || !p1 || !n) throw std::invalid_argument("null argument");
  if (s->committed) throw std::logic_error("scene already committed");
  return s->hs.add_plane(p1, n, material);
  PTC_GUARD_END
}
int ptc_scene_add_quad(ptc_scene *s, const float base[3], const float e0[3], const float e1[3], const float n[3], float d,
                       float inv0, float inv1, int material) {
  PTC_GUARD_BEGIN
  if (!s || !base || !e0 || !e1 || !n) throw std::invalid_argument("null argument");
  if (s->committed) throw std::logic_error("scene already committed");
  return s->hs.add_quad(base, e0, e1, n, d, inv0, inv1, material);
  PTC_GUARD_END
}
int ptc_scene_add_cube(ptc_scene *s, const float o2w[16], const float w2o[16], int material) {
  PTC_GUARD_BEGIN
  if (!s || !o2w || !w2o) throw std::invalid_argument("null argument");
  if (s->committed) throw std::logic_error("scene already committed");
  return s->hs.add_cube(o2w, w2o, material);
  PTC_GUARD_END
}
int ptc_scene_add_mesh(ptc_scene *s, const float *tris, int64_t n, const float o2w[16], const float w2o[16], int material) {
  PTC_GUARD_BEGIN
  if (!s || !o2w || !w2o) throw std::invalid_argument("null argument");
  if (s->committed) throw std::logic_error("scene already committed");
  return s->hs.add_mesh(tris, n, o2w, w2o, material);
  PTC_GUARD_END
}
int ptc_scene_set_sky_hdr(ptc_scene *s, const float *rgb, int32_t w, int32_t h) {
  PTC_GUARD_BEGIN
  if (!s) throw std::invalid_argument("null argument");
  if (s->committed) throw std::logic_error("scene already committed");
  s->hs.set_sky(rgb, w, h);
  return 0;
  PTC_GUARD_END
}

int ptc_scene_set_lens(ptc_scene *s, const ptc_lens *lenses, int32_t n) {
  PTC_GUARD_BEGIN
  if (!s || n < 0 || (n > 0 && !lenses)) throw std::invalid_argument("bad argument");
  for (int32_t k = 0; k < n; k++) {
    const float r = lenses[k].aperture_radius, f = lenses[k].focus_distance;
    if (!(r >= 0.0f) || !std::isfinite(r)) throw std::invalid_argument("aperture_radius must be >= 0 and finite");
    if (!(f > 0.0f) || !std::isfinite(f)) throw std::invalid_argument("focus_distance must be > 0 and finite");
  }
  s->lens.assign(lenses, lenses + n);
  return 0;
  PTC_GUARD_END
}

int ptc_scene_set_object_motion(ptc_scene *s, int32_t object, const float displacement[3]) {
  PTC_GUARD_BEGIN
  if (!s || !displacement) throw std::invalid_argument("null argument");
  if (object < 0 || (size_t)object >= s->hs.objects.size()) throw std::invalid_argument("object index out of range");
  for (int c = 0; c < 3; c++)
    if (!std::isfinite(displacement[c])) throw std::invalid_argument("displacement must be finite");
  if (s->motion.size() <= (size_t)object) s->motion.resize((size_t)object + 1, make_float4(0.0f, 0.0f, 0.0f, 0.0f));
  s->motion[(size_t)object] = make_float4(displacement[0], displacement[1], displacement[2], 0.0f);
  return 0;
  PTC_GUARD_END
}

int ptc_scene_set_camera_motion(ptc_scene *s, const ptc_camera *end_cameras, int32_t n) {
  PTC_GUARD_BEGIN
  if (!s || n < 0 || (n > 0 && !end_cameras)) throw std::invalid_argument("bad argument");
  for (int32_t k = 0; k < n; k++) {
    float f[sizeof(ptc_camera) / sizeof(float)];  // ptc_camera is floats only
    static_assert(sizeof(f) == sizeof(ptc_camera), "ptc_camera is floats only");
    memcpy(f, &end_cameras[k], sizeof(f));
    for (float v : f)
      if (!std::isfinite(v)) throw std::invalid_argument("every field of an end camera must be finite");
  }
  s->end_cams.assign(end_cameras, end_cameras + n);
  return 0;
  PTC_GUARD_END
}

int ptc_scene_build(ptc_scene *s) {
  PTC_GUARD_BEGIN
  if (!s) throw std::invalid_argument("null argument");
  s->hs.build_all();
  return 0;
  PTC_GUARD_END
}

int ptc_scene_commit(ptc_scene *s, int device) { return ptc_scene_commit_ex(s, device, 0); }

int ptc_scene_commit_ex(ptc_scene *s, int device, int flags) {
  PTC_GUARD_BEGIN
  if (!s) throw std::invalid_argument("null argument");
  if (s->committed) throw std::logic_error("scene already committed");
  if ((flags & PTC_COMMIT_FAST_BUILD) && (flags & PTC_COMMIT_DEVICE_SAH))
    throw std::invalid_argument("PTC_COMMIT_FAST_BUILD and PTC_COMMIT_DEVICE_SAH exclude each other");
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess || n == 0) {
    cudaGetLastError();
    throw CudaError("no CUDA device available (this library has no CPU fallback)");
  }
  if (device < 0 || device >= n) throw std::invalid_argument("device index out of range");
  // Flattening.  Step 1 (restating the reference's BVH build for the dead mask and the DFS order) runs ON the device for
  // large meshes: 10-30 ms instead of ~400 ms for 2 M triangles.  The traversal tree then comes from the host's SAH +
  // dynamic-programming collapse by default — the better tree: C5 renders 22 % faster through it than through the
  // device-built one — or, with PTC_COMMIT_FAST_BUILD / PTC_BUILD=device, from the device too (the reference tree itself,
  // re-used as the wide tree: the whole commit of 2 M triangles in ~0.2 s).  PTC_COMMIT_DEVICE_SAH / PTC_BUILD=device-sah
  // builds the host's SAH tree on the device, for meshes of every size.  PTC_BUILD=host keeps everything on the host;
  // a non-default tie order (PTC_REF_TIE, a measurement switch) exists on the host only.
  {
    const char *mode = getenv("PTC_BUILD"), *tie = getenv("PTC_REF_TIE");
    const bool tie_default = !tie || !*tie || !strcmp(tie, "stable");
    const bool force_host = mode && !strcmp(mode, "host");
    const bool sah = (mode && !strcmp(mode, "device-sah")) || (flags & PTC_COMMIT_DEVICE_SAH) != 0;
    const bool fast = !sah && ((mode && !strcmp(mode, "device")) || (flags & PTC_COMMIT_FAST_BUILD) != 0);
    const DevBuildMode dev_mode = sah ? DevBuildMode::Sah : (fast ? DevBuildMode::Median : DevBuildMode::RefOnly);
    s->dev_built.assign(s->hs.meshes.size(), DevMeshBuffers());
    for (size_t mi = 0; mi < s->hs.meshes.size(); mi++) {
      MeshBuild &mb = *s->hs.meshes[mi];
      if (mb.built || force_host || !tie_default || mb.n >= ((int64_t)1 << 27)) continue;  // (the device builder's index width)
      if (dev_mode == DevBuildMode::RefOnly && mb.n < kDeviceRefMinTriangles) continue;
      CK(cudaSetDevice(device));
      DevBuildTiming tm;
      build_mesh_device(mb, s->dev_built[mi], &tm, dev_mode);
      if (getenv("PTC_BUILD_TIMING"))
        fprintf(stderr, "[pt_build_dev] %lld triangles (%lld live)%s: upload %.1f ms, reference-BVH restatement %.1f ms (%d levels), "
                        "binned SAH %.1f ms (%d levels), collapse plan %.1f ms, structure %.1f ms, "
                        "boxes + nodes + triangle records %.1f ms, download %.1f ms, total %.1f ms; %zu wide nodes, depth %d\n",
                (long long)mb.n, (long long)mb.live, dev_mode == DevBuildMode::RefOnly ? " [step 1 only]" : (sah ? " [SAH]" : ""), tm.upload_ms,
                tm.ref_ms, tm.ref_levels, tm.sah_ms, tm.sah_levels, tm.plan_ms, tm.structure_ms, tm.emit_ms, tm.download_ms, tm.total_ms,
                mb.nodes.size(), mb.wide_depth);
    }
  }
  const auto t_host = std::chrono::steady_clock::now();
  s->hs.build_all();  // host flattening of what is left: reference-BVH dead mask -> SAH -> 8-wide quantised BVH
  const auto t_up = std::chrono::steady_clock::now();
  upload_scene(s, s->hs, device);
  if (getenv("PTC_BUILD_TIMING"))
    fprintf(stderr, "[ptc_scene_commit] host flattening %.1f ms, upload %.1f ms\n", std::chrono::duration<double, std::milli>(t_up - t_host).count(),
            std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_up).count());
  return 0;
  PTC_GUARD_END
}

int64_t ptc_scene_last_pool_slots(const ptc_scene *s) { return s ? s->last_pool_slots : 0; }

int ptc_scene_mesh_info(const ptc_scene *s, int object, ptc_mesh_info *info, uint8_t *dead, int32_t *order) {
  PTC_GUARD_BEGIN
  if (!s) throw std::invalid_argument("null argument");
  if (object < 0 || (size_t)object >= s->hs.objects.size() || s->hs.objects[(size_t)object].type != OBJ_MESH)
    throw std::invalid_argument("object is not a mesh");
  const MeshBuild &m = *s->hs.meshes[(size_t)s->hs.objects[(size_t)object].mesh];
  if (!m.built) throw std::logic_error("mesh not built yet (call ptc_scene_build or ptc_scene_commit first)");
  if (info) {
    info->triangles = m.n;
    info->live_triangles = m.live;
    info->ref_nodes = m.ref_nodes;
    info->ref_leaves = m.ref_leaves;
    info->ref_depth = m.ref_depth;
    info->wide_nodes = (int64_t)m.nodes.size();
    info->wide_depth = m.wide_depth;
    info->node_bytes = (int64_t)m.nodes.size() * (int64_t)sizeof(Node8);
    info->triangle_bytes = (int64_t)m.tri48.size() * (int64_t)sizeof(Tri48);
  }
  if (dead) memcpy(dead, m.dead.data(), (size_t)m.n);
  if (order) memcpy(order, m.order.data(), (size_t)m.n * sizeof(int32_t));
  return 0;
  PTC_GUARD_END
}

int ptc_render_accumulate(ptc_scene *s, const ptc_camera *cam, const ptc_render_settings *st, float *d_accum,
                          void *cuda_stream, ptc_stats *stats) {
  PTC_GUARD_BEGIN
  if (!s) throw std::invalid_argument("null argument");
  const ptc_lens *lens = single_lens(s);
  const ptc_camera *end = single_end_cam(s);
  require_committed(s);
  check_render_args(cam, st, d_accum != nullptr);
  // the caller's handle is honoured as given: NULL is the legacy default stream, which orders the film atomics after
  // whatever the caller queued there (a memset of d_accum, a wait on a collective)
  Pass pass;
  if (lens) {
    CK(cudaSetDevice(s->device));
    pass.lens = upload_lens(s, lens, 1, (cudaStream_t)cuda_stream);
  }
  const MotionCall mc = single_motion(s, cam, end);
  if (mc.any()) {
    CK(cudaSetDevice(s->device));
    upload_motion(s, mc, (cudaStream_t)cuda_stream, pass);
  }
  render_accumulate(s, cam, st, d_accum, (cudaStream_t)cuda_stream, stats, pass);
  return 0;
  PTC_GUARD_END
}

// ptc_render (out_rgb) and ptc_render_u32 (out_u32): the render into the scene's film, then one resolve of it with the
// 1/spp of renderer.rs:85 — only the asked-for image crosses PCIe
static int render_to_host(ptc_scene *s, const ptc_camera *cam, const ptc_render_settings *st, float *out_rgb, uint32_t *out_u32,
                          ptc_stats *stats) {
  PTC_GUARD_BEGIN
  if (!s) throw std::invalid_argument("null argument");
  const ptc_lens *lens = single_lens(s);
  const ptc_camera *end = single_end_cam(s);
  require_committed(s);
  check_render_args(cam, st, out_rgb || out_u32);
  Pass pass;
  if (lens) {
    CK(cudaSetDevice(s->device));
    pass.lens = upload_lens(s, lens, 1, s->own_stream);
  }
  const MotionCall mc = single_motion(s, cam, end);
  if (mc.any()) {
    CK(cudaSetDevice(s->device));
    upload_motion(s, mc, s->own_stream, pass);
  }
  render_accumulate(s, cam, st, nullptr, s->own_stream, stats, pass);
  const int launches = resolve_film_to_host(s, (size_t)st->width * st->height, 1.0f / (float)st->spp, nullptr, out_rgb, out_u32, s->own_stream);
  if (stats) stats->kernel_launches += launches;
  return 0;
  PTC_GUARD_END
}

int ptc_render(ptc_scene *s, const ptc_camera *cam, const ptc_render_settings *st, float *out_rgb, ptc_stats *stats) {
  return render_to_host(s, cam, st, out_rgb, nullptr, stats);
}

int ptc_render_u32(ptc_scene *s, const ptc_camera *cam, const ptc_render_settings *st, uint32_t *out_u32, ptc_stats *stats) {
  return render_to_host(s, cam, st, nullptr, out_u32, stats);
}

// ptc_render_batch / ptc_render_batch_accumulate: the arguments, before the scene's state
static void check_batch_args(const ptc_scene *s, const ptc_camera *cams, int32_t n_views, const ptc_render_settings *st, bool has_output) {
  check_render_args(cams, st, has_output);
  if (n_views < 1) throw std::invalid_argument("n_views must be >= 1");
  if (s->lens.size() > 1 && s->lens.size() != (size_t)n_views)
    throw std::invalid_argument("ptc_scene_set_lens gave n lenses: a batch needs n == 1 or n == n_views");
  if (s->end_cams.size() > 1 && s->end_cams.size() != (size_t)n_views)
    throw std::invalid_argument("ptc_scene_set_camera_motion gave n end cameras: a batch needs n == 1 or n == n_views");
  if (st->tile_mod != 0) throw std::invalid_argument("ptc_render_batch renders whole views: tile_mod must be 0");
  // the film index of every padded pixel of every view stays below 2^30 (a pool entry's pixel word keeps kShadowBit)
  const uint64_t padded = (uint64_t)n_views * (((uint64_t)st->width + 31u) & ~31ull) * (((uint64_t)st->height + 31u) & ~31ull);
  if (padded > (1ull << 30)) throw std::invalid_argument("batch too large: n_views * ceil32(width) * ceil32(height) > 2^30");
}

// The batch's cameras and seeds (seeds == NULL: settings->seed for every view) into the scene's device tables, one copy
// each on the stream the render runs on; -> the Pass that renders them.
static Pass batch_pass(ptc_scene *s, const ptc_camera *cams, int32_t n_views, const uint64_t *seeds, const ptc_render_settings *st,
                       cudaStream_t stream) {
  static_assert(sizeof(ptc_camera) == sizeof(DCamera), "ptc_camera and DCamera share one layout");
  CK(cudaSetDevice(s->device));
  const size_t n = (size_t)n_views;
  if (s->d_batch_cams.n < n) s->d_batch_cams.alloc(n), s->d_batch_seeds.alloc(n);
  std::vector<uint64_t> same;
  if (!seeds) same.assign(n, st->seed), seeds = same.data();
  // (from pageable memory: the call returns once the source has been read)
  CK(cudaMemcpyAsync(s->d_batch_cams.p, cams, n * sizeof(DCamera), cudaMemcpyHostToDevice, stream));
  CK(cudaMemcpyAsync(s->d_batch_seeds.p, seeds, n * sizeof(uint64_t), cudaMemcpyHostToDevice, stream));
  Pass pass;
  pass.views = (uint32_t)n_views, pass.cams = s->d_batch_cams.p, pass.seeds = s->d_batch_seeds.p;
  if (!s->lens.empty()) {  // one lens for every view, or one per view
    std::vector<ptc_lens> per(n, s->lens[0]);
    if (s->lens.size() == n) per = s->lens;
    pass.lens = upload_lens(s, per.data(), n, stream);
  }
  // one end camera for every view, or one per view
  upload_motion(s, motion_call(s, cams, n, s->end_cams.data(), s->end_cams.size()), stream, pass);
  return pass;
}

int ptc_render_batch(ptc_scene *s, const ptc_camera *cams, int32_t n_views, const uint64_t *seeds, const ptc_render_settings *st,
                     float *out_rgb, uint32_t *out_u32, ptc_stats *stats) {
  PTC_GUARD_BEGIN
  // the arguments first, the scene's state after them
  if (!s) throw std::invalid_argument("null argument");
  check_batch_args(s, cams, n_views, st, out_rgb || out_u32);
  require_committed(s);
  const Pass pass = batch_pass(s, cams, n_views, seeds, st, s->own_stream);
  render_accumulate(s, cams, st, nullptr, s->own_stream, stats, pass);
  const size_t n_px = (size_t)n_views * st->width * st->height;
  const int launches = resolve_film_to_host(s, n_px, 1.0f / (float)st->spp, nullptr, out_rgb, out_u32, s->own_stream);  // as ptc_render
  if (stats) stats->kernel_launches += launches;
  return 0;
  PTC_GUARD_END
}

int ptc_render_batch_accumulate(ptc_scene *s, const ptc_camera *cams, int32_t n_views, const uint64_t *seeds, const ptc_render_settings *st,
                                float *d_accum, void *cuda_stream, ptc_stats *stats) {
  PTC_GUARD_BEGIN
  if (!s) throw std::invalid_argument("null argument");
  check_batch_args(s, cams, n_views, st, d_accum != nullptr);
  require_committed(s);
  const Pass pass = batch_pass(s, cams, n_views, seeds, st, (cudaStream_t)cuda_stream);
  render_accumulate(s, cams, st, d_accum, (cudaStream_t)cuda_stream, stats, pass);
  return 0;
  PTC_GUARD_END
}

int ptc_render_adaptive(ptc_scene *s, const ptc_camera *cam, const ptc_render_settings *st, const ptc_adaptive *ad, float *out_rgb,
                        uint32_t *out_u32, int32_t *out_spp, ptc_stats *stats) {
  PTC_GUARD_BEGIN
  // the arguments first, the scene's state after them
  if (!s || !ad) throw std::invalid_argument("null argument");
  check_render_args(cam, st, true);  // every output may be NULL
  if (st->sample_begin != 0 || st->sample_end != 0 || st->tile_mod != 0)
    throw std::invalid_argument("ptc_render_adaptive schedules the samples itself: sample_begin, sample_end and tile_mod must be 0");
  if (ad->min_spp < 2 || ad->min_spp % 2 != 0 || ad->min_spp > st->spp) throw std::invalid_argument("min_spp must be even, >= 2 and <= spp");
  if (!(ad->threshold >= 0.0f)) throw std::invalid_argument("threshold must be >= 0");
  const ptc_lens *lens = single_lens(s);
  const ptc_camera *end = single_end_cam(s);
  require_committed(s);
  CK(cudaSetDevice(s->device));
  ensure_ctl(s);
  const uint32_t n_px = (uint32_t)st->width * (uint32_t)st->height;
  if (s->w_adapt_vp.n < (size_t)n_px * 3) s->w_adapt_vp.alloc((size_t)n_px * 3);
  if (s->w_adapt_needs.n < n_px) s->w_adapt_needs.alloc(n_px), s->w_adapt_keep.alloc(n_px), s->w_adapt_spp.alloc(n_px);
  for (auto &l : s->w_adapt_list)
    if (l.n < n_px) l.alloc(n_px);
  if (!s->w_adapt_n.p) s->w_adapt_n.alloc(1);
  size_t tmp_bytes = 0;
  CK(cub::DeviceSelect::Flagged(nullptr, tmp_bytes, (const uint32_t *)nullptr, (const uint8_t *)nullptr, (uint32_t *)nullptr,
                                (uint32_t *)nullptr, (int)n_px));
  if (s->w_adapt_tmp.n < tmp_bytes) s->w_adapt_tmp.alloc(tmp_bytes);
  cudaStream_t stream = s->own_stream;
  const unsigned nb = (n_px + 255u) / 256u;

  ptc_stats total;
  memset(&total, 0, sizeof(total));
  uint64_t &launches = total.kernel_launches;

  // passes 0 and 1 over the tiles, the snapshot between them
  const int half = ad->min_spp / 2;
  Pass first;
  first.lens = lens ? upload_lens(s, lens, 1, stream) : nullptr;
  upload_motion(s, single_motion(s, cam, end), stream, first);
  CK(cudaEventRecord(s->ev_adapt_begin, stream));
  render_pass(s, cam, st, 0, half, first, stream, total);
  const Film f = s->film();
  float *vp = s->w_adapt_vp.p;
  CK(cudaMemsetAsync(vp, 0, (size_t)n_px * 3 * sizeof(float), stream));
  k_film_to_accum<<<(unsigned)(((size_t)n_px * 3 + 255) / 256), 256, 0, stream>>>(f, n_px, vp);
  launches += 1;
  Pass more = first;
  more.clear_film = false;
  render_pass(s, cam, st, half, ad->min_spp, more, stream, total);
  k_adapt_init<<<nb, 256, 0, stream>>>(n_px, st->spp, s->w_adapt_list[0].p, s->w_adapt_needs.p, s->w_adapt_spp.p);
  launches += 1;
  CK(cudaGetLastError());

  // decision, then a pass over the pixels that stay, until none stays or they have all reached spp
  uint32_t n_list = n_px;
  int cur = 0, n = ad->min_spp, m = half;
  while (n < st->spp) {
    const uint32_t *list = s->w_adapt_list[cur].p;
    const unsigned lb = (n_list + 255u) / 256u;
    k_adapt_decide<<<lb, 256, 0, stream>>>(f, list, n_list, n, m, ad->threshold, vp, s->w_adapt_needs.p);
    k_adapt_keep<<<lb, 256, 0, stream>>>(list, n_list, s->w_adapt_needs.p, st->width, st->height, s->w_adapt_keep.p);
    k_adapt_leave<<<lb, 256, 0, stream>>>(list, n_list, s->w_adapt_keep.p, n, s->w_adapt_needs.p, s->w_adapt_spp.p);
    CK(cudaGetLastError());
    size_t tb = s->w_adapt_tmp.n;
    CK(cub::DeviceSelect::Flagged(s->w_adapt_tmp.p, tb, list, s->w_adapt_keep.p, s->w_adapt_list[cur ^ 1].p, s->w_adapt_n.p,
                                  (int)n_list, stream));  // stable: the next list is ascending again
    launches += 5;
    uint32_t kept = 0;
    CK(cudaMemcpyAsync(&kept, s->w_adapt_n.p, sizeof(uint32_t), cudaMemcpyDeviceToHost, stream));
    CK(cudaStreamSynchronize(stream));
    n_list = kept, cur ^= 1;
    if (n_list == 0) break;
    more.pixels = s->w_adapt_list[cur].p, more.n_pixels = n_list;
    const int next = adapt_next_end(n, st->spp);
    render_pass(s, cam, st, n, next, more, stream, total);
    m = n, n = next;
  }

  // one resolve of every pixel at its own count (the scale is unused), the end of render_ms
  launches += resolve_film_to_host(s, n_px, 1.0f, s->w_adapt_spp.p, out_rgb, out_u32, stream, s->ev_adapt_end);
  if (out_spp) film_to_host(s, s->w_adapt_spp.p, out_spp, (size_t)n_px * sizeof(int32_t), stream);
  if (stats) {
    *stats = total;
    float ms = 0.0f;
    CK(cudaEventElapsedTime(&ms, s->ev_adapt_begin, s->ev_adapt_end));
    stats->render_ms = ms;
  }
  return 0;
  PTC_GUARD_END
}

// ptc_render_progressive's schedule: the samples after pass j + 1, given n after pass j
static int progressive_next(int n, int spp, int max_pass_spp) {
  const int64_t step = max_pass_spp > 0 ? std::min(n, max_pass_spp) : n;
  return (int)std::min<int64_t>((int64_t)n + step, spp);
}

int ptc_render_progressive(ptc_scene *s, const ptc_camera *cam, const ptc_render_settings *st, const ptc_progressive *pg,
                           ptc_preview_fn on_preview, void *user, float *out_rgb, uint32_t *out_u32, int32_t *out_samples,
                           ptc_stats *stats) {
  PTC_GUARD_BEGIN
  // the arguments first, the scene's state after them
  if (!s || !pg) throw std::invalid_argument("null argument");
  check_render_args(cam, st, true);  // every output may be NULL
  if (st->sample_begin != 0 || st->sample_end != 0 || st->tile_mod != 0)
    throw std::invalid_argument("ptc_render_progressive schedules the samples itself: sample_begin, sample_end and tile_mod must be 0");
  if (pg->first_spp < 1 || pg->first_spp > st->spp) throw std::invalid_argument("first_spp must be >= 1 and <= spp");
  if (pg->max_pass_spp < 0) throw std::invalid_argument("max_pass_spp must be >= 0");
  const ptc_lens *lens = single_lens(s);
  const ptc_camera *end = single_end_cam(s);
  require_committed(s);
  CK(cudaSetDevice(s->device));
  ensure_ctl(s);
  const size_t n_px = (size_t)st->width * st->height;
  for (int k = 0; k < 2; k++) {
    if (s->w_prog_packed[k].n < n_px) s->w_prog_packed[k].alloc(n_px);
    if (out_rgb && s->w_prog_rgb[k].n < n_px * 3) s->w_prog_rgb[k].alloc(n_px * 3);
    if (!s->ev_prog_slot[k]) CK(cudaEventCreate(&s->ev_prog_slot[k]));
  }
  if (!s->ev_prog_begin) CK(cudaEventCreate(&s->ev_prog_begin));
  if (!s->preview_stream) CK(cudaStreamCreateWithFlags(&s->preview_stream, cudaStreamNonBlocking));
  if (on_preview && s->h_preview_px < n_px) {
    if (s->h_preview) cudaFreeHost(s->h_preview);
    s->h_preview = nullptr, s->h_preview_px = 0;
    CK(cudaMallocHost(&s->h_preview, n_px * sizeof(uint32_t)));
    s->h_preview_px = n_px;
  }
  cudaStream_t stream = s->own_stream;
  const float2 *d_lens = lens ? upload_lens(s, lens, 1, stream) : nullptr;
  Pass moving;  // the motion tables of every pass
  upload_motion(s, single_motion(s, cam, end), stream, moving);

  // What the two threads share, under `mu`.  The worker publishes pass j (ready = j + 1, samples[j % 2]) once its slot
  // event is recorded; the calling thread publishes callback j's return (shown = j + 1) and a stop.
  std::mutex mu;
  std::condition_variable cv;
  int ready = 0, shown = 0;
  int32_t samples[2] = {0, 0};
  bool stop = false, worker_done = false;
  std::exception_ptr worker_error;
  ptc_stats total;
  memset(&total, 0, sizeof(total));
  cudaEvent_t last_slot_event = nullptr;

  auto worker = [&]() {
    try {
      CK(cudaSetDevice(s->device));
      CK(cudaEventRecord(s->ev_prog_begin, stream));
      int n = 0;
      for (int j = 0; n < st->spp; j++) {
        {  // pass j overwrites slot j % 2: preview j - 2 must have been shown
          std::unique_lock<std::mutex> lk(mu);
          cv.wait(lk, [&] { return stop || !on_preview || shown >= j - 1; });
          if (stop) break;
        }
        const int next = j == 0 ? pg->first_spp : progressive_next(n, st->spp, pg->max_pass_spp);
        Pass pass;
        pass.clear_film = j == 0;
        pass.lens = d_lens;
        pass.motion = moving.motion, pass.disp = moving.disp, pass.end_cams = moving.end_cams;
        render_pass(s, cam, st, n, next, pass, stream, total);
        k_resolve_film<<<(unsigned)((n_px + 255) / 256), 256, 0, stream>>>(s->film(), n_px, 1.0f / (float)next, nullptr,
                                                                           out_rgb ? s->w_prog_rgb[j & 1].p : nullptr,
                                                                           s->w_prog_packed[j & 1].p);
        CK(cudaGetLastError());
        total.kernel_launches += 1;
        CK(cudaEventRecord(s->ev_prog_slot[j & 1], stream));
        last_slot_event = s->ev_prog_slot[j & 1];
        n = next;
        {
          std::lock_guard<std::mutex> lk(mu);
          samples[j & 1] = n, ready = j + 1;
        }
        cv.notify_all();
      }
    } catch (...) {
      std::lock_guard<std::mutex> lk(mu);
      worker_error = std::current_exception();
    }
    {
      std::lock_guard<std::mutex> lk(mu);
      worker_done = true;
    }
    cv.notify_all();
  };

  // The worker is joined on every way out of this scope: told to stop, it finishes the pass in flight and starts no other.
  struct Joiner {
    std::thread th;
    std::mutex &mu;
    std::condition_variable &cv;
    bool &stop;
    void join() {
      if (!th.joinable()) return;
      {
        std::lock_guard<std::mutex> lk(mu);
        stop = true;
      }
      cv.notify_all();
      th.join();
    }
    ~Joiner() { join(); }
  } joiner{std::thread(worker), mu, cv, stop};

  int last = -1;  // the preview the outputs are: the one the callback stopped at, else the last pass's
  for (int j = 0;; j++) {
    int32_t n_j;
    {
      std::unique_lock<std::mutex> lk(mu);
      cv.wait(lk, [&] { return ready > j || worker_done; });
      if (ready <= j) break;
      n_j = samples[j & 1];
    }
    last = j;
    if (!on_preview) continue;
    CK(cudaStreamWaitEvent(s->preview_stream, s->ev_prog_slot[j & 1], 0));
    CK(cudaMemcpyAsync(s->h_preview, s->w_prog_packed[j & 1].p, n_px * sizeof(uint32_t), cudaMemcpyDeviceToHost, s->preview_stream));
    CK(cudaStreamSynchronize(s->preview_stream));
    const bool stop_here = on_preview(user, j, n_j, s->h_preview) != 0;
    {
      std::lock_guard<std::mutex> lk(mu);
      shown = j + 1;
      stop = stop || stop_here;
    }
    cv.notify_all();
    if (stop_here) break;
  }
  joiner.join();
  if (worker_error) std::rethrow_exception(worker_error);  // (without an error the worker has published pass 0 at least)
  // the worker is gone: the render stream and the staging buffer are this thread's again
  CK(cudaStreamSynchronize(stream));
  if (out_u32) film_to_host(s, s->w_prog_packed[last & 1].p, out_u32, n_px * sizeof(uint32_t), stream);
  if (out_rgb) film_to_host(s, s->w_prog_rgb[last & 1].p, out_rgb, n_px * 3 * sizeof(float), stream);
  if (out_samples) *out_samples = samples[last & 1];
  if (stats) {
    *stats = total;
    float ms = 0.0f;
    CK(cudaEventElapsedTime(&ms, s->ev_prog_begin, last_slot_event));
    stats->render_ms = ms;
  }
  return 0;
  PTC_GUARD_END
}

// ptc_denoise's filter parameters (the arguments of both denoise entry points; feature_spp is ptc_render_denoised's)
static void check_denoise_filter(const ptc_denoise *dn) {
  if (dn->iterations < 1 || dn->iterations > kDenoiseMaxIterations) throw std::invalid_argument("iterations must be 1..10");
  for (const float sg : {dn->sigma_luminance, dn->sigma_normal, dn->sigma_albedo})
    if (!(sg > 0.0f) || !std::isfinite(sg)) throw std::invalid_argument("the sigmas must be > 0 and finite");
}

// The filter on the device, queued on `stream`: the noisy image (W*H*3, in s->w_film_out), var (W*H), albedo and normal
// (W*H*3) -> s->w_dn_out (W*H*3 denoised) and s->w_packed (W*H, resolve_pixel of it at scale 1).  Returns the number of
// kernels launched.
static int denoise_filter(ptc_scene *s, const ptc_denoise *dn, int32_t width, int32_t height, const float *var, const float *albedo,
                          const float *normal, cudaStream_t stream) {
  const uint32_t n_px = (uint32_t)width * (uint32_t)height;
  for (auto &b : s->w_dn_xv)
    if (b.n < n_px) b.alloc(n_px);
  if (s->w_dn_ga.n < n_px) s->w_dn_ga.alloc(n_px), s->w_dn_gn.alloc(n_px);
  if (s->w_dn_out.n < (size_t)n_px * 3) s->w_dn_out.alloc((size_t)n_px * 3);
  if (s->w_packed.n < n_px) s->w_packed.alloc(n_px);
  const unsigned nb = (n_px + 255u) / 256u;
  k_denoise_prepare<<<nb, 256, 0, stream>>>(s->w_film_out.p, var, albedo, normal, n_px, s->w_dn_xv[0].p, s->w_dn_ga.p, s->w_dn_gn.p);
  const DenoiseParams dp = denoise_params(dn->sigma_luminance, dn->sigma_normal, dn->sigma_albedo);
  const dim3 block(kAtrousBlockX, kAtrousBlockY);
  const dim3 grid((unsigned)(width + kAtrousBlockX - 1) / kAtrousBlockX, (unsigned)(height + kAtrousBlockY - 1) / kAtrousBlockY);
  for (int i = 0; i < dn->iterations; i++)
    k_atrous<<<grid, block, 0, stream>>>(s->w_dn_xv[i & 1].p, s->w_dn_ga.p, s->w_dn_gn.p, width, height, 1 << i, dp, s->w_dn_xv[(i + 1) & 1].p);
  k_denoise_finish<<<nb, 256, 0, stream>>>(s->w_dn_xv[dn->iterations & 1].p, s->w_film_out.p, albedo, n_px, s->w_dn_out.p, s->w_packed.p);
  CK(cudaGetLastError());
  return 2 + dn->iterations;
}

int ptc_render_denoised(ptc_scene *s, const ptc_camera *cam, const ptc_render_settings *st, const ptc_denoise *dn, float *out_rgb,
                        uint32_t *out_u32, float *out_noisy_rgb, float *out_albedo, float *out_normal, float *out_variance,
                        ptc_stats *stats) {
  PTC_GUARD_BEGIN
  // the arguments first, the scene's state after them
  if (!s || !dn) throw std::invalid_argument("null argument");
  check_render_args(cam, st, true);  // every output may be NULL
  if (st->sample_begin != 0 || st->sample_end != 0 || st->tile_mod != 0)
    throw std::invalid_argument("ptc_render_denoised schedules the samples itself: sample_begin, sample_end and tile_mod must be 0");
  if (st->spp < 2) throw std::invalid_argument("ptc_render_denoised needs spp >= 2: the variance comes from two halves of the samples");
  if (dn->feature_spp < 1 || dn->feature_spp > st->spp) throw std::invalid_argument("feature_spp must be >= 1 and <= spp");
  check_denoise_filter(dn);
  const ptc_lens *lens = single_lens(s);
  const ptc_camera *end = single_end_cam(s);
  require_committed(s);
  CK(cudaSetDevice(s->device));
  ensure_ctl(s);
  const uint32_t n_px = (uint32_t)st->width * (uint32_t)st->height;
  const size_t n3 = (size_t)n_px * 3;
  if (s->w_dn_half.n < n3) s->w_dn_half.alloc(n3);
  if (s->w_dn_albedo.n < n3) s->w_dn_albedo.alloc(n3), s->w_dn_normal.alloc(n3);
  if (s->w_dn_rays.n < 2 * n3) s->w_dn_rays.alloc(2 * n3);
  if (s->w_dn_var.n < n_px) s->w_dn_var.alloc(n_px);
  if (s->w_film_out.n < n3) s->w_film_out.alloc(n3);
  if (!s->w_dn_ctl.p) s->w_dn_ctl.alloc(1);
  if (!s->ev_dn_begin) CK(cudaEventCreate(&s->ev_dn_begin));
  if (!s->ev_dn_end) CK(cudaEventCreate(&s->ev_dn_end));
  cudaStream_t stream = s->own_stream;
  const unsigned nb = (n_px + 255u) / 256u;
  ptc_stats total;
  memset(&total, 0, sizeof(total));
  uint64_t &launches = total.kernel_launches;

  // 1. the render in two halves, the fp32 film sums of the first one kept: the film is ptc_render's
  const int half = st->spp / 2;
  Pass first;
  first.lens = lens ? upload_lens(s, lens, 1, stream) : nullptr;
  upload_motion(s, single_motion(s, cam, end), stream, first);
  if (first.motion && s->w_dn_tau.n < n_px) s->w_dn_tau.alloc(n_px);
  CK(cudaEventRecord(s->ev_dn_begin, stream));
  render_pass(s, cam, st, 0, half, first, stream, total);
  CK(cudaMemsetAsync(s->w_dn_half.p, 0, n3 * sizeof(float), stream));
  k_film_to_accum<<<(unsigned)((n3 + 255) / 256), 256, 0, stream>>>(s->film(), n_px, s->w_dn_half.p);
  Pass more = first;
  more.clear_film = false;
  render_pass(s, cam, st, half, st->spp, more, stream, total);
  launches += 1;

  // 2. features: camera samples 0 .. feature_spp - 1 in order, each one's first hits added to the per-pixel sums
  CK(cudaMemsetAsync(s->w_dn_albedo.p, 0, n3 * sizeof(float), stream));
  CK(cudaMemsetAsync(s->w_dn_normal.p, 0, n3 * sizeof(float), stream));
  CK(cudaMemsetAsync(s->w_dn_ctl.p, 0, sizeof(Ctl), stream));
  RenderParams rp;
  memset(&rp, 0, sizeof(rp));
  memcpy(&rp.cam, cam, sizeof(DCamera));
  rp.width = st->width, rp.height = st->height, rp.seed = st->seed;
  float *ray_o = s->w_dn_rays.p, *ray_d = s->w_dn_rays.p + n3;
  for (int k = 0; k < dn->feature_spp; k++) {
    if (first.motion) {
      // the primary rays at their shutter times, intersected at those times
      k_primary_rays_motion<<<nb, 256, 0, stream>>>(rp, (uint32_t)k, ray_o, ray_d, s->w_dn_tau.p, LensTables{first.lens},
                                                    MotionTables{first.disp, first.end_cams, nullptr, nullptr});
      launches += 3 + extend_hook_rays(s, ray_o, ray_d, n_px, kEps, INFINITY, s->w_dn_ctl.p, false, stream, nullptr, nullptr, nullptr,
                                       s->w_dn_tau.p, first.disp);
    } else {
      if (first.lens) k_primary_rays_lens<<<nb, 256, 0, stream>>>(rp, (uint32_t)k, ray_o, ray_d, LensTables{first.lens});
      else k_primary_rays<<<nb, 256, 0, stream>>>(rp, (uint32_t)k, ray_o, ray_d);
      launches += 3 + extend_hook_rays(s, ray_o, ray_d, n_px, kEps, INFINITY, s->w_dn_ctl.p, false, stream);
    }
    const Buffers b = s->ws_hook.buffers();
    k_feature_add<<<nb, 256, 0, stream>>>(b.hit0, b.hit1, s->ds.materials, n_px, s->w_dn_albedo.p, s->w_dn_normal.p);
    launches += 1;
  }
  k_feature_mean<<<(unsigned)((n3 + 255) / 256), 256, 0, stream>>>(s->w_dn_albedo.p, s->w_dn_normal.p, n3, 1.0f / (float)dn->feature_spp);

  // 3. the noisy image (ptc_render's), the variance from the halves, the filter
  k_resolve_film<<<nb, 256, 0, stream>>>(s->film(), n_px, 1.0f / (float)st->spp, nullptr, s->w_film_out.p, nullptr);
  k_denoise_variance<<<nb, 256, 0, stream>>>(s->w_dn_half.p, s->film(), n_px, half, st->spp, s->w_dn_albedo.p, s->w_dn_var.p);
  CK(cudaGetLastError());
  launches += 3 + denoise_filter(s, dn, st->width, st->height, s->w_dn_var.p, s->w_dn_albedo.p, s->w_dn_normal.p, stream);
  CK(cudaEventRecord(s->ev_dn_end, stream));

  if (out_rgb) film_to_host(s, s->w_dn_out.p, out_rgb, n3 * sizeof(float), stream);
  if (out_u32) film_to_host(s, s->w_packed.p, out_u32, (size_t)n_px * sizeof(uint32_t), stream);
  if (out_noisy_rgb) film_to_host(s, s->w_film_out.p, out_noisy_rgb, n3 * sizeof(float), stream);
  if (out_albedo) film_to_host(s, s->w_dn_albedo.p, out_albedo, n3 * sizeof(float), stream);
  if (out_normal) film_to_host(s, s->w_dn_normal.p, out_normal, n3 * sizeof(float), stream);
  if (out_variance) film_to_host(s, s->w_dn_var.p, out_variance, (size_t)n_px * sizeof(float), stream);
  CK(cudaStreamSynchronize(stream));
  if (stats) {
    *stats = total;
    float ms = 0.0f;
    CK(cudaEventElapsedTime(&ms, s->ev_dn_begin, s->ev_dn_end));
    stats->render_ms = ms;
  }
  return 0;
  PTC_GUARD_END
}

int ptc_denoise_image(ptc_scene *s, const ptc_denoise *dn, int32_t width, int32_t height, const float *rgb, const float *variance,
                      const float *albedo, const float *normal, float *out_rgb) {
  PTC_GUARD_BEGIN
  if (!s || !dn || !rgb || !variance || !albedo || !normal || !out_rgb) throw std::invalid_argument("null argument");
  if (width <= 0 || height <= 0) throw std::invalid_argument("bad image size");
  if ((int64_t)width * height > (int64_t)0x3fffffff) throw std::invalid_argument("image too large");
  check_denoise_filter(dn);
  require_committed(s);
  CK(cudaSetDevice(s->device));
  const uint32_t n_px = (uint32_t)width * (uint32_t)height;
  const size_t n3 = (size_t)n_px * 3;
  if (s->w_film_out.n < n3) s->w_film_out.alloc(n3);
  if (s->w_dn_albedo.n < n3) s->w_dn_albedo.alloc(n3), s->w_dn_normal.alloc(n3);
  if (s->w_dn_var.n < n_px) s->w_dn_var.alloc(n_px);
  cudaStream_t stream = s->own_stream;
  CK(cudaMemcpyAsync(s->w_film_out.p, rgb, n3 * sizeof(float), cudaMemcpyHostToDevice, stream));
  CK(cudaMemcpyAsync(s->w_dn_var.p, variance, (size_t)n_px * sizeof(float), cudaMemcpyHostToDevice, stream));
  CK(cudaMemcpyAsync(s->w_dn_albedo.p, albedo, n3 * sizeof(float), cudaMemcpyHostToDevice, stream));
  CK(cudaMemcpyAsync(s->w_dn_normal.p, normal, n3 * sizeof(float), cudaMemcpyHostToDevice, stream));
  denoise_filter(s, dn, width, height, s->w_dn_var.p, s->w_dn_albedo.p, s->w_dn_normal.p, stream);
  film_to_host(s, s->w_dn_out.p, out_rgb, n3 * sizeof(float), stream);
  return 0;
  PTC_GUARD_END
}

int ptc_resolve_device(const float *d_rgb, int64_t n_pixels, float scale, uint32_t *d_out, void *cuda_stream) {
  PTC_GUARD_BEGIN
  if (!d_rgb || !d_out || n_pixels < 0) throw std::invalid_argument("bad argument");
  if (n_pixels == 0) return 0;
  k_resolve<<<(unsigned)((n_pixels + 255) / 256), 256, 0, (cudaStream_t)cuda_stream>>>(d_rgb, (size_t)n_pixels, scale, d_out);
  CK(cudaGetLastError());
  return 0;
  PTC_GUARD_END
}

int ptc_resolve_u32(ptc_scene *s, const float *rgb, int64_t n_pixels, float scale, uint32_t *out) {
  PTC_GUARD_BEGIN
  require_committed(s);
  if (!rgb || !out || n_pixels < 0) throw std::invalid_argument("bad argument");
  if (n_pixels == 0) return 0;
  CK(cudaSetDevice(s->device));
  if (s->w_film_out.n < (size_t)n_pixels * 3) s->w_film_out.alloc((size_t)n_pixels * 3);
  if (s->w_packed.n < (size_t)n_pixels) s->w_packed.alloc((size_t)n_pixels);
  DevBuf<float> &d_in = s->w_film_out;
  DevBuf<uint32_t> &d_out = s->w_packed;
  CK(cudaMemcpyAsync(d_in.p, rgb, (size_t)n_pixels * 3 * sizeof(float), cudaMemcpyHostToDevice, s->own_stream));
  k_resolve<<<(unsigned)((n_pixels + 255) / 256), 256, 0, s->own_stream>>>(d_in.p, (size_t)n_pixels, scale, d_out.p);
  CK(cudaGetLastError());
  CK(cudaMemcpyAsync(out, d_out.p, (size_t)n_pixels * 4, cudaMemcpyDeviceToHost, s->own_stream));
  CK(cudaStreamSynchronize(s->own_stream));
  return 0;
  PTC_GUARD_END
}

int ptc_intersect(ptc_scene *s, const float *origins, const float *dirs, int64_t n, float t_min, float t_max, ptc_hit *out,
                  ptc_stats *stats) {
  PTC_GUARD_BEGIN
  require_committed(s);
  if (n < 0 || (n > 0 && (!origins || !dirs || !out))) throw std::invalid_argument("bad argument");
  if (stats) memset(stats, 0, sizeof(*stats));
  if (n == 0) return 0;
  if (n > (int64_t)0x3fffffff) throw std::invalid_argument("too many rays for one call");
  CK(cudaSetDevice(s->device));
  ensure_ctl(s);
  DevBuf<float> d_o, d_d;
  DevBuf<ptc_hit> d_out;
  DevBuf<Ctl> ctl;
  d_o.upload(origins, (size_t)n * 3);
  d_d.upload(dirs, (size_t)n * 3);
  d_out.alloc((size_t)n);
  Ctl init;
  memset(&init, 0, sizeof(init));
  ctl.upload(&init, 1);
  cudaStream_t st = s->own_stream;
  cudaEvent_t ea, eb;
  CK(cudaEventCreate(&ea));
  CK(cudaEventCreate(&eb));
  const int ext_launches = extend_hook_rays(s, d_o.p, d_d.p, (uint32_t)n, t_min, t_max, ctl.p, true, st, ea, eb);
  const Buffers b = s->ws_hook.buffers();
  k_unpack_hits<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(b.hit0, b.hit1, s->ws_hook.ids.p, (size_t)n, d_out.p);
  CK(cudaGetLastError());
  CK(cudaMemcpyAsync(out, d_out.p, (size_t)n * sizeof(ptc_hit), cudaMemcpyDeviceToHost, st));
  Ctl fin;
  CK(cudaMemcpyAsync(&fin, ctl.p, sizeof(Ctl), cudaMemcpyDeviceToHost, st));
  CK(cudaStreamSynchronize(st));
  if (stats) {
    float ms = 0.0f;
    CK(cudaEventElapsedTime(&ms, ea, eb));
    stats->rays = (uint64_t)n;
    stats->kernel_launches = 3 + (uint64_t)ext_launches;
    stats->render_ms = ms;
    stats->extend_ms = ms;
    stats->extend_launches = 1;
    stats->nodes_visited = fin.nodes;
    stats->tris_tested = fin.tris;
    stats->mesh_rays = fin.mesh_rays;
  }
  cudaEventDestroy(ea);
  cudaEventDestroy(eb);
  return 0;
  PTC_GUARD_END
}

int ptc_intersect_at(ptc_scene *s, const float *origins, const float *dirs, const float *times, int64_t n, float t_min, float t_max,
                     ptc_hit *out, ptc_stats *stats) {
  PTC_GUARD_BEGIN
  require_committed(s);
  if (n < 0 || (n > 0 && (!origins || !dirs || !times || !out))) throw std::invalid_argument("bad argument");
  for (int64_t i = 0; i < n; i++)
    if (!(times[i] >= 0.0f && times[i] <= 1.0f)) throw std::invalid_argument("a ray's time must be in [0, 1]");
  if (stats) memset(stats, 0, sizeof(*stats));
  if (n == 0) return 0;
  if (n > (int64_t)0x3fffffff) throw std::invalid_argument("too many rays for one call");
  CK(cudaSetDevice(s->device));
  const MotionCall mc = motion_call(s, nullptr, 0, nullptr, 0);
  if (!mc.objects) return ptc_intersect(s, origins, dirs, n, t_min, t_max, out, stats);  // nothing moves: today's kernels
  ensure_ctl(s);
  DevBuf<float> d_o, d_d, d_t;
  DevBuf<ptc_hit> d_out;
  DevBuf<Ctl> ctl;
  d_o.upload(origins, (size_t)n * 3);
  d_d.upload(dirs, (size_t)n * 3);
  d_t.upload(times, (size_t)n);
  d_out.alloc((size_t)n);
  Ctl init;
  memset(&init, 0, sizeof(init));
  ctl.upload(&init, 1);
  cudaStream_t st = s->own_stream;
  Pass pass;
  upload_motion(s, mc, st, pass);
  cudaEvent_t ea, eb;
  CK(cudaEventCreate(&ea));
  CK(cudaEventCreate(&eb));
  const int ext_launches = extend_hook_rays(s, d_o.p, d_d.p, (uint32_t)n, t_min, t_max, ctl.p, true, st, ea, eb, nullptr, d_t.p, pass.disp);
  const Buffers b = s->ws_hook.buffers();
  k_unpack_hits<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(b.hit0, b.hit1, s->ws_hook.ids.p, (size_t)n, d_out.p);
  CK(cudaGetLastError());
  CK(cudaMemcpyAsync(out, d_out.p, (size_t)n * sizeof(ptc_hit), cudaMemcpyDeviceToHost, st));
  Ctl fin;
  CK(cudaMemcpyAsync(&fin, ctl.p, sizeof(Ctl), cudaMemcpyDeviceToHost, st));
  CK(cudaStreamSynchronize(st));
  if (stats) {
    float ms = 0.0f;
    CK(cudaEventElapsedTime(&ms, ea, eb));
    stats->rays = (uint64_t)n;
    stats->kernel_launches = 3 + (uint64_t)ext_launches;
    stats->render_ms = ms;
    stats->extend_ms = ms;
    stats->extend_launches = 1;
    stats->nodes_visited = fin.nodes;
    stats->tris_tested = fin.tris;
    stats->mesh_rays = fin.mesh_rays;
  }
  cudaEventDestroy(ea);
  cudaEventDestroy(eb);
  return 0;
  PTC_GUARD_END
}

int ptc_ray_times(ptc_scene *s, const ptc_render_settings *st, int32_t sample, float *out_time) {
  PTC_GUARD_BEGIN
  require_committed(s);
  if (!st || !out_time || st->width <= 0 || st->height <= 0 || sample < 0) throw std::invalid_argument("bad argument");
  if ((int64_t)st->width * st->height > (int64_t)0x3fffffff) throw std::invalid_argument("image too large");
  CK(cudaSetDevice(s->device));
  const uint32_t n = (uint32_t)st->width * (uint32_t)st->height;
  DevBuf<float> d_t;
  d_t.alloc(n);
  k_ray_times<<<(n + 255) / 256, 256, 0, s->own_stream>>>(st->seed, n, (uint32_t)sample, d_t.p);
  CK(cudaGetLastError());
  CK(cudaMemcpyAsync(out_time, d_t.p, (size_t)n * sizeof(float), cudaMemcpyDeviceToHost, s->own_stream));
  CK(cudaStreamSynchronize(s->own_stream));
  return 0;
  PTC_GUARD_END
}

int ptc_primary_rays(ptc_scene *s, const ptc_camera *cam, const ptc_render_settings *st, int32_t sample, float *out_o,
                     float *out_d) {
  PTC_GUARD_BEGIN
  if (!s) throw std::invalid_argument("null argument");
  const ptc_lens *lens = single_lens(s);
  const ptc_camera *end = single_end_cam(s);
  require_committed(s);
  if (!cam || !st || !out_o || !out_d || st->width <= 0 || st->height <= 0) throw std::invalid_argument("bad argument");
  CK(cudaSetDevice(s->device));
  RenderParams rp;
  memset(&rp, 0, sizeof(rp));
  memcpy(&rp.cam, cam, sizeof(DCamera));
  rp.width = st->width, rp.height = st->height, rp.seed = st->seed;
  const size_t n = (size_t)st->width * st->height;
  DevBuf<float> d_o, d_d;
  d_o.alloc(n * 3);
  d_d.alloc(n * 3);
  const MotionCall mc = single_motion(s, cam, end);
  if (!mc.end_cams.empty()) {  // the camera at each ray's shutter time (object motion does not change a camera ray)
    Pass pass;
    upload_motion(s, mc, s->own_stream, pass);
    const LensTables lt{lens ? upload_lens(s, lens, 1, s->own_stream) : nullptr};
    k_primary_rays_motion<<<(unsigned)((n + 255) / 256), 256, 0, s->own_stream>>>(rp, (uint32_t)sample, d_o.p, d_d.p, nullptr, lt,
                                                                                  MotionTables{pass.disp, pass.end_cams, nullptr, nullptr});
  } else if (lens) {
    k_primary_rays_lens<<<(unsigned)((n + 255) / 256), 256, 0, s->own_stream>>>(rp, (uint32_t)sample, d_o.p, d_d.p,
                                                                                LensTables{upload_lens(s, lens, 1, s->own_stream)});
  } else {
    k_primary_rays<<<(unsigned)((n + 255) / 256), 256, 0, s->own_stream>>>(rp, (uint32_t)sample, d_o.p, d_d.p);
  }
  CK(cudaGetLastError());
  CK(cudaMemcpyAsync(out_o, d_o.p, n * 12, cudaMemcpyDeviceToHost, s->own_stream));
  CK(cudaMemcpyAsync(out_d, d_d.p, n * 12, cudaMemcpyDeviceToHost, s->own_stream));
  CK(cudaStreamSynchronize(s->own_stream));
  return 0;
  PTC_GUARD_END
}

int ptc_scatter(ptc_scene *s, int material, const float *ray_dirs, const float *positions, const float *normals,
                const int32_t *front_face, const float *u4, int64_t n, int32_t *scattered, float *out_origin, float *out_dir,
                float *attenuation, float *emitted) {
  PTC_GUARD_BEGIN
  require_committed(s);
  if (material < 0 || (size_t)material >= s->hs.materials.size()) throw std::invalid_argument("material index out of range");
  if (n < 0) throw std::invalid_argument("bad argument");
  if (n == 0) return 0;
  CK(cudaSetDevice(s->device));
  const size_t N = (size_t)n;
  DevBuf<float> d_dir, d_pos, d_nrm, d_u, d_oo, d_od, d_att, d_em;
  DevBuf<int32_t> d_front, d_sc;
  d_dir.upload(ray_dirs, N * 3);
  d_pos.upload(positions, N * 3);
  d_nrm.upload(normals, N * 3);
  d_u.upload(u4, N * 4);
  d_front.upload(front_face, N);
  d_oo.alloc(N * 3), d_od.alloc(N * 3), d_att.alloc(N * 3), d_em.alloc(N * 3), d_sc.alloc(N);
  k_scatter<<<(unsigned)((N + 127) / 128), 128, 0, s->own_stream>>>(s->hs.materials[(size_t)material], d_dir.p, d_pos.p, d_nrm.p,
                                                                    d_front.p, d_u.p, N, d_sc.p, d_oo.p, d_od.p, d_att.p, d_em.p);
  CK(cudaGetLastError());
  CK(cudaMemcpyAsync(scattered, d_sc.p, N * 4, cudaMemcpyDeviceToHost, s->own_stream));
  CK(cudaMemcpyAsync(out_origin, d_oo.p, N * 12, cudaMemcpyDeviceToHost, s->own_stream));
  CK(cudaMemcpyAsync(out_dir, d_od.p, N * 12, cudaMemcpyDeviceToHost, s->own_stream));
  CK(cudaMemcpyAsync(attenuation, d_att.p, N * 12, cudaMemcpyDeviceToHost, s->own_stream));
  CK(cudaMemcpyAsync(emitted, d_em.p, N * 12, cudaMemcpyDeviceToHost, s->own_stream));
  CK(cudaStreamSynchronize(s->own_stream));
  return 0;
  PTC_GUARD_END
}

int ptc_sky_sample(ptc_scene *s, const float *u4, int64_t n, float *out_dir, float *out_pdf, float *out_rgb) {
  PTC_GUARD_BEGIN
  require_committed(s);
  if (n < 0 || (n > 0 && (!u4 || !out_dir || !out_pdf || !out_rgb))) throw std::invalid_argument("bad argument");
  if (!s->ds.sky_dist) throw std::logic_error("the committed scene has no sky distribution (no HDR sky, or an all-zero one)");
  if (n == 0) return 0;
  CK(cudaSetDevice(s->device));
  const size_t N = (size_t)n;
  DevBuf<float> d_u, d_dir, d_pdf, d_rgb;
  d_u.upload(u4, N * 4);
  d_dir.alloc(N * 3), d_pdf.alloc(N), d_rgb.alloc(N * 3);
  k_sky_sample<<<(unsigned)((N + 127) / 128), 128, 0, s->own_stream>>>(s->ds, d_u.p, N, d_dir.p, d_pdf.p, d_rgb.p);
  CK(cudaGetLastError());
  CK(cudaMemcpyAsync(out_dir, d_dir.p, N * 12, cudaMemcpyDeviceToHost, s->own_stream));
  CK(cudaMemcpyAsync(out_pdf, d_pdf.p, N * 4, cudaMemcpyDeviceToHost, s->own_stream));
  CK(cudaMemcpyAsync(out_rgb, d_rgb.p, N * 12, cudaMemcpyDeviceToHost, s->own_stream));
  CK(cudaStreamSynchronize(s->own_stream));
  return 0;
  PTC_GUARD_END
}

int ptc_sky_pdf(ptc_scene *s, const float *dirs, int64_t n, float *out_pdf) {
  PTC_GUARD_BEGIN
  require_committed(s);
  if (n < 0 || (n > 0 && (!dirs || !out_pdf))) throw std::invalid_argument("bad argument");
  if (!s->ds.sky_dist) throw std::logic_error("the committed scene has no sky distribution (no HDR sky, or an all-zero one)");
  if (n == 0) return 0;
  CK(cudaSetDevice(s->device));
  const size_t N = (size_t)n;
  DevBuf<float> d_dir, d_pdf;
  d_dir.upload(dirs, N * 3);
  d_pdf.alloc(N);
  k_sky_pdf<<<(unsigned)((N + 127) / 128), 128, 0, s->own_stream>>>(s->ds, d_dir.p, N, d_pdf.p);
  CK(cudaGetLastError());
  CK(cudaMemcpyAsync(out_pdf, d_pdf.p, N * 4, cudaMemcpyDeviceToHost, s->own_stream));
  CK(cudaStreamSynchronize(s->own_stream));
  return 0;
  PTC_GUARD_END
}

int ptc_light_sample(ptc_scene *s, const float *x, const float *u4, int64_t n, float *out_point, float *out_pdf, int32_t *out_object,
                     int32_t *out_triangle) {
  PTC_GUARD_BEGIN
  require_committed(s);
  if (n < 0 || (n > 0 && (!x || !u4 || !out_point || !out_pdf || !out_object || !out_triangle))) throw std::invalid_argument("bad argument");
  if (s->ds_em.n_lights == 0) throw std::logic_error("the committed scene has no emitter PTC_FLAG_NEE_EMITTERS samples");
  if (n == 0) return 0;
  CK(cudaSetDevice(s->device));
  const size_t N = (size_t)n;
  DevBuf<float> d_x, d_u, d_pt, d_pdf;
  DevBuf<int32_t> d_obj, d_tri;
  d_x.upload(x, N * 3);
  d_u.upload(u4, N * 4);
  d_pt.alloc(N * 3), d_pdf.alloc(N), d_obj.alloc(N), d_tri.alloc(N);
  k_light_sample<<<(unsigned)((N + 127) / 128), 128, 0, s->own_stream>>>(s->ds_em, s->et, d_x.p, d_u.p, N, d_pt.p, d_pdf.p, d_obj.p, d_tri.p);
  CK(cudaGetLastError());
  CK(cudaMemcpyAsync(out_point, d_pt.p, N * 12, cudaMemcpyDeviceToHost, s->own_stream));
  CK(cudaMemcpyAsync(out_pdf, d_pdf.p, N * 4, cudaMemcpyDeviceToHost, s->own_stream));
  CK(cudaMemcpyAsync(out_object, d_obj.p, N * 4, cudaMemcpyDeviceToHost, s->own_stream));
  CK(cudaMemcpyAsync(out_triangle, d_tri.p, N * 4, cudaMemcpyDeviceToHost, s->own_stream));
  CK(cudaStreamSynchronize(s->own_stream));
  return 0;
  PTC_GUARD_END
}

int ptc_light_pdf(ptc_scene *s, const float *origins, const float *dirs, int64_t n, float *out_pdf) {
  PTC_GUARD_BEGIN
  require_committed(s);
  if (n < 0 || (n > 0 && (!origins || !dirs || !out_pdf))) throw std::invalid_argument("bad argument");
  if (s->ds_em.n_lights == 0) throw std::logic_error("the committed scene has no emitter PTC_FLAG_NEE_EMITTERS samples");
  if (n == 0) return 0;
  if (n > (int64_t)0x3fffffff) throw std::invalid_argument("too many rays for one call");
  CK(cudaSetDevice(s->device));
  ensure_ctl(s);
  const size_t N = (size_t)n;
  DevBuf<float> d_o, d_d, d_pdf;
  DevBuf<Ctl> ctl;
  d_o.upload(origins, N * 3);
  d_d.upload(dirs, N * 3);
  d_pdf.alloc(N);
  Ctl init;
  memset(&init, 0, sizeof(init));
  ctl.upload(&init, 1);
  cudaStream_t st = s->own_stream;
  // the render's extend kernels, on the object table whose hit records carry the PTC_FLAG_NEE_EMITTERS light ids
  extend_hook_rays(s, d_o.p, d_d.p, (uint32_t)n, kEps, INFINITY, ctl.p, false, st, nullptr, nullptr, &s->ds_em);
  const Buffers b = s->ws_hook.buffers();
  k_light_pdf<<<(unsigned)((N + 127) / 128), 128, 0, st>>>(s->ds_em, s->et, d_o.p, d_d.p, b.hit0, b.hit1, N, d_pdf.p);
  CK(cudaGetLastError());
  CK(cudaMemcpyAsync(out_pdf, d_pdf.p, N * 4, cudaMemcpyDeviceToHost, st));
  CK(cudaStreamSynchronize(st));
  return 0;
  PTC_GUARD_END
}

int ptc_philox(ptc_scene *s, const uint32_t ctr[4], const uint32_t key[2], uint32_t out[4]) {
  PTC_GUARD_BEGIN
  require_committed(s);
  if (!ctr || !key || !out) throw std::invalid_argument("null argument");
  CK(cudaSetDevice(s->device));
  DevBuf<uint32_t> d;
  d.alloc(4);
  k_philox<<<1, 1, 0, s->own_stream>>>(U4{ctr[0], ctr[1], ctr[2], ctr[3]}, key[0], key[1], d.p);
  CK(cudaGetLastError());
  CK(cudaMemcpyAsync(out, d.p, 16, cudaMemcpyDeviceToHost, s->own_stream));
  CK(cudaStreamSynchronize(s->own_stream));
  return 0;
  PTC_GUARD_END
}

// ---- in-process multi-GPU ------------------------------------------------------------------------------------
int ptc_multi_create(ptc_scene *primary, const int *devices, int n, ptc_multi **out) {
  PTC_GUARD_BEGIN
  require_committed(primary);
  if (!devices || !out || n < 1) throw std::invalid_argument("bad argument");
  if (devices[0] != primary->device) throw std::invalid_argument("devices[0] must be the device the scene was committed on");
  int have = 0;
  CK(cudaGetDeviceCount(&have));
  for (int i = 0; i < n; i++) {
    if (devices[i] < 0 || devices[i] >= have) throw std::invalid_argument("device index out of range");
    for (int j = 0; j < i; j++)
      if (devices[j] == devices[i]) throw std::invalid_argument("duplicate device");
  }
  std::unique_ptr<ptc_multi> m(new ptc_multi());
  m->primary = primary;
  m->devices.assign(devices, devices + n);
  m->scenes.push_back(primary);
  for (int i = 1; i < n; i++) {  // the host-side flattening (BVH build) is done once, by the primary
    std::unique_ptr<ptc_scene> r(new ptc_scene());
    upload_scene(r.get(), primary->hs, devices[i]);
    m->scenes.push_back(r.get());
    m->replicas.push_back(std::move(r));
  }
  if (n > 1) {
    m->nccl.load();
    m->init_comms();
  }
  CK(cudaSetDevice(primary->device));
  *out = m.release();
  return 0;
  PTC_GUARD_END
}

void ptc_multi_destroy(ptc_multi *m) { delete m; }

static int multi_render(ptc_multi *m, const ptc_camera *cam, const ptc_render_settings *st, int shard_mode, float *out_rgb, uint32_t *out_u32,
                        ptc_stats *stats) {
  PTC_GUARD_BEGIN
  if (!m) throw std::invalid_argument("null argument");
  check_render_args(cam, st, out_rgb || out_u32);
  if (st->tile_mod > 0) throw std::invalid_argument("ptc_multi_render shards by itself: tile_mod must be 0");
  if (shard_mode != PTC_SHARD_SAMPLES && shard_mode != PTC_SHARD_TILES) throw std::invalid_argument("bad shard mode");
  // every device renders through the primary handle's lens
  const ptc_lens *lens = single_lens(m->primary);
  // ... and with the primary handle's motion at the time of the call
  const MotionCall mc = single_motion(m->primary, cam, single_end_cam(m->primary));
  const int n = (int)m->scenes.size();
  int s_begin, s_end;
  sample_range(st, s_begin, s_end);
  const size_t n_px = (size_t)st->width * st->height;
  std::vector<ptc_stats> per((size_t)n);
  std::vector<std::string> errors((size_t)n);
  const auto t0 = std::chrono::steady_clock::now();
  // Everything that can fail for lack of memory happens before the first thread starts: a worker that dropped out
  // ahead of the collective would leave the other devices waiting in ncclReduce for ever.
  if (n > 1 && m->comms_dead) m->init_comms();
  for (int i = 0; i < n; i++) {
    ptc_scene *s = m->scenes[(size_t)i];
    CK(cudaSetDevice(s->device));
    ensure_film(s, n_px);
    if (lens && s->d_lens.n < 1) s->d_lens.alloc(1);
    if (mc.any()) ensure_motion(s, mc);
  }
  std::mutex abort_mutex;
  auto work = [&](int i) {
    ptc_scene *s = m->scenes[(size_t)i];
    cudaStream_t stream = s->own_stream;
    bool film_ok = false;
    try {
      CK(cudaSetDevice(s->device));
      ptc_render_settings mine = *st;
      bool idle = false;
      if (shard_mode == PTC_SHARD_SAMPLES) {  // contiguous, balanced split of the sample range
        const int total = s_end - s_begin, base = total / n, rem = total % n;
        mine.sample_begin = s_begin + i * base + std::min(i, rem);
        mine.sample_end = mine.sample_begin + base + (i < rem ? 1 : 0);
        idle = mine.sample_end == mine.sample_begin;
      } else {  // interleaved 32x32 tiles
        mine.sample_begin = s_begin, mine.sample_end = s_end;
        mine.tile_mod = n, mine.tile_rem = i;
      }
      memset(&per[(size_t)i], 0, sizeof(ptc_stats));
      Pass pass;
      pass.lens = lens && !idle ? upload_lens(s, lens, 1, stream) : nullptr;
      if (!idle) upload_motion(s, mc, stream, pass);
      if (idle) clear_film(s, n_px, stream);
      else render_accumulate(s, cam, &mine, nullptr, stream, &per[(size_t)i], pass);  // leaves the shard in the device's fixed-point film
      film_ok = true;
    } catch (std::exception &e) {
      errors[(size_t)i] = e.what();
    }
    if (n == 1) {
      if (film_ok && cudaStreamSynchronize(stream) != cudaSuccess) errors[(size_t)i] = "cudaStreamSynchronize failed";
      return;
    }
    // the single exchange step of the path (SURVEY.md 8e): the films are summed onto devices[0].  The sums are 64-bit
    // integers, so the reduced film — and the image — is the one-GPU film bit for bit, whatever the number of devices and
    // the order NCCL adds in.  A device whose render failed still takes part, with a zeroed film, so that the others return;
    // if it cannot even do that the communicators are aborted (and re-created by the next call).
    try {
      if (!film_ok) clear_film(s, n_px, stream);
      m->nccl.check(m->nccl.Reduce(s->film_sum.p, s->film_sum.p, n_px * 3, ncclInt64, ncclSum, 0, m->comms[(size_t)i], stream), "ncclReduce(film)");
      m->nccl.check(m->nccl.Reduce(s->film_flags.p, s->film_flags.p, n_px, ncclUint64, ncclSum, 0, m->comms[(size_t)i], stream), "ncclReduce(flags)");
      CK(cudaStreamSynchronize(stream));
    } catch (std::exception &e) {
      if (errors[(size_t)i].empty()) errors[(size_t)i] = e.what();
      std::lock_guard<std::mutex> lock(abort_mutex);
      if (!m->comms_dead) m->abort_comms();
    }
  };
  std::vector<std::thread> threads;
  for (int i = 1; i < n; i++) threads.emplace_back(work, i);
  work(0);
  for (auto &t : threads) t.join();
  for (int i = 0; i < n; i++)
    if (!errors[(size_t)i].empty()) throw CudaError("device " + std::to_string(m->devices[(size_t)i]) + ": " + errors[(size_t)i]);
  ptc_scene *root = m->primary;
  CK(cudaSetDevice(root->device));
  const int launches = resolve_film_to_host(root, n_px, 1.0f / (float)st->spp, nullptr, out_rgb, out_u32, root->own_stream);  // renderer.rs:85
  if (stats) {
    memset(stats, 0, sizeof(*stats));
    for (const ptc_stats &p : per) {
      stats->paths += p.paths, stats->rays += p.rays, stats->kernel_launches += p.kernel_launches;
      stats->iterations = std::max(stats->iterations, p.iterations);
      stats->nodes_visited += p.nodes_visited, stats->tris_tested += p.tris_tested, stats->mesh_rays += p.mesh_rays;
    }
    stats->kernel_launches += launches;
    // wall clock of the whole call on the host: renders on all devices, the reduce, the resolve and the copy out
    stats->render_ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
  }
  return 0;
  PTC_GUARD_END
}

int ptc_multi_render(ptc_multi *m, const ptc_camera *cam, const ptc_render_settings *st, int shard_mode, float *out_rgb, ptc_stats *stats) {
  if (!out_rgb) return fail(PTC_E_INVALID, "null argument");
  return multi_render(m, cam, st, shard_mode, out_rgb, nullptr, stats);
}
int ptc_multi_render_u32(ptc_multi *m, const ptc_camera *cam, const ptc_render_settings *st, int shard_mode, uint32_t *out_u32,
                         ptc_stats *stats) {
  if (!out_u32) return fail(PTC_E_INVALID, "null argument");
  return multi_render(m, cam, st, shard_mode, nullptr, out_u32, stats);
}

}  // extern "C"
