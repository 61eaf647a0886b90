// dts_api.cu — the C ABI of libdtsim.so (include/dtsim.h): handle management, host->device
// staging of maps and episode parameters, and stream-ordered launches of the kernels.
#include <algorithm>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <dlfcn.h>
#include <string>
#include <vector>

#include "dts_kernels.h"

using namespace dts;

namespace {
thread_local std::string g_create_error;

#define DTS_CUDA(expr)                                                                          \
  do {                                                                                          \
    cudaError_t _e = (expr);                                                                    \
    if (_e != cudaSuccess) return sim->fail("%s failed: %s", #expr, cudaGetErrorString(_e));     \
  } while (0)
}  // namespace

struct dts_sim {
  dts_config cfg;
  StepCfg step_cfg;
  DState S;
  std::vector<void*> allocs;           // freed in dts_destroy
  std::vector<std::vector<void*>> map_allocs;
  std::vector<DMap> h_maps;
  DMap* d_maps = nullptr;
  // reset staging (device) sized num_envs
  struct { int32_t* map_id; double *pos_x, *pos_z, *angle, *wheel_dist, *trim; float *f1[3]; float *f3[5];
           float* light_pos; int32_t* light_stale; uint32_t* hidden; } stage{};
  // render
  void* render_scratch = nullptr;
  int render_ctas = 0, max_prims = 0, bin_cap = 0, max_lat = 0, items_max = 0;
  FishTab fish{};   // fused fisheye tables (dts_set_fisheye_lut)
  int32_t* d_err = nullptr;
  int32_t* h_status = nullptr;          // mapped pinned host word: bit 0 = a frame overflowed its frame memory
  int32_t* d_status = nullptr;          // its device address
  // fused end-of-rollout gather over peer memory (dts_gather_*)
  uint8_t* gather_buf = nullptr;        // [world][bytes_per_rank], this rank's copy of everybody's observations
  uint64_t gather_bytes = 0;
  int gather_world = 0, gather_rank = 0;
  void* gather_peer[DTS_MAX_PEERS] = {};   // peers' buffers opened with cudaIpcOpenMemHandle (own entry = gather_buf)
  bool gather_next = false;
  int render_mode = 0;                  // dts_set_render_mode             // the next dts_render also stores into the gather buffers
  // fused ResizeWrapper (dts_set_resize): full-size render target + tap tables
  int resize_w = 0, resize_h = 0;
  int resize_band = 0, resize_cap = 0;   // k_resize_band: output rows per CTA and the largest source-row span of a band (0: untiled kernel)
  uint8_t* resize_src = nullptr;
  int16_t *resize_xtab = nullptr, *resize_ytab = nullptr;
  // per-kernel timing (dts_profile_*): event pairs recorded around the render launches
  int profiling = 0;                    // 0 off, 1 events around k_raster only, 2 around every render kernel
  std::vector<cudaEvent_t> prof_events; // kProfMarks events per profiled frame
  int64_t prof_frames = 0;
  // query scratch
  double* q_in = nullptr; double* q_outd = nullptr; int32_t* q_outi = nullptr; uint32_t* q_hidden = nullptr; int q_cap = 0;
  // nccl (dlopen'ed)
  void* nccl_lib = nullptr; void* nccl_comm = nullptr;
  uint64_t launches = 0;
  bool seeded = false;
  dts_output_format fmt{DTS_OBS_HWC, DTS_OBS_U8, DTS_REWARD_RAW, DTS_ACTIONS_CONTINUOUS, 1.0};
  std::string err;

  int fail(const char* fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    err = buf;
    return 1;
  }
  template <typename T> int dalloc(T** p, size_t count, std::vector<void*>* owner = nullptr) {
    void* q = nullptr;
    cudaError_t e = cudaMalloc(&q, count * sizeof(T) + 16);
    if (e != cudaSuccess) return fail("cudaMalloc(%zu B) failed: %s", count * sizeof(T), cudaGetErrorString(e));
    cudaMemset(q, 0, count * sizeof(T) + 16);
    (owner ? *owner : allocs).push_back(q);
    *p = (T*)q;
    return 0;
  }
  template <typename T> int upload(const T** dst, const T* src, size_t count, std::vector<void*>* owner) {
    T* d = nullptr;
    if (dalloc(&d, count ? count : 1, owner)) return 1;
    if (count && src) {
      cudaError_t e = cudaMemcpy(d, src, count * sizeof(T), cudaMemcpyHostToDevice);
      if (e != cudaSuccess) return fail("cudaMemcpy H2D failed: %s", cudaGetErrorString(e));
    }
    *dst = d;
    return 0;
  }
};

extern "C" {

const char* dts_last_error(dts_sim* sim) { return sim ? sim->err.c_str() : g_create_error.c_str(); }

int dts_create(const dts_config* cfg, dts_sim** out) {
  if (!cfg || !out) { g_create_error = "null argument"; return 1; }
  if (cfg->abi_version != DTS_ABI_VERSION) { g_create_error = "dts_config.abi_version mismatch"; return 1; }
  if (cfg->num_envs <= 0 || cfg->cam_width <= 0 || cfg->cam_height <= 0 || cfg->max_maps <= 0) {
    g_create_error = "num_envs, cam_width, cam_height and max_maps must be positive";
    return 1;
  }
  if (cfg->cam_width > 800 || cfg->cam_height > 800) {  // guard band of the rasteriser: 2.5*size*64 < 2^17
    g_create_error = "camera larger than 800x800 is not supported by the rasteriser's fixed-point range";
    return 1;
  }
  cudaError_t e = cudaSetDevice(cfg->device);
  if (e != cudaSuccess) { g_create_error = std::string("cudaSetDevice failed: ") + cudaGetErrorString(e); return 1; }
  dts_sim* sim = new dts_sim();
  sim->cfg = *cfg;
  const int n = cfg->num_envs;
  StepCfg& c = sim->step_cfg;
  c.dt = 1.0 / cfg->frame_rate;                       // S:300
  c.robot_speed = cfg->robot_speed;
  c.accept_angle_deg = cfg->accept_start_angle_deg;
  c.gain = cfg->gain; c.trim = cfg->trim; c.radius = cfg->radius; c.k = cfg->k; c.limit = cfg->limit;
  c.dyn = DynParams{cfg->dyn_u1, cfg->dyn_u2, cfg->dyn_u3, cfg->dyn_w1, cfg->dyn_w2, cfg->dyn_w3,
                    cfg->dyn_uar, cfg->dyn_ual, cfg->dyn_war, cfg->dyn_wal, 0};
  // a command issued at t acts on integration intervals starting at or after t + delay
  int d = 0;
  while (d * c.dt < cfg->dyn_delay - 1e-12) d++;
  if (d > DTS_MAX_DELAY) { g_create_error = "dyn_delay exceeds DTS_MAX_DELAY steps"; delete sim; return 1; }
  c.dyn.delay_steps = d;
  c.frame_skip = cfg->frame_skip; c.max_steps = cfg->max_steps; c.action_mode = cfg->action_mode; c.flags = cfg->flags;
  c.seed = cfg->seed; c.env_id_offset = cfg->env_id_offset;
  c.random_maps = cfg->random_maps;
  c.reward_mode = DTS_REWARD_RAW; c.action_map = DTS_ACTIONS_CONTINUOUS; c.action_vel_scale = 1.0;
  if (cfg->num_tris_distractors < 0 || cfg->n_dr_ops < 0 || cfg->n_dr_ops > DTS_MAX_DR_OPS) {
    g_create_error = "num_tris_distractors / n_dr_ops out of range"; delete sim; return 1;
  }
  c.num_tris_distractors = cfg->num_tris_distractors;
  for (int k = 0; k < 3; k++) { c.color_sky[k] = cfg->color_sky[k]; c.color_ground[k] = cfg->color_ground[k]; }
  if (cfg->n_dr_ops > 0) {
    c.n_dr_ops = cfg->n_dr_ops;
    for (int k = 0; k < cfg->n_dr_ops; k++) {
      c.dr_ops[k] = cfg->dr_ops[k];
      const dts_dr_op& op = cfg->dr_ops[k];
      if (op.type < DTS_DR_INT || op.type > DTS_DR_NORMAL || op.size < 0 || op.target < DTS_DR_NONE || op.target > DTS_DR_TRIM) {
        g_create_error = "bad dts_dr_op"; delete sim; return 1;
      }
    }
  } else {   // randomization/config/default_dr.json, keys sorted (randomizer.py:33)
    const dts_dr_op def[7] = {
        {DTS_DR_UNIFORM, 1, DTS_DR_CAMERA_ANGLE, 0, {0.8, 0, 0}, {1.2, 0, 0}},
        {DTS_DR_UNIFORM, 1, DTS_DR_CAMERA_FOV_Y, 0, {0.8, 0, 0}, {1.2, 0, 0}},
        {DTS_DR_UNIFORM, 1, DTS_DR_CAMERA_HEIGHT, 0, {0.92, 0, 0}, {1.08, 0, 0}},
        {DTS_DR_UNIFORM, 3, DTS_DR_CAMERA_NOISE, 0, {-0.005, -0.005, -0.005}, {0.005, 0.005, 0.005}},
        {DTS_DR_INT, 1, DTS_DR_HORZ_MODE, 0, {0, 0, 0}, {4, 0, 0}},
        {DTS_DR_UNIFORM, 3, DTS_DR_LIGHT_POS, 0, {-150, 170, -150}, {150, 220, 150}},
        {DTS_DR_NORMAL, 1, DTS_DR_TRIM, 0, {0, 0, 0}, {0.02, 0, 0}}};
    c.n_dr_ops = 7;
    for (int k = 0; k < 7; k++) c.dr_ops[k] = def[k];
  }
  DState& S = sim->S;
  S.n = n;
  int bad = 0;
  double** dbl[] = {&S.cx, &S.cy, &S.ctheta, &S.vu, &S.vw, &S.pos_x, &S.pos_z, &S.angle, &S.speed, &S.reward,
                    &S.lane_dist, &S.lane_dot, &S.lane_angle, &S.prox, &S.wheel_dist, &S.trim};
  for (auto p : dbl) bad |= sim->dalloc(p, n);
  bad |= sim->dalloc(&S.fifo, (size_t)DTS_MAX_DELAY * 2 * n);
  int32_t** i32[] = {&S.step_count, &S.tile_i, &S.tile_j, &S.map_id, &S.episode};
  for (auto p : i32) bad |= sim->dalloc(p, n);
  uint8_t** u8[] = {&S.done_code, &S.in_lane, &S.collided};
  for (auto p : u8) bad |= sim->dalloc(p, n);
  bad |= sim->dalloc(&S.rng, 6 * (size_t)n);
  bad |= sim->dalloc(&S.rep, n);
  bad |= sim->dalloc(&sim->d_maps, cfg->max_maps);
  bad |= sim->dalloc(&sim->d_err, 32);
  if (cudaHostAlloc((void**)&sim->h_status, 64, cudaHostAllocMapped) != cudaSuccess ||
      cudaHostGetDevicePointer((void**)&sim->d_status, sim->h_status, 0) != cudaSuccess) {
    sim->fail("cudaHostAlloc(mapped status word) failed"); bad = 1;
  } else {
    memset(sim->h_status, 0, 64);
  }
  auto& st = sim->stage;
  bad |= sim->dalloc(&st.map_id, n);
  double** sd[] = {&st.pos_x, &st.pos_z, &st.angle, &st.wheel_dist, &st.trim};
  for (auto p : sd) bad |= sim->dalloc(p, n);
  for (auto& p : st.f1) bad |= sim->dalloc(&p, n);
  for (auto& p : st.f3) bad |= sim->dalloc(&p, 3 * (size_t)n);
  bad |= sim->dalloc(&st.light_pos, 4 * (size_t)n);
  bad |= sim->dalloc(&st.light_stale, n);
  bad |= sim->dalloc(&st.hidden, 8 * (size_t)n);
  if (bad) { g_create_error = sim->err; dts_destroy(sim); return 1; }
  sim->h_maps.assign(cfg->max_maps, DMap{});
  sim->map_allocs.resize(cfg->max_maps);
  *out = sim;
  return 0;
}

void dts_destroy(dts_sim* sim) {
  if (!sim) return;
  cudaSetDevice(sim->cfg.device);
  cudaDeviceSynchronize();
  for (void* p : sim->allocs) cudaFree(p);
  for (auto& v : sim->map_allocs) for (void* p : v) cudaFree(p);
  void* extra[] = {sim->render_scratch, (void*)sim->fish.src_xy, (void*)sim->fish.cbox, (void*)sim->fish.fbox, (void*)sim->fish.rbox,
                   (void*)sim->fish.cell_start, (void*)sim->fish.cell_bins, (void*)sim->fish.home_start, (void*)sim->fish.home_ent,
                   sim->q_in, sim->q_outd, sim->q_outi, sim->q_hidden};
  for (void* p : extra) if (p) cudaFree(p);
  for (int p = 0; p < sim->gather_world; p++)
    if (sim->gather_peer[p] && sim->gather_peer[p] != sim->gather_buf) cudaIpcCloseMemHandle(sim->gather_peer[p]);
  if (sim->gather_buf) cudaFree(sim->gather_buf);
  void* rz[] = {sim->resize_src, sim->resize_xtab, sim->resize_ytab};
  for (void* p : rz) if (p) cudaFree(p);
  if (sim->h_status) cudaFreeHost(sim->h_status);
  for (cudaEvent_t e : sim->prof_events) cudaEventDestroy(e);
  delete sim;
}

int dts_upload_map(dts_sim* sim, int map_id, const dts_map_blob* b) {
  if (!sim) return 1;
  if (!b || map_id < 0 || map_id >= sim->cfg.max_maps) return sim->fail("bad map_id %d", map_id);
  if (b->n_objects > DTS_MAX_OBJECTS) return sim->fail("map has %d objects, limit %d", b->n_objects, DTS_MAX_OBJECTS);
  if (b->grid_w <= 0 || b->grid_h <= 0 || !(b->tile_size > 0)) return sim->fail("invalid tile grid");
  if (b->n_dyn < 0 || b->n_dyn > DTS_MAX_DYN) return sim->fail("map has %d dynamic obstacles, limit %d", b->n_dyn, DTS_MAX_DYN);
  // validate the whole blob BEFORE the slot's previous allocations are released: a rejected upload leaves the
  // old map intact
  for (int o = 0; o < b->n_objects; o++) {
    const dts_object& s = b->objects[o];
    if (s.mesh_id < 0 || s.mesh_id >= b->n_meshes) return sim->fail("object %d: bad mesh_id", o);
    if (s.alt_tex_to >= b->n_textures || s.alt_tex_from >= b->n_textures) return sim->fail("object %d: alt texture out of range", o);
    if (s.dyn_slot >= b->n_dyn) return sim->fail("object %d: dyn_slot %d out of range", o, s.dyn_slot);
  }
  for (int t = 0; t < b->n_textures; t++) {
    const dts_texture& s = b->textures[t];
    if (s.width <= 0 || s.height <= 0 || (s.width & (s.width - 1)) || (s.height & (s.height - 1)))
      return sim->fail("texture %d: %dx%d is not a power of two", t, s.width, s.height);
  }
  for (int s = 0; s < b->n_dyn; s++) {
    const dts_dyn_object& q = b->dyn[s];
    if (q.kind != DTS_DYN_DUCKIE && q.kind != DTS_DYN_DUCKIEBOT && q.kind != DTS_DYN_TRAFFICLIGHT) return sim->fail("dyn %d: bad kind %d", s, q.kind);
    if (q.object_index < 0 || q.object_index >= b->n_objects || b->objects[q.object_index].dyn_slot != s)
      return sim->fail("dyn %d: object_index %d does not point back to this slot", s, q.object_index);
  }
  DTS_CUDA(cudaSetDevice(sim->cfg.device));
  DTS_CUDA(cudaDeviceSynchronize());
  auto& own = sim->map_allocs[map_id];
  for (void* p : own) cudaFree(p);
  own.clear();
  sim->h_maps[map_id].valid = 0;   // until the new map is complete, the slot holds nothing (a failed cudaMalloc below leaves it empty)
  DMap m{};
  const size_t T = (size_t)b->grid_w * b->grid_h;
  m.tile_size = b->tile_size; m.grid_w = b->grid_w; m.grid_h = b->grid_h; m.n_tiles = (int)T;
  int bad = 0;
  bad |= sim->upload(&m.tile_kind, b->tile_kind, T, &own);
  bad |= sim->upload(&m.tile_angle, b->tile_angle, T, &own);
  bad |= sim->upload(&m.tile_drivable, b->tile_drivable, T, &own);
  bad |= sim->upload(&m.tile_tex, b->tile_tex, T, &own);
  bad |= sim->upload(&m.tile_curve_off, b->tile_curve_off, T, &own);
  bad |= sim->upload(&m.tile_curve_cnt, b->tile_curve_cnt, T, &own);
  bad |= sim->upload(&m.curves, b->curves, (size_t)b->n_curves * 12, &own);
  m.n_coll = b->n_coll;
  bad |= sim->upload(&m.coll_corners, b->coll_corners, (size_t)b->n_coll * 8, &own);
  bad |= sim->upload(&m.coll_norms, b->coll_norms, (size_t)b->n_coll * 4, &own);
  bad |= sim->upload(&m.coll_centers, b->coll_centers, (size_t)b->n_coll * 3, &own);
  bad |= sim->upload(&m.coll_radii, b->coll_radii, (size_t)b->n_coll, &own);
  std::vector<int32_t> drv;
  for (int j = 0; j < b->grid_h; j++)       // reference scan order S:810-860
    for (int i = 0; i < b->grid_w; i++)
      if (b->tile_kind[j * b->grid_w + i] >= 0 && b->tile_drivable[j * b->grid_w + i]) { drv.push_back(i); drv.push_back(j); }
  m.start_i = b->start_tile[0]; m.start_j = b->start_tile[1];
  if (m.start_i < 0 || m.start_j < 0 || m.start_i >= b->grid_w || m.start_j >= b->grid_h) { m.start_i = -1; m.start_j = -1; }
  m.has_start_pose = b->has_start_pose != 0;
  for (int k = 0; k < 3; k++) m.start_pose[k] = b->start_pose[k];
  m.n_drivable = (int)drv.size() / 2;
  bad |= sim->upload(&m.drivable_ij, drv.data(), drv.size(), &own);
  // objects: add spawn radius (S:1467) and a bounding sphere per placed mesh
  std::vector<DObject> objs(b->n_objects);
  for (int o = 0; o < b->n_objects; o++) {
    const dts_object& s = b->objects[o];
    if (s.mesh_id < 0 || s.mesh_id >= b->n_meshes) return sim->fail("object %d: bad mesh_id", o);
    const dts_mesh& me = b->meshes[s.mesh_id];
    DObject& d = objs[o];
    for (int k = 0; k < 3; k++) { d.pos[k] = (float)s.pos[k]; d.dpos[k] = s.pos[k]; }   // glTranslatef takes floats
    d.dyn_slot = s.dyn_slot;
    d.alt_from = s.alt_tex_from; d.alt_to = s.alt_tex_to;
    if (s.alt_tex_to >= b->n_textures || s.alt_tex_from >= b->n_textures) return sim->fail("object %d: alt texture out of range", o);
    if (s.dyn_slot >= b->n_dyn) return sim->fail("object %d: dyn_slot %d out of range", o, s.dyn_slot);
    d.scale = s.scale; d.y_rot_deg = s.y_rot_deg; d.mesh_id = s.mesh_id; d.optional = s.optional;
    d.tri_offset = me.tri_offset; d.tri_count = me.tri_count;
    d.seg_tex = (me.seg_flat_tex >= 0 && me.seg_flat_tex < b->n_textures) ? me.seg_flat_tex : -1; d.pad_ = 0;
    float lo[3] = {1e30f, 1e30f, 1e30f}, hi[3] = {-1e30f, -1e30f, -1e30f};
    for (int t = 0; t < me.tri_count * 3; t++)
      for (int k = 0; k < 3; k++) {
        const float v = b->tri_pos[((size_t)me.tri_offset * 3 + t) * 3 + k];
        lo[k] = v < lo[k] ? v : lo[k];
        hi[k] = v > hi[k] ? v : hi[k];
      }
    float mx = hi[0] > hi[1] ? hi[0] : hi[1];
    mx = mx > hi[2] ? mx : hi[2];
    d.spawn_rad = mx * 0.5f * s.scale + 0.25f;     // MIN_SPAWN_OBJ_DIST S:156
    float r2 = 0.f;
    for (int k = 0; k < 3; k++) { d.centre[k] = 0.5f * (lo[k] + hi[k]); const float h = 0.5f * (hi[k] - lo[k]); r2 += h * h; }
    d.bound_rad = sqrtf(r2);
  }
  m.n_objects = b->n_objects;
  bad |= sim->upload(&m.objects, objs.data(), objs.size(), &own);
  m.n_tris = b->n_tris;
  bad |= sim->upload(&m.tri_pos, b->tri_pos, (size_t)b->n_tris * 9, &own);
  bad |= sim->upload(&m.tri_nrm, b->tri_nrm, (size_t)b->n_tris * 9, &own);
  bad |= sim->upload(&m.tri_uv, b->tri_uv, (size_t)b->n_tris * 6, &own);
  bad |= sim->upload(&m.tri_col, b->tri_col, (size_t)b->n_tris * 9, &own);
  bad |= sim->upload(&m.tri_tex, b->tri_tex, (size_t)b->n_tris, &own);
  std::vector<DTexture> tex(b->n_textures);
  {
    size_t pool_bytes = 0;
    std::vector<size_t> off(b->n_textures);
    for (int t = 0; t < b->n_textures; t++) {
      const dts_texture& s = b->textures[t];
      off[t] = pool_bytes;
      pool_bytes += ((size_t)s.width * s.height * 4 + 255) & ~size_t(255);
    }
    if (pool_bytes >= (size_t(1) << 32)) return sim->fail("textures exceed 4 GB");
    std::vector<uint8_t> pool(pool_bytes ? pool_bytes : 256, 0);
    for (int t = 0; t < b->n_textures; t++) {
      const dts_texture& s = b->textures[t];
      memcpy(pool.data() + off[t], s.rgba, (size_t)s.width * s.height * 4);
    }
    bad |= sim->upload(&m.tex_pool, pool.data(), pool.size(), &own);
    for (int t = 0; t < b->n_textures && !bad; t++) {
      const dts_texture& s = b->textures[t];
      int lw = 0, lh = 0;
      while ((1 << lw) < s.width) lw++;
      while ((1 << lh) < s.height) lh++;
      if (lw > 15 || lh > 15) return sim->fail("texture %d: %dx%d too large", t, s.width, s.height);
      tex[t].w = s.width; tex[t].h = s.height; tex[t].rgba = m.tex_pool + off[t];
      tex[t].info = (uint32_t)(off[t] >> 8) | ((uint32_t)lw << 24) | ((uint32_t)lh << 28);
      tex[t].pad = 0;
    }
  }
  m.n_textures = b->n_textures;
  bad |= sim->upload(&m.textures, tex.data(), tex.size(), &own);
  {
    std::vector<int16_t> seg(b->n_textures > 0 ? b->n_textures : 1);
    for (int t = 0; t < b->n_textures; t++) {
      const int v = b->tex_segment ? b->tex_segment[t] : -1;
      seg[t] = (int16_t)((v >= 0 && v < b->n_textures) ? v : t);
    }
    bad |= sim->upload(&m.tex_segment, seg.data(), seg.size(), &own);
    DObject ag{};
    if (b->agent_mesh >= 0 && b->agent_mesh < b->n_meshes) {   // self.mesh, drawn by top-down views at cur_pos (S:1923-1929)
      const dts_mesh& me = b->meshes[b->agent_mesh];
      ag.scale = 1.0f; ag.mesh_id = b->agent_mesh; ag.tri_offset = me.tri_offset; ag.tri_count = me.tri_count;
      ag.dyn_slot = -1; ag.alt_from = ag.alt_to = -1;
      ag.seg_tex = (me.seg_flat_tex >= 0 && me.seg_flat_tex < b->n_textures) ? me.seg_flat_tex : -1;
      float lo[3] = {1e30f, 1e30f, 1e30f}, hi[3] = {-1e30f, -1e30f, -1e30f};
      for (int t = 0; t < me.tri_count * 3; t++)
        for (int k = 0; k < 3; k++) {
          const float v = b->tri_pos[((size_t)me.tri_offset * 3 + t) * 3 + k];
          lo[k] = v < lo[k] ? v : lo[k];
          hi[k] = v > hi[k] ? v : hi[k];
        }
      float r2 = 0.f;
      for (int k = 0; k < 3; k++) { ag.centre[k] = 0.5f * (lo[k] + hi[k]); const float h = 0.5f * (hi[k] - lo[k]); r2 += h * h; }
      ag.bound_rad = sqrtf(r2);
    }
    m.agent = ag;
  }
  // dynamic obstacles: constants + every env's copy of the load-time state ([field][slot][env])
  m.n_dyn = b->n_dyn;
  {
    const size_t N = sim->cfg.num_envs, D = b->n_dyn;
    std::vector<DDyn> par(D);
    std::vector<double> st((size_t)DTS_DYN_FIELDS * D * N);
    for (size_t s = 0; s < D; s++) {
      const dts_dyn_object& q = b->dyn[s];
      if (q.kind != DTS_DYN_DUCKIE && q.kind != DTS_DYN_DUCKIEBOT && q.kind != DTS_DYN_TRAFFICLIGHT) return sim->fail("dyn %zu: bad kind %d", s, q.kind);
      if (q.object_index < 0 || q.object_index >= b->n_objects || b->objects[q.object_index].dyn_slot != (int)s)
        return sim->fail("dyn %zu: object_index %d does not point back to this slot", s, q.object_index);
      DDyn& p = par[s];
      p.kind = q.kind; p.object_index = q.object_index; p.pos_y = q.pos[1];
      for (int k = 0; k < 4; k++) p.norms[k] = q.norms[k / 2][k % 2];
      p.safety_radius = q.safety_radius; p.walk_distance = q.walk_distance; p.wiggle = q.wiggle; p.angle0 = q.angle;
      p.follow_dist = q.follow_dist; p.velocity = q.velocity; p.gain = q.gain; p.trim = q.trim; p.radius = q.radius;
      p.k = q.k; p.limit = q.limit; p.wheel_dist = q.wheel_dist; p.robot_width = q.robot_width; p.robot_length = q.robot_length;
      double f[DTS_DYN_FIELDS] = {};
      f[DTS_DYN_PX] = q.pos[0]; f[DTS_DYN_PZ] = q.pos[2]; f[DTS_DYN_ANGLE] = q.angle;
      f[DTS_DYN_YROT] = q.angle * (180.0 / 3.14159265358979323846);       // np.rad2deg O:57
      for (int k = 0; k < 4; k++) { f[DTS_DYN_CORNERS + 2 * k] = q.corners[k][0]; f[DTS_DYN_CORNERS + 2 * k + 1] = q.corners[k][1]; }
      f[DTS_DYN_START_X] = q.pos[0]; f[DTS_DYN_START_Z] = q.pos[2];
      f[DTS_DYN_WAIT] = q.wait_time; f[DTS_DYN_VEL] = q.vel; f[DTS_DYN_TIME] = 0.0; f[DTS_DYN_ACTIVE] = 0.0;
      p.freq = q.freq; p.tl_first = -1; p.pad = 0;
      if (q.kind == DTS_DYN_TRAFFICLIGHT) f[DTS_DYN_PATTERN] = q.pattern ? 1.0 : 0.0;
      for (int k = 0; k < DTS_DYN_FIELDS; k++)
        for (size_t e = 0; e < N; e++) st[((size_t)k * D + s) * N + e] = f[k];
    }
    int tl_first = -1, tl_last = -1;
    for (size_t s = 0; s < D; s++)
      if (par[s].kind == DTS_DYN_TRAFFICLIGHT) { if (tl_first < 0) tl_first = (int)s; tl_last = (int)s; }
    for (size_t s = 0; s < D; s++) par[s].tl_first = tl_first;
    if (tl_first >= 0)   // every constructor assigns the shared mesh's card (O:453): the last light's pattern shows
      for (size_t e = 0; e < N; e++) st[((size_t)DTS_DYN_SHOWN * D + tl_first) * N + e] = b->dyn[tl_last].pattern ? 1.0 : 0.0;
    bad |= sim->upload(&m.dyn, par.data(), par.size(), &own);
    const double* dst = nullptr;
    bad |= sim->upload(&dst, st.data(), st.size(), &own);
    m.dyn_state = const_cast<double*>(dst);
    std::vector<double> init((size_t)DTS_DYN_FIELDS * D);
    for (int k = 0; k < DTS_DYN_FIELDS; k++)
      for (size_t s = 0; s < D; s++) init[(size_t)k * D + s] = N ? st[((size_t)k * D + s) * N] : 0.0;
    bad |= sim->upload(&m.dyn_init, init.data(), init.size(), &own);
  }
  if (bad) {
    DMap empty{};
    cudaMemcpy(sim->d_maps + map_id, &empty, sizeof(DMap), cudaMemcpyHostToDevice);
    return 1;
  }
  m.valid = 1;
  if (sim->render_scratch) { cudaFree(sim->render_scratch); sim->render_scratch = nullptr; }   // re-sized for the new scene on the next render
  sim->h_maps[map_id] = m;
  DTS_CUDA(cudaMemcpy(sim->d_maps + map_id, &m, sizeof(DMap), cudaMemcpyHostToDevice));
  return 0;
}

int dts_set_fisheye_lut(dts_sim* sim, const float* rmapx, const float* rmapy, int width, int height) {
  if (!sim) return 1;
  if (!rmapx || !rmapy) return sim->fail("fisheye LUT is NULL");
  if (width != sim->cfg.cam_width || height != sim->cfg.cam_height)
    return sim->fail("fisheye LUT is %dx%d but the camera is %dx%d", width, height, sim->cfg.cam_width, sim->cfg.cam_height);
  DTS_CUDA(cudaSetDevice(sim->cfg.device));
  // distortion.py:118 gathers img[rint(rmapy), rint(rmapx)].  The rasteriser renders those source pixels directly
  // (FishTab): per output pixel the source position, per 8x4 fine / 32x8 coarse output bin / row of coarse bins the
  // bounding box of its source pixels (the bins prims are sorted into).
  const int W = width, H = height;
  const int cbx_n = (W + 31) / 32, cby_n = (H + 7) / 8, cbins = cbx_n * cby_n;
  std::vector<int32_t> src((size_t)W * H);
  const short4 empty = make_short4(32767, 32767, -32768, -32768);
  std::vector<short4> cbox(cbins, empty), fbox((size_t)cbins * 8, empty), rbox(cby_n, empty);
  auto grow = [](short4& b, int x, int y) {
    b.x = (short)(x < b.x ? x : b.x); b.y = (short)(y < b.y ? y : b.y);
    b.z = (short)(x > b.z ? x : b.z); b.w = (short)(y > b.w ? y : b.w);
  };
  for (int y = 0; y < H; y++)
    for (int x = 0; x < W; x++) {
      const float fx = rmapx[(size_t)y * W + x], fy = rmapy[(size_t)y * W + x];
      // NaN, +-inf and |v| >= 2^31 have no int value (the cast would be undefined): such entries point outside
      const bool finite = fabsf(fx) < 2147483648.0f && fabsf(fy) < 2147483648.0f;
      const int sx = finite ? (int)rintf(fx) : -1, sy = finite ? (int)rintf(fy) : -1;   // round-half-even like the kernel's rintf
      const bool ok = sx >= 0 && sx < W && sy >= 0 && sy < H;
      src[(size_t)y * W + x] = ok ? (int32_t)((uint32_t)(sx & 0xffff) | ((uint32_t)sy << 16)) : (int32_t)0x80008000u;
      if (!ok) continue;
      const int cb = (y / 8) * cbx_n + x / 32, f = ((y & 7) >> 2) * 4 + ((x & 31) >> 3);
      grow(cbox[cb], sx, sy); grow(fbox[(size_t)cb * 8 + f], sx, sy); grow(rbox[y / 8], sx, sy);
    }
  // int32 edge functions inside a coarse bin need |A x + B y| < 2^30 over its source box: |A| <= 5*64*H, |B| <= 5*64*W
  // (4x guard band), x <= 64*w, y <= 64*h  ->  H*w + W*h < 2^30 / (5*64*64)
  for (int b = 0; b < cbins; b++) {
    if (cbox[b].z < cbox[b].x) continue;
    const long long w = cbox[b].z - cbox[b].x + 2, h = cbox[b].w - cbox[b].y + 2;
    if ((long long)H * w + (long long)W * h >= (1LL << 30) / (5 * 64 * 64))
      return sim->fail("fisheye LUT sends output bin %d to a %lldx%lld px source region: too wide for the rasteriser's int32 edge functions", b, w, h);
  }
  // inverse index: source cell (same 32x8 grid, over the source image) -> output bins whose source box meets it
  std::vector<int32_t> cell_start(cbins + 1, 0);
  std::vector<uint16_t> cell_bins;
  {
    std::vector<std::vector<uint16_t>> lists(cbins);
    for (int b = 0; b < cbins; b++) {
      if (cbox[b].z < cbox[b].x) continue;
      for (int cy = cbox[b].y / 8; cy <= cbox[b].w / 8; cy++)
        for (int cx = cbox[b].x / 32; cx <= cbox[b].z / 32; cx++) lists[cy * cbx_n + cx].push_back((uint16_t)b);
    }
    for (int c = 0; c < cbins; c++) {
      cell_start[c] = (int32_t)cell_bins.size();
      cell_bins.insert(cell_bins.end(), lists[c].begin(), lists[c].end());
    }
    cell_start[cbins] = (int32_t)cell_bins.size();
    if (cell_bins.empty()) cell_bins.push_back(0);
  }
  // ... and the index by HOME cell (the cell of the box's top-left corner): each bin once, with its box
  std::vector<int32_t> home_start(cbins + 1, 0);
  std::vector<int4> home_ent;
  int ext_x = 0, ext_y = 0;
  {
    std::vector<std::vector<int>> lists(cbins);
    for (int b = 0; b < cbins; b++) {
      if (cbox[b].z < cbox[b].x) continue;
      lists[(cbox[b].y / 8) * cbx_n + cbox[b].x / 32].push_back(b);
      ext_x = std::max(ext_x, cbox[b].z / 32 - cbox[b].x / 32);
      ext_y = std::max(ext_y, cbox[b].w / 8 - cbox[b].y / 8);
    }
    for (int c = 0; c < cbins; c++) {
      home_start[c] = (int32_t)home_ent.size();
      for (int b : lists[c])
        home_ent.push_back(make_int4((int)((uint32_t)(uint16_t)cbox[b].x | ((uint32_t)(uint16_t)cbox[b].y << 16)),
                                     (int)((uint32_t)(uint16_t)cbox[b].z | ((uint32_t)(uint16_t)cbox[b].w << 16)), b, 0));
    }
    home_start[cbins] = (int32_t)home_ent.size();
    if (home_ent.empty()) home_ent.push_back(make_int4(0, 0, 0, 0));
  }
  void* old[] = {(void*)sim->fish.src_xy, (void*)sim->fish.cbox, (void*)sim->fish.fbox, (void*)sim->fish.rbox,
                 (void*)sim->fish.cell_start, (void*)sim->fish.cell_bins, (void*)sim->fish.home_start, (void*)sim->fish.home_ent};
  DTS_CUDA(cudaDeviceSynchronize());
  for (void* p : old) if (p) cudaFree(p);
  sim->fish = FishTab{};
  int32_t* d_src = nullptr; short4 *d_c = nullptr, *d_f = nullptr, *d_r = nullptr;
  DTS_CUDA(cudaMalloc(&d_src, src.size() * sizeof(int32_t)));
  DTS_CUDA(cudaMalloc(&d_c, cbox.size() * sizeof(short4)));
  DTS_CUDA(cudaMalloc(&d_f, fbox.size() * sizeof(short4)));
  DTS_CUDA(cudaMalloc(&d_r, rbox.size() * sizeof(short4)));
  DTS_CUDA(cudaMemcpy(d_src, src.data(), src.size() * sizeof(int32_t), cudaMemcpyHostToDevice));
  DTS_CUDA(cudaMemcpy(d_c, cbox.data(), cbox.size() * sizeof(short4), cudaMemcpyHostToDevice));
  DTS_CUDA(cudaMemcpy(d_f, fbox.data(), fbox.size() * sizeof(short4), cudaMemcpyHostToDevice));
  DTS_CUDA(cudaMemcpy(d_r, rbox.data(), rbox.size() * sizeof(short4), cudaMemcpyHostToDevice));
  int32_t* d_cs = nullptr; uint16_t* d_cb = nullptr;
  DTS_CUDA(cudaMalloc(&d_cs, cell_start.size() * sizeof(int32_t)));
  DTS_CUDA(cudaMalloc(&d_cb, cell_bins.size() * sizeof(uint16_t)));
  DTS_CUDA(cudaMemcpy(d_cs, cell_start.data(), cell_start.size() * sizeof(int32_t), cudaMemcpyHostToDevice));
  DTS_CUDA(cudaMemcpy(d_cb, cell_bins.data(), cell_bins.size() * sizeof(uint16_t), cudaMemcpyHostToDevice));
  int32_t* d_hs = nullptr; int4* d_he = nullptr;
  DTS_CUDA(cudaMalloc(&d_hs, home_start.size() * sizeof(int32_t)));
  DTS_CUDA(cudaMalloc(&d_he, home_ent.size() * sizeof(int4)));
  DTS_CUDA(cudaMemcpy(d_hs, home_start.data(), home_start.size() * sizeof(int32_t), cudaMemcpyHostToDevice));
  DTS_CUDA(cudaMemcpy(d_he, home_ent.data(), home_ent.size() * sizeof(int4), cudaMemcpyHostToDevice));
  sim->fish = FishTab{d_src, d_c, d_f, d_r, d_cs, d_cb, d_hs, d_he, ext_x, ext_y};
  return 0;
}

// > 0: round-robin over that many slots; < 0: uniform draw over -n slots; 0: the env keeps its map
static int map_select(const dts_sim* sim) { return sim->cfg.random_maps > 0 ? -sim->cfg.random_maps : sim->cfg.cycle_maps; }

static int check_maps(dts_sim* sim) {
  if (!sim->h_maps[0].valid) return sim->fail("no map uploaded in slot 0");
  const int cyc = sim->cfg.cycle_maps > sim->cfg.random_maps ? sim->cfg.cycle_maps : sim->cfg.random_maps;
  for (int k = 0; k < cyc; k++)
    if (k >= sim->cfg.max_maps || !sim->h_maps[k].valid) return sim->fail("cycle_maps / random_maps = %d but slot %d is empty", cyc, k);
  return 0;
}

int dts_reset(dts_sim* sim, const uint8_t* mask_dev, const dts_episode_params* p, void* stream) {
  if (!sim) return 1;
  if (check_maps(sim)) return 1;
  DTS_CUDA(cudaSetDevice(sim->cfg.device));
  cudaStream_t st = (cudaStream_t)stream;
  const size_t n = sim->cfg.num_envs;
  ResetStaging rs{};
  auto& sg = sim->stage;
  dts_episode_params z{};
  if (!p) p = &z;
  if (p->map_id) {
    for (size_t e = 0; e < n; e++)
      if (p->map_id[e] < 0 || p->map_id[e] >= sim->cfg.max_maps || !sim->h_maps[p->map_id[e]].valid)
        return sim->fail("episode map_id[%zu]=%d has no uploaded map", e, p->map_id[e]);
  }
#define STAGE(field, dst, cnt)                                                                         \
  if (p->field) { DTS_CUDA(cudaMemcpyAsync(dst, p->field, (cnt) * sizeof(*p->field), cudaMemcpyHostToDevice, st)); rs.field = dst; }
  STAGE(map_id, sg.map_id, n)
  STAGE(pos_x, sg.pos_x, n) STAGE(pos_z, sg.pos_z, n) STAGE(angle, sg.angle, n)
  STAGE(wheel_dist, sg.wheel_dist, n) STAGE(trim, sg.trim, n)
  STAGE(cam_height, sg.f1[0], n) STAGE(cam_angle_deg, sg.f1[1], n) STAGE(cam_fov_y_deg, sg.f1[2], n)
  STAGE(cam_noise, sg.f3[0], 3 * n) STAGE(horizon_color, sg.f3[1], 3 * n) STAGE(light_ambient, sg.f3[2], 3 * n)
  STAGE(light_diffuse, sg.f3[3], 3 * n) STAGE(ground_color, sg.f3[4], 3 * n)
  STAGE(light_pos, sg.light_pos, 4 * n) STAGE(light_stale, sg.light_stale, n) STAGE(obj_hidden, sg.hidden, 8 * n)
#undef STAGE
  launch_reset_params(sim->S, sim->d_maps, sim->step_cfg, mask_dev, rs, st);
  sim->launches++;
  DTS_CUDA(cudaGetLastError());
  // the staging buffers are pageable-host copies: make them safe to reuse before returning
  DTS_CUDA(cudaStreamSynchronize(st));
  return 0;
}

int dts_seed_streams(dts_sim* sim, const uint8_t* mask_host, const uint64_t* streams) {
  if (!sim) return 1;
  if (!streams) return sim->fail("streams is NULL");
  DTS_CUDA(cudaSetDevice(sim->cfg.device));
  const size_t n = sim->cfg.num_envs;
  std::vector<uint64_t> soa(6 * n);
  DTS_CUDA(cudaMemcpy(soa.data(), sim->S.rng, 6 * n * sizeof(uint64_t), cudaMemcpyDeviceToHost));
  for (size_t e = 0; e < n; e++) {
    if (mask_host && !mask_host[e]) continue;
    for (int k = 0; k < 6; k++) soa[k * n + e] = streams[6 * e + k];
  }
  DTS_CUDA(cudaMemcpy(sim->S.rng, soa.data(), 6 * n * sizeof(uint64_t), cudaMemcpyHostToDevice));
  sim->seeded = true;
  return 0;
}

int dts_reset_random(dts_sim* sim, const uint8_t* mask_dev, void* stream) {
  if (!sim) return 1;
  if (check_maps(sim)) return 1;
  if (!sim->seeded) return sim->fail("dts_seed_streams must be called before a device-side reset");
  DTS_CUDA(cudaSetDevice(sim->cfg.device));
  launch_reset_random(sim->S, sim->d_maps, sim->step_cfg, map_select(sim), mask_dev, (cudaStream_t)stream);
  sim->launches++;
  DTS_CUDA(cudaGetLastError());
  return 0;
}

static int ensure_render(dts_sim* sim) {
  if (sim->render_scratch) return 0;
  int sms = 148;
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, sim->cfg.device);
  const bool tess = (sim->cfg.flags & DTS_FLAG_TESSELLATE) != 0;
  int max_tris = 2, max_lat = 1, items_max = 1;
  for (const DMap& m : sim->h_maps) {
    if (!m.valid) continue;
    int t = 2 + (tess ? 98 : 6) * m.n_tiles + m.agent.tri_count;   // a clipped tile quad fans into a few triangles
    std::vector<DObject> objs(m.n_objects);
    if (m.n_objects) cudaMemcpy(objs.data(), m.objects, sizeof(DObject) * m.n_objects, cudaMemcpyDeviceToHost);
    for (const DObject& o : objs) t += o.tri_count;
    max_tris = t > max_tris ? t : max_tris;
    max_lat = m.n_tiles > max_lat ? m.n_tiles : max_lat;
    const int items = 1 + m.n_tiles + m.n_objects + 1;   // + the agent's own mesh (top-down views)
    items_max = items > items_max ? items : items_max;
  }
  sim->render_ctas = sms * render_ctas_per_sm();
  sim->max_prims = max_tris + max_tris / 4 + 64;  // clipping can add fan triangles
  if (items_max > 65535) return sim->fail("scene too large: %d draw items per frame (limit 65535)", items_max);
  if (sim->max_prims > 65535) return sim->fail("scene too large: %d triangles per frame (limit 65535)", sim->max_prims);
  sim->max_lat = max_lat;
  sim->items_max = items_max;
  const int cbins = ((sim->cfg.cam_width + 31) / 32) * ((sim->cfg.cam_height + 7) / 8);
  // (prim, coarse bin) pairs.  Upper bound per env: the ground fan (<= 8 x cbins), a few screen-filling tiles and one
  // screen-filling prop; under the fused fisheye the bins are overlapping source boxes (x ~4).  The batch shares ONE
  // pool, each env taking exactly what its frame needs: capacity = that bound x num_envs, capped at DTS_PAIR_POOL_GB
  // (default 16) of records — a typical frame uses a small fraction of its bound.
  const long long per_env = (3LL * sim->max_prims + 24LL * cbins + 256) * ((sim->cfg.flags & DTS_FLAG_DISTORTION) ? 4 : 1);
  double pool_gb = 16.0;
  if (const char* e = getenv("DTS_PAIR_POOL_GB")) pool_gb = atof(e) > 0 ? atof(e) : pool_gb;
  long long pool = per_env * sim->cfg.num_envs;
  const long long cap = (long long)(pool_gb * 1073741824.0 / 84.0);
  if (pool > cap) pool = cap;
  if (pool > 2000000000LL) pool = 2000000000LL;
  if (pool < per_env) pool = per_env;
  sim->bin_cap = (int)pool;
  const size_t frame = (size_t)sim->items_max;   // (env, item) work-list entries per env
  const size_t bytes = render_scratch_bytes(sim->cfg.num_envs, sim->max_prims, cbins, sim->bin_cap, sim->max_lat, frame);
  cudaError_t e = cudaMalloc(&sim->render_scratch, bytes);
  if (e != cudaSuccess) return sim->fail("render scratch cudaMalloc(%zu) failed: %s", bytes, cudaGetErrorString(e));
  return 0;
}

int dts_render(dts_sim* sim, void* obs_dev, void* stream) {
  if (!sim) return 1;
  if (!obs_dev) return sim->fail("obs_dev is NULL");
  if (check_maps(sim)) return 1;
  DTS_CUDA(cudaSetDevice(sim->cfg.device));
  if (ensure_render(sim)) return 1;
  if ((sim->cfg.flags & DTS_FLAG_DISTORTION) && !sim->fish.src_xy) return sim->fail("distortion enabled but no fisheye LUT set");
  RenderCfg rc{sim->cfg.cam_width, sim->cfg.cam_height, sim->cfg.flags, sim->cfg.num_envs,
               (sim->cfg.flags & DTS_FLAG_TESSELLATE) ? 1 : 0, sim->fmt.obs_layout, sim->fmt.obs_dtype, sim->render_mode};
  if (*(volatile int32_t*)sim->h_status & 1)
    return sim->fail("an earlier frame overflowed its render frame memory (prim slab / bin lists) and was left incomplete");
  cudaEvent_t* marks = nullptr;
  if (sim->profiling) {
    const size_t base = sim->prof_events.size();
    sim->prof_events.resize(base + kProfMarks);
    for (int k = 0; k < kProfMarks; k++) DTS_CUDA(cudaEventCreate(&sim->prof_events[base + k]));
    marks = sim->prof_events.data() + base;
    sim->prof_frames++;
  }
  const int mark_level = sim->profiling;
  void* target = obs_dev;
  if (sim->resize_w) {   // render full size, packed u8 HWC, into the library's buffer; k_resize writes the caller's tensor
    rc.obs_layout = DTS_OBS_HWC; rc.obs_dtype = DTS_OBS_U8;
    target = sim->resize_src;
  }
  GatherTab gt{};
  if (sim->gather_next) {
    if (sim->resize_w) return sim->fail("the fused gather writes the rasteriser's own output: not combined with dts_set_resize");
    gt.n = sim->gather_world;
    for (int p = 0; p < sim->gather_world; p++)
      gt.base[p] = reinterpret_cast<uint8_t*>(sim->gather_peer[p]) + (uint64_t)sim->gather_rank * sim->gather_bytes;
    sim->gather_next = false;
  }
  int k = launch_render(sim->S, sim->d_maps, rc, target, sim->render_scratch, sim->render_ctas, sim->max_prims,
                        sim->bin_cap, sim->max_lat, sim->items_max, sim->fish, gt, sim->d_err,
                        sim->d_status, marks, mark_level, (cudaStream_t)stream);
  if (sim->resize_w) {
    launch_resize(sim->resize_src, sim->cfg.cam_width, sim->cfg.cam_height, sim->resize_w, sim->resize_h, sim->cfg.num_envs,
                  sim->resize_xtab, sim->resize_ytab, obs_dev, sim->fmt.obs_layout, sim->fmt.obs_dtype, sim->resize_band, sim->resize_cap,
                  (cudaStream_t)stream);
    k++;
  }
  if (marks && mark_level >= 2) cudaEventRecord(marks[kProfMarks - 1], (cudaStream_t)stream);   // closes the "post" interval
  sim->launches += k;
  DTS_CUDA(cudaGetLastError());
  return 0;
}

int dts_step(dts_sim* sim, const float* actions_dev, void* obs_dev, float* reward_dev, uint8_t* done_dev,
             void* stream) {
  if (!sim) return 1;
  if (!actions_dev) return sim->fail("actions_dev is NULL");
  if (check_maps(sim)) return 1;
  DTS_CUDA(cudaSetDevice(sim->cfg.device));
  if ((sim->cfg.flags & DTS_FLAG_AUTO_RESET) && !sim->seeded)
    return sim->fail("auto-reset needs seeded streams: call dts_seed_streams first");
  launch_step_logic(sim->S, sim->d_maps, sim->step_cfg, map_select(sim), actions_dev, reward_dev, done_dev,
                    (cudaStream_t)stream);
  sim->launches++;
  DTS_CUDA(cudaGetLastError());
  if (obs_dev) return dts_render(sim, obs_dev, stream);
  return 0;
}

int dts_get_state(dts_sim* sim, dts_state_view* v) {
  if (!sim || !v) return 1;
  const DState& S = sim->S;
  *v = dts_state_view{S.pos_x, S.pos_z, S.angle, S.speed, S.reward, S.lane_dist, S.lane_dot, S.lane_angle, S.prox,
                      S.wheel_dist, S.step_count, S.tile_i, S.tile_j, S.map_id, S.episode, S.done_code, S.in_lane,
                      S.collided};
  return 0;
}

int dts_query_poses(dts_sim* sim, int map_id, int dyn_env, int n, const double* query, const uint32_t* hidden,
                    double* out_f64, int32_t* out_i32, void* stream) {
  cudaStream_t qs = (cudaStream_t)stream;   // ordered after the caller's in-flight steps (they move the dynamic obstacles)
  if (!sim) return 1;
  if (map_id < 0 || map_id >= sim->cfg.max_maps || !sim->h_maps[map_id].valid) return sim->fail("bad map_id %d", map_id);
  if (dyn_env >= sim->cfg.num_envs) return sim->fail("dyn_env %d out of range", dyn_env);
  if (n <= 0) return 0;
  DTS_CUDA(cudaSetDevice(sim->cfg.device));
  if (n > sim->q_cap) {
    void* old[] = {sim->q_in, sim->q_outd, sim->q_outi, sim->q_hidden};
    for (void* p : old) if (p) cudaFree(p);
    sim->q_cap = n;
    DTS_CUDA(cudaMalloc(&sim->q_in, (size_t)n * 32));
    DTS_CUDA(cudaMalloc(&sim->q_outd, (size_t)n * 32));
    DTS_CUDA(cudaMalloc(&sim->q_outi, (size_t)n * 32));
    DTS_CUDA(cudaMalloc(&sim->q_hidden, (size_t)n * 32));
  }
  DTS_CUDA(cudaMemcpyAsync(sim->q_in, query, (size_t)n * 32, cudaMemcpyHostToDevice, qs));
  if (hidden) DTS_CUDA(cudaMemcpyAsync(sim->q_hidden, hidden, (size_t)n * 32, cudaMemcpyHostToDevice, qs));
  launch_query(sim->d_maps, map_id, dyn_env < 0 ? -1 : dyn_env, sim->cfg.num_envs, n, sim->q_in, hidden ? sim->q_hidden : nullptr, sim->q_outd, sim->q_outi, qs);
  sim->launches++;
  DTS_CUDA(cudaGetLastError());
  DTS_CUDA(cudaMemcpyAsync(out_f64, sim->q_outd, (size_t)n * 32, cudaMemcpyDeviceToHost, qs));
  DTS_CUDA(cudaMemcpyAsync(out_i32, sim->q_outi, (size_t)n * 32, cudaMemcpyDeviceToHost, qs));
  DTS_CUDA(cudaStreamSynchronize(qs));
  return 0;
}

int dts_assign_maps(dts_sim* sim, const uint8_t* mask_dev, const int32_t* map_id_host, void* stream) {
  if (!sim) return 1;
  if (!map_id_host) return sim->fail("map_id_host is NULL");
  const size_t n = sim->cfg.num_envs;
  for (size_t e = 0; e < n; e++)
    if (map_id_host[e] < 0 || map_id_host[e] >= sim->cfg.max_maps || !sim->h_maps[map_id_host[e]].valid)
      return sim->fail("dts_assign_maps: map_id[%zu]=%d has no uploaded map", e, map_id_host[e]);
  DTS_CUDA(cudaSetDevice(sim->cfg.device));
  cudaStream_t st = (cudaStream_t)stream;
  DTS_CUDA(cudaMemcpyAsync(sim->stage.map_id, map_id_host, n * sizeof(int32_t), cudaMemcpyHostToDevice, st));
  launch_assign_maps(sim->S, sim->d_maps, mask_dev, sim->stage.map_id, st);
  sim->launches++;
  DTS_CUDA(cudaGetLastError());
  DTS_CUDA(cudaStreamSynchronize(st));   // pageable host source
  return 0;
}

// cv2.resize INTER_CUBIC tap table of one axis (OpenCV resize(): fx = (float)((d + 0.5) * scale - 0.5), interpolateCubic
// with A = -0.75 in float32, taps = saturate_cast<short>(w * 2048), indices clamped to the image)
static void cubic_axis_table(int src, int dst, std::vector<int16_t>& tab) {
  tab.assign((size_t)dst * 8, 0);
  const double inv = (double)dst / (double)src, scale = 1.0 / inv;
  for (int d = 0; d < dst; d++) {
    float fx = (float)((d + 0.5) * scale - 0.5);
    const int sx = (int)floorf(fx);
    fx -= (float)sx;
    const float A = -0.75f, x = fx;
    float c[4];
    c[0] = ((A * (x + 1) - 5 * A) * (x + 1) + 8 * A) * (x + 1) - 4 * A;
    c[1] = ((A + 2) * x - (A + 3)) * x * x + 1;
    c[2] = ((A + 2) * (1 - x) - (A + 3)) * (1 - x) * (1 - x) + 1;
    c[3] = 1.f - c[0] - c[1] - c[2];
    for (int k = 0; k < 4; k++) {
      int idx = sx - 1 + k;
      idx = idx < 0 ? 0 : (idx > src - 1 ? src - 1 : idx);
      tab[(size_t)d * 8 + k] = (int16_t)idx;
      tab[(size_t)d * 8 + 4 + k] = (int16_t)lrintf(c[k] * 2048.0f);
    }
  }
}

int dts_set_resize(dts_sim* sim, int out_w, int out_h) {
  if (!sim) return 1;
  if (out_w < 0 || out_h < 0 || (out_w == 0) != (out_h == 0)) return sim->fail("bad resize target %dx%d", out_w, out_h);
  if (out_w > 4096 || out_h > 4096) return sim->fail("resize target %dx%d too large", out_w, out_h);
  DTS_CUDA(cudaSetDevice(sim->cfg.device));
  DTS_CUDA(cudaDeviceSynchronize());
  void* old[] = {sim->resize_src, sim->resize_xtab, sim->resize_ytab};
  for (void* p : old) if (p) cudaFree(p);
  sim->resize_src = nullptr; sim->resize_xtab = sim->resize_ytab = nullptr;
  sim->resize_w = sim->resize_h = 0;
  if (!out_w) return 0;
  std::vector<int16_t> xt, yt;
  cubic_axis_table(sim->cfg.cam_width, out_w, xt);
  cubic_axis_table(sim->cfg.cam_height, out_h, yt);
  DTS_CUDA(cudaMalloc(&sim->resize_src, (size_t)sim->cfg.num_envs * sim->cfg.cam_width * sim->cfg.cam_height * 3));
  DTS_CUDA(cudaMalloc(&sim->resize_xtab, xt.size() * 2));
  DTS_CUDA(cudaMalloc(&sim->resize_ytab, yt.size() * 2));
  DTS_CUDA(cudaMemcpy(sim->resize_xtab, xt.data(), xt.size() * 2, cudaMemcpyHostToDevice));
  DTS_CUDA(cudaMemcpy(sim->resize_ytab, yt.data(), yt.size() * 2, cudaMemcpyHostToDevice));
  sim->resize_w = out_w; sim->resize_h = out_h;
  // band height of the tiled kernel: the tallest band (<= 16 output rows) whose source rows + horizontal sums fit in 40 KB
  // of shared memory (several CTAs per SM); 0 = no band fits even in the opt-in maximum, use the untiled kernel
  sim->resize_band = sim->resize_cap = 0;
  const char* untiled = getenv("DTS_RESIZE_UNTILED");   // A/B switch
  const size_t budget = (size_t)(getenv("DTS_RESIZE_SMEM_KB") ? atoi(getenv("DTS_RESIZE_SMEM_KB")) : 40) * 1024;   // A/B: shared memory per band
  for (int R = 16; R >= 1 && !(untiled && untiled[0] == '1'); R--) {
    int cap = 0;
    for (int r0 = 0; r0 < out_h; r0 += R) {
      const int r1 = std::min(r0 + R, out_h);
      cap = std::max(cap, (int)yt[(size_t)8 * (r1 - 1) + 3] - (int)yt[(size_t)8 * r0] + 1);
    }
    const size_t smem = resize_band_smem(sim->cfg.cam_width, out_w, cap);
    if (smem <= budget || (R == 1 && smem <= 200 * 1024)) { sim->resize_band = R; sim->resize_cap = cap; break; }
  }
  return 0;
}

// ---- fused end-of-rollout gather: peer buffers over cudaIpc, written by the rasteriser itself --------------------
int dts_gather_alloc(dts_sim* sim, uint64_t bytes_per_rank, int rank, int world, uint8_t handle_out[64], void** buf_out) {
  if (!sim) return 1;
  if (world < 1 || world > DTS_MAX_PEERS || rank < 0 || rank >= world) return sim->fail("bad rank %d / world %d (max %d)", rank, world, DTS_MAX_PEERS);
  static_assert(sizeof(cudaIpcMemHandle_t) == 64, "cudaIpcMemHandle_t is 64 bytes");
  DTS_CUDA(cudaSetDevice(sim->cfg.device));
  if (sim->gather_buf) return sim->fail("gather buffer already allocated");
  DTS_CUDA(cudaMalloc(&sim->gather_buf, bytes_per_rank * (uint64_t)world));
  DTS_CUDA(cudaMemset(sim->gather_buf, 0, bytes_per_rank * (uint64_t)world));
  sim->gather_bytes = bytes_per_rank; sim->gather_rank = rank; sim->gather_world = world;
  for (int p = 0; p < DTS_MAX_PEERS; p++) sim->gather_peer[p] = nullptr;
  sim->gather_peer[rank] = sim->gather_buf;
  cudaIpcMemHandle_t h;
  DTS_CUDA(cudaIpcGetMemHandle(&h, sim->gather_buf));
  memcpy(handle_out, &h, 64);
  if (buf_out) *buf_out = sim->gather_buf;
  return 0;
}

int dts_gather_open(dts_sim* sim, const uint8_t* handles /*[world][64]*/) {
  if (!sim || !sim->gather_buf) return sim ? sim->fail("dts_gather_alloc first") : 1;
  DTS_CUDA(cudaSetDevice(sim->cfg.device));
  for (int p = 0; p < sim->gather_world; p++) {
    if (p == sim->gather_rank) continue;
    cudaIpcMemHandle_t h;
    memcpy(&h, handles + 64 * p, 64);
    cudaError_t e = cudaIpcOpenMemHandle(&sim->gather_peer[p], h, cudaIpcMemLazyEnablePeerAccess);
    if (e != cudaSuccess) return sim->fail("cudaIpcOpenMemHandle(rank %d) failed: %s", p, cudaGetErrorString(e));
  }
  return 0;
}

int dts_gather_next(dts_sim* sim) {
  if (!sim || !sim->gather_buf) return sim ? sim->fail("dts_gather_alloc first") : 1;
  for (int p = 0; p < sim->gather_world; p++)
    if (!sim->gather_peer[p]) return sim->fail("dts_gather_open first (rank %d not mapped)", p);
  sim->gather_next = true;
  return 0;
}

int dts_blend4(dts_sim* sim, const uint8_t* const frames_dev[4], const double weights[4], double* out_dev, uint64_t n, void* stream) {
  if (!sim) return 1;
  if (!frames_dev || !weights || !out_dev) return sim->fail("NULL argument");
  for (int k = 0; k < 4; k++) if (!frames_dev[k]) return sim->fail("frame %d is NULL", k);
  DTS_CUDA(cudaSetDevice(sim->cfg.device));
  launch_blend4(frames_dev, weights, out_dev, (size_t)n, (cudaStream_t)stream);
  sim->launches++;
  DTS_CUDA(cudaGetLastError());
  return 0;
}

int dts_set_timing(dts_sim* sim, double delta_time, int frame_skip, int action_mode) {
  if (!sim) return 1;
  if (!(delta_time > 0) || frame_skip < 1) return sim->fail("bad delta_time / frame_skip");
  if (action_mode != DTS_ACTION_PWM && action_mode != DTS_ACTION_VEL_STEER) return sim->fail("bad action_mode");
  int d = 0;
  while (d * delta_time < sim->cfg.dyn_delay - 1e-12) d++;
  if (d > DTS_MAX_DELAY) return sim->fail("dyn_delay / delta_time exceeds DTS_MAX_DELAY steps");
  sim->step_cfg.dt = delta_time; sim->step_cfg.frame_skip = frame_skip; sim->step_cfg.action_mode = action_mode;
  sim->step_cfg.dyn.delay_steps = d;
  sim->cfg.frame_skip = frame_skip; sim->cfg.action_mode = action_mode; sim->cfg.frame_rate = 1.0 / delta_time;
  return 0;
}

int dts_set_render_mode(dts_sim* sim, int mode) {
  if (!sim) return 1;
  if (mode & ~(DTS_RENDER_SEGMENT | DTS_RENDER_TOP_DOWN)) return sim->fail("bad render mode %d", mode);
  sim->render_mode = mode;
  return 0;
}

int dts_resize_frames(dts_sim* sim, const uint8_t* src_dev, void* dst_dev, void* stream) {
  if (!sim) return 1;
  if (!sim->resize_w) return sim->fail("dts_set_resize first");
  if (!src_dev || !dst_dev) return sim->fail("NULL frame pointer");
  DTS_CUDA(cudaSetDevice(sim->cfg.device));
  launch_resize(src_dev, sim->cfg.cam_width, sim->cfg.cam_height, sim->resize_w, sim->resize_h, sim->cfg.num_envs,
                sim->resize_xtab, sim->resize_ytab, dst_dev, sim->fmt.obs_layout, sim->fmt.obs_dtype, sim->resize_band, sim->resize_cap,
                (cudaStream_t)stream);
  sim->launches++;
  DTS_CUDA(cudaGetLastError());
  return 0;
}

int dts_status(dts_sim* sim) { return (sim && sim->h_status) ? *(volatile int32_t*)sim->h_status : 0; }

int dts_profile_enable(dts_sim* sim, int on) {
  if (!sim) return 1;
  sim->profiling = on < 0 ? 0 : (on > 2 ? 2 : on);
  return 0;
}

int dts_profile_read(dts_sim* sim, double ms_out[8], int64_t* frames) {
  if (!sim || !ms_out) return 1;
  DTS_CUDA(cudaSetDevice(sim->cfg.device));
  for (int k = 0; k < 8; k++) ms_out[k] = 0.0;
  const size_t per = kProfMarks;
  DTS_CUDA(cudaDeviceSynchronize());
  for (size_t f = 0; f + per <= sim->prof_events.size(); f += per) {
    for (size_t k = 0; k + 1 < per; k++) {
      float ms = 0.f;   // an interval whose events were not recorded (level 1 marks only k_raster) reports an error: skipped
      if (cudaEventElapsedTime(&ms, sim->prof_events[f + k], sim->prof_events[f + k + 1]) == cudaSuccess) ms_out[k] += ms;
    }
  }
  cudaGetLastError();
  if (frames) *frames = sim->prof_frames;
  for (cudaEvent_t e : sim->prof_events) cudaEventDestroy(e);
  sim->prof_events.clear();
  sim->prof_frames = 0;
  return 0;
}

int dts_set_output_format(dts_sim* sim, const dts_output_format* f) {
  if (!sim) return 1;
  if (!f) return sim->fail("format is NULL");
  if (f->obs_layout < DTS_OBS_HWC || f->obs_layout > DTS_OBS_CWH) return sim->fail("bad obs_layout %d", f->obs_layout);
  if (f->obs_dtype != DTS_OBS_U8 && f->obs_dtype != DTS_OBS_F32_UNIT) return sim->fail("bad obs_dtype %d", f->obs_dtype);
  if (f->reward_mode != DTS_REWARD_RAW && f->reward_mode != DTS_REWARD_DT) return sim->fail("bad reward_mode %d", f->reward_mode);
  if (f->action_map != DTS_ACTIONS_CONTINUOUS && f->action_map != DTS_ACTIONS_DISCRETE3) return sim->fail("bad action_map %d", f->action_map);
  if (f->action_map == DTS_ACTIONS_DISCRETE3 && sim->cfg.action_mode != DTS_ACTION_VEL_STEER)
    return sim->fail("discrete actions are [vel, steering] pairs (DiscreteWrapper wraps DuckietownEnv): action_mode must be VEL_STEER");
  sim->fmt = *f;
  sim->step_cfg.reward_mode = f->reward_mode; sim->step_cfg.action_map = f->action_map;
  sim->step_cfg.action_vel_scale = f->action_vel_scale;
  return 0;
}

int dts_get_dyn_state(dts_sim* sim, int map_id, double** state_dev, int32_t* n_dyn) {
  if (!sim) return 1;
  if (map_id < 0 || map_id >= sim->cfg.max_maps || !sim->h_maps[map_id].valid) return sim->fail("bad map_id %d", map_id);
  if (state_dev) *state_dev = sim->h_maps[map_id].n_dyn ? sim->h_maps[map_id].dyn_state : nullptr;
  if (n_dyn) *n_dyn = sim->h_maps[map_id].n_dyn;
  return 0;
}

uint64_t dts_launch_count(dts_sim* sim) { return sim ? sim->launches : 0; }

int dts_debug_episode(dts_sim* sim, int env, void* out144) {
  if (!sim) return 1;
  if (env < 0 || env >= sim->cfg.num_envs) return sim->fail("env out of range");
  DTS_CUDA(cudaSetDevice(sim->cfg.device));
  DTS_CUDA(cudaMemcpy(out144, sim->S.rep + env, sizeof(RenderEp), cudaMemcpyDeviceToHost));
  return 0;
}

/* debug: frame setup of `env` in the last dts_render (synchronises) */
int dts_debug_frame(dts_sim* sim, int env, double V[12], float P[4], int32_t counts[4], float* lattice_by_cell, int n_cells) {
  if (!sim) return 1;
  if (env < 0 || env >= sim->cfg.num_envs) return sim->fail("env out of range");
  if (!sim->render_scratch) return sim->fail("nothing rendered yet");
  if (sim->cfg.flags & DTS_FLAG_TESSELLATE) return sim->fail("dts_debug_frame reads the analytic-tile lattice (tile mode 1)");
  DTS_CUDA(cudaSetDevice(sim->cfg.device));
  DTS_CUDA(cudaDeviceSynchronize());
  const int cbins = ((sim->cfg.cam_width + 31) / 32) * ((sim->cfg.cam_height + 7) / 8);
  const size_t frame = (size_t)sim->items_max;
  if (debug_frame_copy(sim->render_scratch, sim->cfg.num_envs, sim->max_prims, cbins, sim->bin_cap, sim->max_lat, frame, env, V, P,
                       counts, lattice_by_cell, n_cells, 2))
    return sim->fail("debug_frame_copy failed");
  return 0;
}

/* debug: copy the 32 int32 diagnostic counters (word 0 = overflow flag; 8.. = DTS_STATS counters) */
int dts_debug_counters(dts_sim* sim, int32_t out[32]) {
  if (!sim) return 1;
  DTS_CUDA(cudaSetDevice(sim->cfg.device));
  DTS_CUDA(cudaMemcpy(out, sim->d_err, 32 * sizeof(int32_t), cudaMemcpyDeviceToHost));
  return 0;
}

// ---- multi-GPU: one NCCL all-gather of the end-of-rollout observation batch (SURVEY 8e) ----------
// libnccl is dlopen'ed (the torch-bundled copy); the communicator is created from a unique id that
// the Python side broadcasts with torch.distributed.

int dts_comm_load(dts_sim* sim, const char* libnccl_path) {
  if (!sim) return 1;
  if (sim->nccl_lib) return 0;
  sim->nccl_lib = dlopen(libnccl_path, RTLD_NOW | RTLD_GLOBAL);
  if (!sim->nccl_lib) return sim->fail("dlopen(%s) failed: %s", libnccl_path, dlerror());
  return 0;
}

int dts_comm_unique_id(dts_sim* sim, uint8_t out[128]) {
  if (!sim || !sim->nccl_lib) return sim ? sim->fail("dts_comm_load first") : 1;
  auto f = (int (*)(void*))dlsym(sim->nccl_lib, "ncclGetUniqueId");
  if (!f) return sim->fail("ncclGetUniqueId not found");
  const int r = f(out);
  return r ? sim->fail("ncclGetUniqueId -> %d", r) : 0;
}

struct nccl_uid { char b[128]; };

int dts_comm_init(dts_sim* sim, const uint8_t id[128], int rank, int world) {
  if (!sim || !sim->nccl_lib) return sim ? sim->fail("dts_comm_load first") : 1;
  DTS_CUDA(cudaSetDevice(sim->cfg.device));
  auto f = (int (*)(void**, int, nccl_uid, int))dlsym(sim->nccl_lib, "ncclCommInitRank");
  if (!f) return sim->fail("ncclCommInitRank not found");
  nccl_uid u;
  memcpy(u.b, id, 128);
  const int r = f(&sim->nccl_comm, world, u, rank);
  return r ? sim->fail("ncclCommInitRank -> %d", r) : 0;
}

int dts_allgather_obs(dts_sim* sim, const void* send_dev, void* recv_dev, uint64_t bytes_per_rank, void* stream) {
  if (!sim || !sim->nccl_comm) return sim ? sim->fail("dts_comm_init first") : 1;
  DTS_CUDA(cudaSetDevice(sim->cfg.device));
  auto f = (int (*)(const void*, void*, size_t, int, void*, cudaStream_t))dlsym(sim->nccl_lib, "ncclAllGather");
  if (!f) return sim->fail("ncclAllGather not found");
  const int r = f(send_dev, recv_dev, (size_t)bytes_per_rank, /*ncclUint8*/ 1, sim->nccl_comm, (cudaStream_t)stream);
  return r ? sim->fail("ncclAllGather -> %d", r) : 0;
}

}  // extern "C"
