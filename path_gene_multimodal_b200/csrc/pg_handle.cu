// Handle, error text and grow-only workspace of libpathgraph.so.
#include <cstdarg>
#include <cstdlib>
#include <new>
#include "pg_common.cuh"

static std::string g_create_error;

int pg_pdl_mask() {
  static int mask = [] {
    const char* e = getenv("PG_PDL_MASK");
    return e ? (int)strtol(e, nullptr, 0) : 0x7fffffff;
  }();
  return mask;
}

int pg_set_error(pg_handle* h, int code, const char* fmt, ...) {
  char buf[1024];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof(buf), fmt, ap);
  va_end(ap);
  if (h)
    h->err = buf;
  else
    g_create_error = buf;
  return code;
}

int pg_reserve(pg_handle* h, pg_buf& b, size_t bytes) {
  if (bytes <= b.cap) return PG_OK;
  // grow-only with 25 % slack so a stream of slightly different slides settles quickly
  size_t want = bytes + bytes / 4 + 256;
  if (b.p) {
    PG_CUDA(h, cudaDeviceSynchronize());
    PG_CUDA(h, cudaFree(b.p));
    b.p = nullptr;
    b.cap = 0;
  }
  cudaError_t e = cudaMalloc(&b.p, want);
  if (e != cudaSuccess) {
    cudaGetLastError();
    b.p = nullptr;
    return pg_set_error(h, PG_ERR_NOMEM, "workspace cudaMalloc(%zu) failed: %s", want,
                        cudaGetErrorString(e));
  }
  b.cap = want;
  return PG_OK;
}

int pg_check_input_flag(pg_handle* h) {
  if (h->build_epoch != 0 && h->pinned[8] == h->build_epoch)
    return pg_set_error(h, PG_ERR_INVALID, "coordinates must be finite (the last pg_grid_build met NaN or inf)");
  return PG_OK;
}

static void pg_profile_clear(pg_handle* h) {
  for (auto& r : h->prof) { cudaEventDestroy(r.e0); cudaEventDestroy(r.e1); }
  h->prof.clear();
}

extern "C" {

int pg_version(void) { return 100; }

int pg_create(int device, pg_handle** out) {
  if (!out) return pg_set_error(nullptr, PG_ERR_INVALID, "pg_create: out is NULL");
  *out = nullptr;
  int count = 0;
  cudaError_t e = cudaGetDeviceCount(&count);
  if (e != cudaSuccess || count == 0) {
    cudaGetLastError();
    return pg_set_error(nullptr, PG_ERR_CUDA,
                        "pg_create: no CUDA device (%s); libpathgraph has no CPU fallback",
                        e != cudaSuccess ? cudaGetErrorString(e) : "device count is 0");
  }
  if (device < 0 || device >= count)
    return pg_set_error(nullptr, PG_ERR_INVALID, "pg_create: device %d out of range [0,%d)", device, count);
  e = cudaSetDevice(device);
  if (e != cudaSuccess)
    return pg_set_error(nullptr, PG_ERR_CUDA, "cudaSetDevice(%d): %s", device, cudaGetErrorString(e));
  cudaDeviceProp prop;
  e = cudaGetDeviceProperties(&prop, device);
  if (e != cudaSuccess)
    return pg_set_error(nullptr, PG_ERR_CUDA, "cudaGetDeviceProperties: %s", cudaGetErrorString(e));
  if (prop.major != 10)
    return pg_set_error(nullptr, PG_ERR_CUDA,
                        "pg_create: device %d is sm_%d%d; libpathgraph is built for sm_100a only", device,
                        prop.major, prop.minor);
  pg_handle* h = new (std::nothrow) pg_handle();
  if (!h) return pg_set_error(nullptr, PG_ERR_NOMEM, "pg_create: out of host memory");
  h->device = device;
  h->sm_count = prop.multiProcessorCount;
  e = cudaHostAlloc((void**)&h->pinned, 64 * sizeof(int32_t), cudaHostAllocDefault);
  if (e != cudaSuccess) {
    delete h;
    return pg_set_error(nullptr, PG_ERR_NOMEM, "cudaHostAlloc: %s", cudaGetErrorString(e));
  }
  for (int i = 0; i < 64; ++i) h->pinned[i] = 0;
  int rc = pg_reserve(h, h->misc, PG_MISC_BYTES);
  if (rc == PG_OK) {
    e = cudaMemset(h->misc.p, 0, PG_MISC_BYTES);
    if (e != cudaSuccess) rc = pg_set_error(nullptr, PG_ERR_CUDA, "cudaMemset: %s", cudaGetErrorString(e));
  } else {
    g_create_error = h->err;
  }
  if (rc != PG_OK) {
    cudaFreeHost(h->pinned);
    delete h;
    return rc;
  }
  *out = h;
  return PG_OK;
}

int pg_destroy(pg_handle* h) {
  if (!h) return PG_OK;
  cudaSetDevice(h->device);
  cudaDeviceSynchronize();
  pg_buf* bufs[] = {&h->cell_count, &h->cell_start, &h->cell_of, &h->rank,      &h->s_rec,     &h->s_pos,     &h->s_gid,     &h->knn_retry,     &h->pt_meta,   &h->tmp_ent,   &h->row_off,
                    &h->row_count,  &h->scan_state, &h->misc,    &h->sym_extra, &h->sym_cursor, &h->sym_recip, &h->hull,
                    &h->enrich_lab, &h->enrich_cnt, &h->ac_z,    &h->ac_idx,    &h->ac_deg,     &h->ac_sims,    &h->ac_part,
                    &h->ac_misc,    &h->lk_cnt,     &h->lk_off,  &h->lk_ord,
                    &h->cl_parent,  &h->cl_count,   &h->cl_scan, &h->cl_order,  &h->cl_off};
  for (pg_buf* b : bufs)
    if (b->p) cudaFree(b->p);
  if (h->pinned) cudaFreeHost(h->pinned);
  pg_profile_clear(h);
  delete h;
  return PG_OK;
}

const char* pg_last_error(pg_handle* h) { return h ? h->err.c_str() : g_create_error.c_str(); }

int64_t pg_workspace_bytes(pg_handle* h) {
  if (!h) return 0;
  pg_buf* bufs[] = {&h->cell_count, &h->cell_start, &h->cell_of, &h->rank,      &h->s_rec,     &h->s_pos,     &h->s_gid,     &h->knn_retry,     &h->pt_meta,   &h->tmp_ent,   &h->row_off,
                    &h->row_count,  &h->scan_state, &h->misc,    &h->sym_extra, &h->sym_cursor, &h->sym_recip, &h->hull,
                    &h->enrich_lab, &h->enrich_cnt, &h->ac_z,    &h->ac_idx,    &h->ac_deg,     &h->ac_sims,    &h->ac_part,
                    &h->ac_misc,    &h->lk_cnt,     &h->lk_off,  &h->lk_ord,
                    &h->cl_parent,  &h->cl_count,   &h->cl_scan, &h->cl_order,  &h->cl_off};
  int64_t t = 0;
  for (pg_buf* b : bufs) t += (int64_t)b->cap;
  return t;
}

int64_t pg_launch_count(pg_handle* h) { return h ? h->launches : 0; }

int pg_profile_enable(pg_handle* h, int on) {
  if (!h) return PG_ERR_INVALID;
  PG_CUDA(h, cudaSetDevice(h->device));
  PG_CUDA(h, cudaDeviceSynchronize());
  pg_profile_clear(h);
  h->profiling = on != 0;
  return PG_OK;
}

int pg_profile_count(pg_handle* h) {
  if (!h) return PG_ERR_INVALID;
  PG_CUDA(h, cudaSetDevice(h->device));
  PG_CUDA(h, cudaDeviceSynchronize());
  return (int)h->prof.size();
}

int pg_profile_get(pg_handle* h, int i, const char** name, float* ms) {
  if (!h || i < 0 || i >= (int)h->prof.size()) return PG_ERR_INVALID;
  if (name) *name = h->prof[i].name;
  if (ms) PG_CUDA(h, cudaEventElapsedTime(ms, h->prof[i].e0, h->prof[i].e1));
  return PG_OK;
}

int pg_check_overflow(pg_handle* h) {
  if (!h) return PG_ERR_INVALID;
  PG_CUDA(h, cudaSetDevice(h->device));
  int32_t* flag = (int32_t*)((char*)h->misc.p + PG_MISC_OVERFLOW);
  PG_CUDA(h, cudaMemcpyAsync(&h->pinned[3], flag, sizeof(int32_t), cudaMemcpyDeviceToHost, h->last_stream));
  PG_CUDA(h, cudaMemcpyAsync(&h->pinned[8], (char*)h->misc.p + PG_MISC_BADINPUT, sizeof(int32_t), cudaMemcpyDeviceToHost, h->last_stream));
  PG_CUDA(h, cudaMemsetAsync(flag, 0, sizeof(int32_t), h->last_stream));
  PG_CUDA(h, cudaStreamSynchronize(h->last_stream));
  int rc_in = pg_check_input_flag(h);
  if (rc_in) return rc_in;
  if (h->pinned[3] != 0)
    return pg_set_error(h, PG_ERR_CAPACITY, "an output buffer was smaller than the result (capacity overflow)");
  return PG_OK;
}

}  // extern "C"
