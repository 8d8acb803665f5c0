// Host-side internals shared by the API translation units of libgpb200 (not part of the C ABI).
#pragma once
#include "../../include/gpb200.h"

#include <algorithm>
#include <cmath>
#include <cstdlib>
#include <new>

#include "common.cuh"
#include "gram.cuh"

struct gpb200_handle_s : public gpb::Handle {};

namespace gpb {

// ---- workspace arena ----------------------------------------------------------------------------
struct Arena {
  char *base = nullptr;
  size_t cap = 0, off = 0;
  template <typename T>
  T *take(size_t count) {
    size_t bytes = (count * sizeof(T) + 255) & ~(size_t)255;
    if (off + bytes > cap) return nullptr;
    T *p = reinterpret_cast<T *>(base + off);
    off += bytes;
    return p;
  }
};

inline size_t pad256(size_t b) { return (b + 255) & ~(size_t)255; }
constexpr int MAX_DENSE_N = 65535 - TILE;  // pack / unpack put the column index in gridDim.y (<= 65535)

int ws_reserve(Handle *h, size_t bytes, Arena *a);

// ---- tile task lists (host-built once per tile count, cached on the device) ---------------------
enum TaskKind { TK_CHOL = 1, TK_CHOL_TRAIL, TK_CHOL_LA1, TK_CHOL_LA2, TK_TRTRI_S, TK_TRTRI_W, TK_LAUUM, TK_TAN_T1, TK_TAN_A, TK_TAN_LDOT, TK_COND_V,
                TK_COND_COV, TK_MUL_WB, TK_MUL_WTB, TK_MUL_LZ, TK_SINV_Y, TK_SINV_D, TK_SINV_Z, TK_SINV_ZD };

struct TaskList {
  const TileTask *dev = nullptr;
  const std::vector<int> *offsets = nullptr;
  int count(int step) const { return (*offsets)[step + 1] - (*offsets)[step]; }
  const TileTask *at(int step) const { return dev + (*offsets)[step]; }
  int steps() const { return (int)offsets->size() - 1; }
};

int upload_tasks(Handle *h, long long key, const std::vector<TileTask> &tasks, const std::vector<int> &offsets,
                 TaskList *out);
bool cached(Handle *h, long long key, TaskList *out);
inline long long tkey(int kind, int a, int b = 0) { return ((long long)kind << 48) | ((long long)a << 24) | (long long)b; }
void sort_desc(std::vector<TileTask> &v, size_t from);
int tasks_chol(Handle *h, int nt, int pt, TaskList *upd, TaskList *trail);
int tasks_trtri(Handle *h, int nt, TaskList *s_out, TaskList *w_out);
int tasks_lauum(Handle *h, int nt, TaskList *out);

// ---- engines on padded device buffers ---------------------------------------------------------
inline MatRef mref(double *p, long long ld, long long stride) { return MatRef{p, ld, stride}; }
int chol_panel_tiles(int nt, int batch);
bool chol_uses_lookahead(const Handle *h, int nt, int batch);
int chol_lookahead_panel(const Handle *h, int nt);
int chol_batched(Handle *h, double *Lbuf, int np, long long stride, int n, int batch, int *info_dev, const int *env = nullptr);
int sinv_batched(Handle *h, double *Lbuf, double *Sbuf, int np, long long stride, const int *env, int batch);
int trtri_batched(Handle *h, double *Lbuf, double *Sbuf, int np, long long stride, int batch);
int extract_diag(Handle *h, int np, const double *L, long long stride, double *dvec, int batch);

// ---- host <-> device staging (direction follows the handle's pointer mode) --------------------
int to_device(Handle *h, const double *src, double *dev, size_t count);
int from_device(Handle *h, const void *dev, void *dst, size_t bytes);
int to_device_2d(Handle *h, const double *src, long long lds, double *dev, long long ldd, int rows, int cols);
int from_device_2d(Handle *h, const double *dev, long long lds, double *dst, long long ldd, int rows, int cols);
int finish(Handle *h);
int read_info(Handle *h, const int *info_dev, int *out);

}  // namespace gpb

// Every entry point runs on the handle's device and gives the caller its own current device back on every return
// path (a process may hold torch tensors or other handles on another GPU).
struct DeviceGuard {
  int prev = -1;
  bool ok = true;
  explicit DeviceGuard(int dev) {
    if (cudaGetDevice(&prev) != cudaSuccess) prev = -1;
    if (prev != dev) ok = cudaSetDevice(dev) == cudaSuccess;
  }
  ~DeviceGuard() {
    int cur = -1;
    if (prev >= 0 && cudaGetDevice(&cur) == cudaSuccess && cur != prev) cudaSetDevice(prev);
  }
};
#define CHECK_H(h)                                   \
  if (!(h)) return -1;                               \
  (h)->err[0] = 0;                                   \
  DeviceGuard device_guard__((h)->device);      \
  if (!device_guard__.ok) return -1000
#define BAD_ARG(h, k, msg)                                  \
  do {                                                      \
    snprintf((h)->err, sizeof((h)->err), "%s", msg);       \
    return -(k);                                            \
  } while (0)
#define RC(x)               \
  do {                      \
    int rc__ = (x);         \
    if (rc__) return rc__;  \
  } while (0)
