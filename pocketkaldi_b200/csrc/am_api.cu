// C-ABI entry points of the acoustic model, the device-resident batch pipeline and
// the model-file readers (AcousticModel::Read, src/am.cc:23-63; Nnet::Read /
// ReadLayer, src/nnet.cc:80-147; Matrix::Read, src/matrix.cc:287-319; Vector::Read,
// src/vector.cc:392-425; Configuration::Read, src/configuration.cc:14-71).

#include <ctype.h>
#include <math.h>
#include <string.h>

#include <algorithm>
#include <map>
#include <memory>
#include <string>

#include "decoder.cuh"
#include "nnet.cuh"

using pkb::BatchMeta;
using pkb::Ctx;
using pkb::InputView;
using pkb::Workspace;

// ---------------------------------------------------------------- file readers
namespace {

struct File {
  FILE *f = nullptr;
  std::string name;
  ~File() { if (f) fclose(f); }
  int open(const std::string &path) {
    name = path;
    f = fopen(path.c_str(), "rb");
    if (!f) {
      pkb::set_error("IOError: unable to open %s", path.c_str());
      return PKB_ERR_IO;
    }
    return PKB_OK;
  }
  int read(void *dst, size_t n) {
    if (fread(dst, 1, n, f) != n) {
      pkb::set_error("IOError: failed to read %zu bytes from %s", n, name.c_str());
      return PKB_ERR_IO;
    }
    return PKB_OK;
  }
  int expect(const char *tag) {
    char buf[8] = {0};
    PKB_TRY(read(buf, 4));
    if (memcmp(buf, tag, 4) != 0) {
      pkb::set_error("Corruption: section '%s' expected in %s", tag, name.c_str());
      return PKB_ERR_CORRUPT;
    }
    return PKB_OK;
  }
  int read_i32(int32_t *v) { return read(v, 4); }
};

template <typename T>
int read_vec(File *fd, std::vector<T> *out) {
  static_assert(sizeof(T) == 4, "VEC0 payload is 4 bytes per element");
  int32_t size = 0, dim = 0;
  PKB_TRY(fd->expect("VEC0"));
  PKB_TRY(fd->read_i32(&size));
  PKB_TRY(fd->read_i32(&dim));
  if (dim < 0 || size != 4 * dim + 4) {
    pkb::set_error("Corruption: VEC0 section_size = %d * 4 + 4 expected, but %d found: %s", dim, size,
                   fd->name.c_str());
    return PKB_ERR_CORRUPT;
  }
  out->resize(dim);
  if (dim) PKB_TRY(fd->read(out->data(), sizeof(T) * dim));
  return PKB_OK;
}

int read_mat(File *fd, std::vector<float> *out, int *rows, int *cols) {
  int32_t size = 0, r = 0, c = 0;
  PKB_TRY(fd->expect("MAT0"));
  PKB_TRY(fd->read_i32(&size));
  if (size != 8) {
    pkb::set_error("Corruption: MAT0 section_size == 8 expected, but %d found (%s)", size,
                   fd->name.c_str());
    return PKB_ERR_CORRUPT;
  }
  PKB_TRY(fd->read_i32(&r));
  PKB_TRY(fd->read_i32(&c));
  if (r < 0 || c < 0) {
    pkb::set_error("Corruption: MAT0 negative shape in %s", fd->name.c_str());
    return PKB_ERR_CORRUPT;
  }
  out->resize(static_cast<size_t>(r) * c);
  std::vector<float> row;
  for (int i = 0; i < r; ++i) {
    PKB_TRY(read_vec(fd, &row));
    if (static_cast<int>(row.size()) != c) {
      pkb::set_error("Corruption: MAT0 row %d has %zu columns, %d expected (%s)", i, row.size(), c,
                     fd->name.c_str());
      return PKB_ERR_CORRUPT;
    }
    memcpy(out->data() + static_cast<size_t>(i) * c, row.data(), sizeof(float) * c);
  }
  *rows = r;
  *cols = c;
  return PKB_OK;
}

struct HostNnet {
  std::vector<int32_t> types;
  std::vector<std::vector<float>> W, b;
  std::vector<int32_t> out_dims, in_dims;
};

int read_nnet(const std::string &path, HostNnet *net) {
  File fd;
  PKB_TRY(fd.open(path));
  int32_t size = 0, n = 0;
  PKB_TRY(fd.expect("NNT0"));
  PKB_TRY(fd.read_i32(&size));
  PKB_TRY(fd.read_i32(&n));
  std::vector<float> pending_scale;  // MUL layer waiting for the next linear layer
  for (int i = 0; i < n; ++i) {
    int32_t lsize = 0, type = 0;
    PKB_TRY(fd.expect("LAY0"));
    PKB_TRY(fd.read_i32(&lsize));
    PKB_TRY(fd.read_i32(&type));
    if (lsize != 4) {
      pkb::set_error("Corruption: read_layer: section_size == 4 expected, but %d found (%s)", lsize,
                     path.c_str());
      return PKB_ERR_CORRUPT;
    }
    if (type == 0) {
      std::vector<float> W, b;
      int r = 0, c = 0;
      PKB_TRY(read_mat(&fd, &W, &r, &c));
      PKB_TRY(read_vec(&fd, &b));
      if (static_cast<int>(b.size()) != r) {
        pkb::set_error("Corruption: linear layer: W has %d rows but b has %zu (%s)", r, b.size(),
                       path.c_str());
        return PKB_ERR_CORRUPT;
      }
      if (!pending_scale.empty()) {
        // y = W (x * v) + b  ==  (W diag(v)) x + b
        if (static_cast<int>(pending_scale.size()) != c) {
          pkb::set_error("Corruption: MUL layer of dim %zu in front of a linear layer with %d inputs (%s)",
                         pending_scale.size(), c, path.c_str());
          return PKB_ERR_CORRUPT;
        }
        for (int i2 = 0; i2 < r; ++i2)
          for (int j = 0; j < c; ++j) W[static_cast<size_t>(i2) * c + j] *= pending_scale[j];
        pending_scale.clear();
      }
      net->W.push_back(std::move(W));
      net->b.push_back(std::move(b));
      net->out_dims.push_back(r);
      net->in_dims.push_back(c);
    } else if (type == 5) {
      // MUL layer (tool/convert_am.py:86-110,213-217 writes one for Kaldi's FixedScaleComponent):
      // y = x * v element-wise. The reference reader rejects it (src/nnet.cc:122-126), so real
      // nnet2 models with a FixedScaleComponent cannot be loaded there; here it is folded into the
      // neighbouring LinearLayer at load time (SURVEY 8(f)-3) and costs nothing at run time.
      std::vector<float> v;
      PKB_TRY(read_vec(&fd, &v));
      if (!net->types.empty() && net->types.back() == 0) {
        // directly after a linear layer: y = v * (W x + b) == (diag(v) W) x + v * b
        std::vector<float> &W = net->W.back(), &b = net->b.back();
        const int r = net->out_dims.back(), c = net->in_dims.back();
        if (static_cast<int>(v.size()) != r) {
          pkb::set_error("Corruption: MUL layer of dim %zu after a linear layer with %d outputs (%s)",
                         v.size(), r, path.c_str());
          return PKB_ERR_CORRUPT;
        }
        for (int i2 = 0; i2 < r; ++i2) {
          for (int j = 0; j < c; ++j) W[static_cast<size_t>(i2) * c + j] *= v[i2];
          b[i2] *= v[i2];
        }
      } else if (pending_scale.empty()) {
        pending_scale = std::move(v);  // folded into the next linear layer
      } else {
        if (pending_scale.size() != v.size()) {
          pkb::set_error("Corruption: consecutive MUL layers of dims %zu and %zu (%s)",
                         pending_scale.size(), v.size(), path.c_str());
          return PKB_ERR_CORRUPT;
        }
        for (size_t j = 0; j < v.size(); ++j) pending_scale[j] *= v[j];
      }
      continue;  // not a layer of the executed stack
    } else if ((type < 0 || type > 3) && type != PKB_LAYER_SIGMOID) {
      // ADD (4) is defined by the converter but never written by it; rejected like the
      // reference reader does (src/nnet.cc:122-126)
      pkb::set_error("Corruption: read_layer: unexpected layer type: %d (%s)", type, path.c_str());
      return PKB_ERR_CORRUPT;
    }
    if (type != 0 && !pending_scale.empty()) break;  // relu(x * v) / normalize(x * v) do not fold
    net->types.push_back(type);
  }
  if (!pending_scale.empty()) {
    pkb::set_error("MUL layer that is not adjacent to a linear layer cannot be folded (%s)", path.c_str());
    return PKB_ERR_UNSUPPORTED;
  }
  return PKB_OK;
}

std::string trim(const std::string &s) {
  size_t a = 0, b = s.size();
  while (a < b && isspace(static_cast<unsigned char>(s[a]))) ++a;
  while (b > a && isspace(static_cast<unsigned char>(s[b - 1]))) --b;
  return s.substr(a, b - a);
}

int read_conf(const std::string &path, std::map<std::string, std::string> *table) {
  FILE *f = fopen(path.c_str(), "r");
  if (!f) {
    pkb::set_error("IOError: unable to open %s", path.c_str());
    return PKB_ERR_IO;
  }
  char line[4096];
  int rc = PKB_OK;
  while (fgets(line, sizeof(line), f)) {
    std::string s = trim(line);
    if (s.empty() || s[0] == '#') continue;
    size_t eq = s.find('=');
    if (eq == std::string::npos || s.find('=', eq + 1) != std::string::npos) {
      pkb::set_error("Corruption: Unexpected line in %s: %s", path.c_str(), s.c_str());
      rc = PKB_ERR_CORRUPT;
      break;
    }
    std::string key = trim(s.substr(0, eq)), val = trim(s.substr(eq + 1));
    for (auto &ch : key) ch = static_cast<char>(tolower(static_cast<unsigned char>(ch)));
    if (val.empty()) {
      pkb::set_error("Corruption: Value cound not be empty: %s", path.c_str());
      rc = PKB_ERR_CORRUPT;
      break;
    }
    (*table)[key] = val;
  }
  fclose(f);
  return rc;
}

int conf_get(const std::map<std::string, std::string> &t, const std::string &conf,
             const char *key, std::string *val) {
  auto it = t.find(key);
  if (it == t.end()) {
    pkb::set_error("Corruption: Unable to find key '%s' in '%s'", key, conf.c_str());
    return PKB_ERR_CORRUPT;
  }
  *val = it->second;
  return PKB_OK;
}

std::string conf_path(const std::string &conf, const std::string &v) {
  if (!v.empty() && v[0] == '/') return v;
  size_t pos = conf.rfind('/');
  if (pos == std::string::npos) return v;
  return conf.substr(0, pos + 1) + v;
}

int conf_int(const std::map<std::string, std::string> &t, const std::string &conf, const char *key,
             int *out) {
  std::string v;
  PKB_TRY(conf_get(t, conf, key, &v));
  char *end = nullptr;
  long x = strtol(v.c_str(), &end, 10);
  if (end == v.c_str()) {
    pkb::set_error("Corruption: key '%s' in '%s' is not an integer: %s", key, conf.c_str(), v.c_str());
    return PKB_ERR_CORRUPT;
  }
  *out = static_cast<int>(x);
  return PKB_OK;
}

}  // namespace

// ---------------------------------------------------------------- batch object
struct pkb_batch {
  Ctx *c = nullptr;
  pkb_am *am = nullptr;
  BatchMeta meta;
  float prob_scale = 1.0f;
  float global_stats[PKB_CMVN_STATS_DIM];
  pkb::DevBuf pcm, raw, feats, loglik, sum;
  bool compact = false;             // nnet stage writes loglik16 + loglik_off instead of loglik
  pkb::DevBuf loglik16, loglik_off;
  pkb::DevBuf vit_work, vit_out, vit_tid2pdf;  // GPU Viterbi: workspace, results, device tid2pdf
  pkb::DevBuf lat_log, lat_aux, lat_arcs;      // lattices: arc logs, offsets and results, kept arcs
  int64_t lat_total = -1;                      // kept arcs of the latest pkb_batch_lattice
  const pkb_fst *lat_fst = nullptr;            // its graph, while its records are valid
  pkb::LatticeRecords lat_rec;                 // its records on the device
  pkb::DevBuf nbest_work;                      // outputs of pkb_batch_nbest
  Workspace ws;
  pkb::Refine rf;
  pkb::PaddedPlanes planes;
  int64_t padded = 0, gemm_rows = 0;
  std::vector<int64_t> pad_off;  // host copy: first padded row of every utterance
};

extern "C" {

// ---------------------------------------------------------------- AM
int pkb_am_create(pkb_ctx_t *c, int n_layers, const int32_t *layer_types,
                  const float *const *weights, const float *const *biases, const int32_t *out_dims,
                  const int32_t *in_dims, const float *prior, int num_pdfs, int left_context,
                  int right_context, const int32_t *tid2pdf, int n_tid2pdf, int precision,
                  pkb_am_t **am) {
  return pkb::am_build(c, n_layers, layer_types, weights, biases, out_dims, in_dims, prior, num_pdfs,
                       left_context, right_context, tid2pdf, n_tid2pdf, precision, am);
}

int pkb_am_load(pkb_ctx_t *c, const char *conf_file, int precision, pkb_am_t **am) {
  PKB_REQUIRE(c && conf_file && am, "pkb_am_load: NULL argument");
  const std::string conf = conf_file;
  std::map<std::string, std::string> t;
  PKB_TRY(read_conf(conf, &t));
  std::string v;
  HostNnet net;
  PKB_TRY(conf_get(t, conf, "nnet", &v));
  PKB_TRY(read_nnet(conf_path(conf, v), &net));
  std::vector<float> prior;
  {
    PKB_TRY(conf_get(t, conf, "prior", &v));
    File fd;
    PKB_TRY(fd.open(conf_path(conf, v)));
    PKB_TRY(read_vec(&fd, &prior));
  }
  int left = 0, right = 0, num_pdfs = 0;
  PKB_TRY(conf_int(t, conf, "left_context", &left));
  PKB_TRY(conf_int(t, conf, "right_context", &right));
  PKB_TRY(conf_int(t, conf, "num_pdfs", &num_pdfs));
  std::vector<int32_t> tid2pdf;
  {
    PKB_TRY(conf_get(t, conf, "tid2pdf", &v));
    File fd;
    PKB_TRY(fd.open(conf_path(conf, v)));
    PKB_TRY(read_vec(&fd, &tid2pdf));
  }
  if (static_cast<int>(prior.size()) != num_pdfs) {
    pkb::set_error("Corruption: prior has %zu entries but num_pdfs = %d (%s)", prior.size(), num_pdfs,
                   conf.c_str());
    return PKB_ERR_CORRUPT;
  }
  std::vector<const float *> W, b;
  for (size_t i = 0; i < net.W.size(); ++i) {
    W.push_back(net.W[i].data());
    b.push_back(net.b[i].data());
  }
  return pkb::am_build(c, static_cast<int>(net.types.size()), net.types.data(), W.data(), b.data(),
                       net.out_dims.data(), net.in_dims.data(), prior.data(), num_pdfs, left, right,
                       tid2pdf.data(), static_cast<int>(tid2pdf.size()), precision, am);
}

void pkb_am_destroy(pkb_am_t *am) {
  if (!am) return;
  if (am->c) cudaSetDevice(am->c->device);
  delete am;
}

int pkb_am_num_pdfs(const pkb_am_t *am) { return am ? am->num_pdfs : 0; }
int pkb_am_input_dim(const pkb_am_t *am) { return am ? am->input_dim : 0; }
int pkb_am_left_context(const pkb_am_t *am) { return am ? am->left : 0; }
int pkb_am_right_context(const pkb_am_t *am) { return am ? am->right : 0; }
int pkb_am_num_tids(const pkb_am_t *am) { return am ? static_cast<int>(am->tid2pdf.size()) : 0; }
int pkb_am_tid2pdf(const pkb_am_t *am, int tid) {
  if (!am || tid < 0 || tid >= static_cast<int>(am->tid2pdf.size())) return -1;
  return am->tid2pdf[tid];
}

// Shared body of pkb_am_compute / pkb_am_compute_chunked: everything up to the log-likelihoods in
// am->out_f32 (padded-row layout); pad_off receives the first padded row of every utterance.
static int am_compute_device(pkb_ctx_t *c, pkb_am_t *am, const float *feats, const int32_t *num_frames,
                             int n_utts, int feat_dim, float prob_scale, const char *who,
                             std::vector<int64_t> *pad_off) {
  PKB_REQUIRE(c && am, "%s: NULL argument", who);
  PKB_REQUIRE(am->c == c, "%s: model belongs to another context", who);
  PKB_REQUIRE(am->feat_dim > 0 && feat_dim == am->feat_dim,
              "%s: feat_dim %d does not match the model (nnet input %d, context %d+1+%d)", who,
              feat_dim, am->input_dim, am->left, am->right);
  PKB_CUDA(cudaSetDevice(c->device));
  BatchMeta &m = am->meta;
  PKB_TRY(m.build_from_frames(num_frames, n_utts));
  if (m.total_frames == 0) return PKB_OK;
  PKB_REQUIRE(feats != nullptr, "%s: feats is NULL", who);
  PKB_TRY(m.upload(c->stream));
  int64_t padded = 0, rows = 0;
  pkb::padded_rows(m, am->left, am->right, pad_off, &padded, &rows);
  Workspace &ws = am->ws;
  PKB_TRY(pkb::workspace_ensure(am, &ws, rows));
  const int dp = am->feat_dim_pad;
  PKB_TRY(ws.feat_hi.ensure(static_cast<size_t>(padded) * dp * 2));
  if (am->planes == 2) PKB_TRY(ws.feat_lo.ensure(static_cast<size_t>(padded) * dp * 2));
  PKB_TRY(ws.pad_off.ensure(pad_off->size() * sizeof(int64_t)));
  PKB_TRY(ws.row_map.ensure(static_cast<size_t>(rows) * sizeof(int32_t)));
  // pageable source: staged by the runtime before the call returns
  PKB_CUDA(cudaMemcpyAsync(ws.pad_off.p, pad_off->data(), pad_off->size() * sizeof(int64_t),
                           cudaMemcpyHostToDevice, c->stream));
  const size_t in_bytes = static_cast<size_t>(m.total_frames) * feat_dim * sizeof(float);
  const size_t out_bytes = static_cast<size_t>(rows) * am->num_pdfs * sizeof(float);  // padded rows
  PKB_TRY(am->in_f32.ensure(in_bytes));
  PKB_TRY(am->out_f32.ensure(out_bytes));
  PKB_CUDA(cudaMemcpyAsync(am->in_f32.p, feats, in_bytes, cudaMemcpyHostToDevice, c->stream));
  PKB_CUDA(cudaMemsetAsync(ws.row_map.p, 0xFF, static_cast<size_t>(rows) * sizeof(int32_t), c->stream));
  __nv_bfloat16 *hi = ws.feat_hi.as<__nv_bfloat16>();
  __nv_bfloat16 *lo = am->planes == 2 ? ws.feat_lo.as<__nv_bfloat16>() : nullptr;
  PKB_TRY(pkb::launch_pack_padded(c, am->in_f32.as<float>(), m, feat_dim, dp, am->left, am->right,
                                  ws.pad_off.as<int64_t>(), hi, lo, ws.row_map.as<int32_t>(), am->fp16));
  InputView in;
  in.hi = hi;
  in.lo = lo;
  in.rows = rows;
  in.cols = (am->left + am->right + 1) * dp;
  in.pitch_elems = dp;
  return pkb::nnet_forward_refined(am, &ws, &am->rf, in, ws.row_map.as<int32_t>(), pkb::kFinalLoglik,
                                   prob_scale, am->out_f32.as<float>());
}

int pkb_am_compute(pkb_ctx_t *c, pkb_am_t *am, const float *feats, const int32_t *num_frames,
                   int n_utts, int feat_dim, float prob_scale, float *loglik_out) {
  std::vector<int64_t> pad_off;
  PKB_TRY(am_compute_device(c, am, feats, num_frames, n_utts, feat_dim, prob_scale, "pkb_am_compute",
                            &pad_off));
  const BatchMeta &m = am->meta;
  if (m.total_frames == 0) return PKB_OK;
  PKB_REQUIRE(loglik_out != nullptr, "pkb_am_compute: loglik_out is NULL");
  PKB_TRY(pkb::copy_rows_compact(c, loglik_out, am->out_f32.p, m, pad_off, am->num_pdfs, 0,
                                 m.total_frames));
  PKB_CUDA(cudaStreamSynchronize(c->stream));
  return pkb::check_device_error(c, "pkb_am_compute");
}

struct pkb_event {
  pkb_ctx_t *c = nullptr;
  cudaEvent_t ev = nullptr;
  bool recorded = false;
};

int pkb_event_create(pkb_ctx_t *c, pkb_event_t **out) {
  PKB_REQUIRE(c && out, "pkb_event_create: NULL argument");
  *out = nullptr;
  PKB_CUDA(cudaSetDevice(c->device));
  cudaEvent_t e;
  PKB_CUDA(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
  pkb_event *ev = new pkb_event;
  ev->c = c;
  ev->ev = e;
  *out = ev;
  return PKB_OK;
}

void pkb_event_destroy(pkb_event_t *ev) {
  if (ev == nullptr) return;
  cudaEventDestroy(ev->ev);
  delete ev;
}

int pkb_event_record(pkb_ctx_t *c, pkb_event_t *ev) {
  PKB_REQUIRE(c && ev && ev->c == c, "pkb_event_record: NULL argument or event of another context");
  PKB_CUDA(cudaEventRecord(ev->ev, c->stream));
  ev->recorded = true;
  return PKB_OK;
}

int pkb_event_wait(pkb_event_t *ev) {
  PKB_REQUIRE(ev != nullptr, "pkb_event_wait: NULL event");
  PKB_REQUIRE(ev->recorded, "pkb_event_wait: event was never recorded");
  PKB_CUDA(cudaEventSynchronize(ev->ev));
  return PKB_OK;
}

int pkb_event_query(pkb_event_t *ev, int *done) {
  PKB_REQUIRE(ev && done, "pkb_event_query: NULL argument");
  *done = 0;
  if (!ev->recorded) return PKB_OK;
  const cudaError_t e = cudaEventQuery(ev->ev);
  if (e == cudaSuccess) {
    *done = 1;
    return PKB_OK;
  }
  if (e == cudaErrorNotReady) return PKB_OK;
  PKB_CUDA(e);
  return PKB_OK;
}

int pkb_am_compute_chunked(pkb_ctx_t *c, pkb_am_t *am, const float *feats, int32_t num_frames,
                           int feat_dim, float prob_scale, float *loglik_out, int chunk_frames,
                           pkb_event_t *const *events, int n_events) {
  PKB_REQUIRE(chunk_frames > 0, "pkb_am_compute_chunked: chunk_frames must be positive");
  PKB_REQUIRE(num_frames >= 0, "pkb_am_compute_chunked: num_frames < 0");
  const int n_chunks = (num_frames + chunk_frames - 1) / chunk_frames;
  PKB_REQUIRE(n_events >= n_chunks && (events != nullptr || n_chunks == 0),
              "pkb_am_compute_chunked: %d events for %d chunks", n_events, n_chunks);
  for (int i = 0; i < n_chunks; ++i)
    PKB_REQUIRE(events[i] != nullptr && events[i]->c == c,
                "pkb_am_compute_chunked: event %d is NULL or belongs to another context", i);
  std::vector<int64_t> pad_off;
  PKB_TRY(am_compute_device(c, am, feats, &num_frames, 1, feat_dim, prob_scale,
                            "pkb_am_compute_chunked", &pad_off));
  if (num_frames == 0) return PKB_OK;
  PKB_REQUIRE(loglik_out != nullptr, "pkb_am_compute_chunked: loglik_out is NULL");
  const BatchMeta &m = am->meta;
  for (int i = 0; i < n_chunks; ++i) {
    const int64_t r0 = static_cast<int64_t>(i) * chunk_frames;
    const int64_t n = std::min<int64_t>(chunk_frames, num_frames - r0);
    PKB_TRY(pkb::copy_rows_compact(c, loglik_out + r0 * am->num_pdfs, am->out_f32.p, m,
                                   pad_off, am->num_pdfs, r0, n));
    PKB_TRY(pkb_event_record(c, events[i]));
  }
  return PKB_OK;
}

int pkb_nnet_propagate(pkb_ctx_t *c, pkb_am_t *am, const float *in_host, int rows, int in_dim,
                       float *out) {
  PKB_REQUIRE(c && am, "pkb_nnet_propagate: NULL argument");
  PKB_REQUIRE(am->c == c, "pkb_nnet_propagate: model belongs to another context");
  PKB_REQUIRE(in_dim == am->input_dim, "pkb_nnet_propagate: in_dim %d != nnet input dim %d", in_dim,
              am->input_dim);
  PKB_REQUIRE(rows >= 0, "pkb_nnet_propagate: rows < 0");
  if (rows == 0) return PKB_OK;
  PKB_REQUIRE(in_host && out, "pkb_nnet_propagate: in / out is NULL");
  PKB_CUDA(cudaSetDevice(c->device));
  Workspace &ws = am->ws;
  PKB_TRY(pkb::workspace_ensure(am, &ws, rows));
  // the column layout stage 0 was packed for: feat_dim_pad columns per context frame, or one
  // group of in_dim columns padded to 16 bytes
  const int group = am->feat_dim > 0 ? am->feat_dim : in_dim;
  const int group_pad = am->feat_dim > 0 ? am->feat_dim_pad : (in_dim + 7) / 8 * 8;
  const int groups = in_dim / group;
  const int dp = groups * group_pad;
  const int out_dim = am->stages.back().out_dim;
  PKB_TRY(ws.feat_hi.ensure(static_cast<size_t>(rows) * dp * 2));
  if (am->planes == 2) PKB_TRY(ws.feat_lo.ensure(static_cast<size_t>(rows) * dp * 2));
  const size_t in_bytes = static_cast<size_t>(rows) * in_dim * sizeof(float);
  const size_t out_bytes = static_cast<size_t>(rows) * out_dim * sizeof(float);
  PKB_TRY(am->in_f32.ensure(in_bytes));
  PKB_TRY(am->out_f32.ensure(out_bytes));
  PKB_CUDA(cudaMemcpyAsync(am->in_f32.p, in_host, in_bytes, cudaMemcpyHostToDevice, c->stream));
  __nv_bfloat16 *hi = ws.feat_hi.as<__nv_bfloat16>();
  __nv_bfloat16 *lo = am->planes == 2 ? ws.feat_lo.as<__nv_bfloat16>() : nullptr;
  PKB_TRY(pkb::launch_pack_plain(c, am->in_f32.as<float>(), rows, groups, group, group_pad, hi, lo, am->fp16));
  InputView in;
  in.hi = hi;
  in.lo = lo;
  in.rows = rows;
  in.cols = dp;
  in.pitch_elems = dp;
  const pkb::FinalMode mode = am->softmax_last ? pkb::kFinalProb : pkb::kFinalRaw;
  PKB_TRY(pkb::nnet_forward(am, &ws, in, mode, 1.0f, am->out_f32.as<float>()));
  PKB_CUDA(cudaMemcpyAsync(out, am->out_f32.p, out_bytes, cudaMemcpyDeviceToHost, c->stream));
  PKB_CUDA(cudaStreamSynchronize(c->stream));
  return pkb::check_device_error(c, "pkb_nnet_propagate");
}

// ---------------------------------------------------------------- batch pipeline
int pkb_batch_create(pkb_ctx_t *c, pkb_am_t *am, int n_utts, const int32_t *num_samples,
                     const float *global_stats, float prob_scale, pkb_batch_t **out) {
  PKB_REQUIRE(c && out, "pkb_batch_create: NULL argument");
  PKB_REQUIRE(global_stats, "pkb_batch_create: global_stats is NULL");
  PKB_REQUIRE(n_utts == 0 || num_samples, "pkb_batch_create: num_samples is NULL");
  PKB_REQUIRE(!am || am->c == c, "pkb_batch_create: model belongs to another context");
  PKB_REQUIRE(!am || am->feat_dim == pkb::kMel,
              "pkb_batch_create: the model's feature dim must be %d", pkb::kMel);
  PKB_CUDA(cudaSetDevice(c->device));
  std::unique_ptr<pkb_batch, decltype(&pkb_batch_destroy)> b(new pkb_batch(), pkb_batch_destroy);
  b->c = c;
  b->am = am;
  b->prob_scale = prob_scale;
  memcpy(b->global_stats, global_stats, sizeof(b->global_stats));
  PKB_TRY(b->meta.build_from_samples(num_samples, n_utts));
  PKB_TRY(b->meta.upload(c->stream));
  const BatchMeta &m = b->meta;
  const size_t feat_bytes = static_cast<size_t>(m.total_frames) * pkb::kMel * sizeof(float);
  PKB_TRY(b->pcm.ensure(std::max<size_t>(2, static_cast<size_t>(m.total_samples) * 2)));
  PKB_TRY(b->raw.ensure(std::max<size_t>(4, feat_bytes)));
  PKB_TRY(b->feats.ensure(std::max<size_t>(4, feat_bytes)));
  PKB_TRY(b->sum.ensure(sizeof(double)));
  if (am) {
    std::vector<int64_t> &pad_off = b->pad_off;
    pkb::padded_rows(m, am->left, am->right, &pad_off, &b->padded, &b->gemm_rows);
    Workspace &ws = b->ws;
    ws.fast_only = am->refine != 0;  // the FP8 operand planes only exist for the refined rows
    PKB_TRY(pkb::workspace_ensure(am, &ws, b->gemm_rows));
    const int dp = am->feat_dim_pad;
    const size_t plane_bytes = std::max<size_t>(16, static_cast<size_t>(b->padded) * dp * 2);
    PKB_TRY(ws.feat_hi.ensure(plane_bytes));
    if (am->planes == 2) PKB_TRY(ws.feat_lo.ensure(plane_bytes));
    PKB_TRY(ws.pad_off.ensure(std::max<size_t>(8, pad_off.size() * sizeof(int64_t))));
    PKB_TRY(ws.row_map.ensure(std::max<size_t>(4, static_cast<size_t>(b->gemm_rows) * 4)));
    // padded-row layout: one output row per GEMM row
    PKB_TRY(b->loglik.ensure(
        std::max<size_t>(4, static_cast<size_t>(b->gemm_rows) * am->num_pdfs * sizeof(float))));
    if (!pad_off.empty())
      PKB_TRY(pkb::upload(c, ws.pad_off.p, pad_off.data(), pad_off.size() * sizeof(int64_t)));
    // zero the planes once: rows of empty utterances are never written
    cudaMemsetAsync(ws.feat_hi.p, 0, plane_bytes, c->stream);
    if (am->planes == 2) cudaMemsetAsync(ws.feat_lo.p, 0, plane_bytes, c->stream);
    PKB_TRY(pkb::launch_row_map(c, m, am->left, am->right, ws.pad_off.as<int64_t>(),
                                ws.row_map.as<int32_t>(), b->gemm_rows));
    b->planes.hi = ws.feat_hi.as<__nv_bfloat16>();
    b->planes.lo = am->planes == 2 ? ws.feat_lo.as<__nv_bfloat16>() : nullptr;
    b->planes.d_pad_off = ws.pad_off.as<int64_t>();
    b->planes.left = am->left;
    b->planes.right = am->right;
    b->planes.dim_pad = dp;
    b->planes.fp16 = am->fp16;
  }
  PKB_TRY(pkb::prepare_cmvn_tables(c, global_stats));
  PKB_CUDA(cudaStreamSynchronize(c->stream));
  *out = b.release();
  return PKB_OK;
}

void pkb_batch_destroy(pkb_batch_t *b) {
  if (!b) return;
  if (b->c) {
    cudaSetDevice(b->c->device);
    cudaStreamSynchronize(b->c->stream);
  }
  delete b;
}

int64_t pkb_batch_num_frames(const pkb_batch_t *b) { return b ? b->meta.total_frames : 0; }
int64_t pkb_batch_num_samples(const pkb_batch_t *b) { return b ? b->meta.total_samples : 0; }

int pkb_batch_set_pcm_i16(pkb_batch_t *b, const int16_t *pcm) {
  PKB_REQUIRE(b, "pkb_batch_set_pcm_i16: batch is NULL");
  if (b->meta.total_samples == 0) return PKB_OK;
  PKB_REQUIRE(pcm, "pkb_batch_set_pcm_i16: pcm is NULL");
  PKB_CUDA(cudaSetDevice(b->c->device));
  PKB_CUDA(cudaMemcpyAsync(b->pcm.p, pcm, static_cast<size_t>(b->meta.total_samples) * 2,
                           cudaMemcpyHostToDevice, b->c->stream));
  return PKB_OK;
}

int pkb_batch_synth_pcm(pkb_batch_t *b, uint64_t seed, uint64_t first_utt_id) {
  PKB_REQUIRE(b, "pkb_batch_synth_pcm: batch is NULL");
  PKB_CUDA(cudaSetDevice(b->c->device));
  return pkb::launch_synth_pcm(b->c, b->pcm.as<int16_t>(), b->meta, seed, first_utt_id);
}

int pkb_batch_run(pkb_batch_t *b, int stages) {
  PKB_REQUIRE(b, "pkb_batch_run: batch is NULL");
  Ctx *c = b->c;
  PKB_CUDA(cudaSetDevice(c->device));
  if (stages & PKB_STAGE_FBANK)
    PKB_TRY(pkb::launch_fbank_i16(c, b->pcm.as<int16_t>(), b->meta, b->raw.as<float>()));
  if (stages & PKB_STAGE_CMVN) {
    PKB_TRY(pkb::prepare_cmvn_tables(c, b->global_stats));
    const bool skip_f32 = (stages & PKB_STAGE_NO_FEATS) && b->am;
    PKB_TRY(pkb::launch_cmvn(c, b->raw.as<float>(), b->meta, skip_f32 ? nullptr : b->feats.as<float>(),
                             b->am ? &b->planes : nullptr));
  }
  if (stages & PKB_STAGE_NNET) {
    PKB_REQUIRE(b->am, "pkb_batch_run: PKB_STAGE_NNET needs a model");
    pkb_am *am = b->am;
    InputView in;
    in.hi = b->planes.hi;
    in.lo = b->planes.lo;
    in.rows = b->gemm_rows;
    in.cols = (am->left + am->right + 1) * am->feat_dim_pad;
    in.pitch_elems = am->feat_dim_pad;
    const int32_t *row_map = b->ws.row_map.as<int32_t>();
    if (b->compact)
      PKB_TRY(pkb::nnet_forward_refined(am, &b->ws, &b->rf, in, row_map, pkb::kFinalCompact, b->prob_scale,
                                        nullptr, b->loglik16.as<uint16_t>(), b->loglik_off.as<float>()));
    else
      PKB_TRY(pkb::nnet_forward_refined(am, &b->ws, &b->rf, in, row_map, pkb::kFinalLoglik, b->prob_scale,
                                        b->loglik.as<float>()));
  }
  return PKB_OK;
}

int pkb_batch_refine_stats(const pkb_batch_t *b, int64_t *rows, int64_t *refined) {
  PKB_REQUIRE(b, "pkb_batch_refine_stats: batch is NULL");
  if (rows) *rows = b->rf.last_rows;
  if (refined) *refined = b->rf.last_selected;
  return PKB_OK;
}

int pkb_am_set_refine_margin(pkb_am_t *am, float margin) {
  PKB_REQUIRE(am, "pkb_am_set_refine_margin: model is NULL");
  PKB_REQUIRE(margin >= 0.0f && margin < 1.0e4f, "pkb_am_set_refine_margin: margin %g out of range", margin);
  am->refine_margin = margin;
  return PKB_OK;
}

int pkb_batch_set_compact(pkb_batch_t *b, int on) {
  PKB_REQUIRE(b, "pkb_batch_set_compact: batch is NULL");
  PKB_REQUIRE(b->am, "pkb_batch_set_compact: the batch has no model");
  if ((on != 0) == b->compact) return PKB_OK;
  PKB_REQUIRE(!on || b->am->softmax_last, "pkb_batch_set_compact: the model does not end in a softmax");
  PKB_CUDA(cudaSetDevice(b->c->device));
  PKB_CUDA(cudaStreamSynchronize(b->c->stream));  // nothing may still be writing the buffer we free
  const size_t elems = std::max<size_t>(4, static_cast<size_t>(b->gemm_rows) * b->am->num_pdfs);
  if (on) {
    b->loglik.release();
    PKB_TRY(b->loglik16.ensure(elems * sizeof(uint16_t)));
    PKB_TRY(b->loglik_off.ensure(std::max<size_t>(4, static_cast<size_t>(b->gemm_rows) * sizeof(float))));
  } else {
    b->loglik16.release();
    b->loglik_off.release();
    PKB_TRY(b->loglik.ensure(elems * sizeof(float)));
  }
  b->compact = on != 0;
  return PKB_OK;
}

int pkb_loglik16_expand(const uint16_t *h, const float *off, int64_t n_frames, int num_pdfs,
                        float prob_scale, float *out) {
  PKB_REQUIRE(n_frames >= 0 && num_pdfs >= 0, "pkb_loglik16_expand: negative size");
  if (n_frames == 0 || num_pdfs == 0) return PKB_OK;
  PKB_REQUIRE(h && off && out, "pkb_loglik16_expand: NULL argument");
  for (int64_t t = 0; t < n_frames; ++t) {
    const uint16_t *row = h + t * num_pdfs;
    float *dst = out + t * num_pdfs;
    const float o = off[t];
    for (int p = 0; p < num_pdfs; ++p) {
      __half_raw r;
      r.x = row[p];
      dst[p] = prob_scale * (__half2float(__half(r)) + o);
    }
  }
  return PKB_OK;
}

static int batch_buf(pkb_batch_t *b, int which, char **ptr, size_t *row_bytes, int64_t *rows) {
  switch (which) {
    case PKB_BUF_PCM:
      *ptr = b->pcm.as<char>();
      *row_bytes = 2;
      *rows = b->meta.total_samples;
      return PKB_OK;
    case PKB_BUF_RAW:
      *ptr = b->raw.as<char>();
      *row_bytes = pkb::kMel * sizeof(float);
      *rows = b->meta.total_frames;
      return PKB_OK;
    case PKB_BUF_FEATS:
      *ptr = b->feats.as<char>();
      *row_bytes = pkb::kMel * sizeof(float);
      *rows = b->meta.total_frames;
      return PKB_OK;
    case PKB_BUF_LOGLIK:
      PKB_REQUIRE(b->am, "batch has no model: no log-likelihood buffer");
      PKB_REQUIRE(!b->compact, "the batch writes the compact output: read PKB_BUF_LOGLIK16 / PKB_BUF_LOGLIK_OFF");
      *ptr = b->loglik.as<char>();
      *row_bytes = static_cast<size_t>(b->am->num_pdfs) * sizeof(float);
      *rows = b->meta.total_frames;
      return PKB_OK;
    case PKB_BUF_LOGLIK16:
    case PKB_BUF_LOGLIK_OFF:
      PKB_REQUIRE(b->am && b->compact, "the compact output is off (pkb_batch_set_compact)");
      *ptr = which == PKB_BUF_LOGLIK16 ? b->loglik16.as<char>() : b->loglik_off.as<char>();
      *row_bytes = which == PKB_BUF_LOGLIK16 ? static_cast<size_t>(b->am->num_pdfs) * sizeof(uint16_t)
                                             : sizeof(float);
      *rows = b->meta.total_frames;
      return PKB_OK;
  }
  pkb::set_error("unknown buffer id %d", which);
  return PKB_ERR_INVALID;
}

int pkb_batch_get_rows(pkb_batch_t *b, int which, int64_t row0, int64_t n_rows, void *host_dst) {
  PKB_REQUIRE(b, "pkb_batch_get_rows: batch is NULL");
  char *ptr = nullptr;
  size_t row_bytes = 0;
  int64_t rows = 0;
  PKB_TRY(batch_buf(b, which, &ptr, &row_bytes, &rows));
  PKB_REQUIRE(row0 >= 0 && n_rows >= 0 && row0 + n_rows <= rows,
              "pkb_batch_get_rows: range [%lld, %lld) outside [0, %lld)", (long long)row0,
              (long long)(row0 + n_rows), (long long)rows);
  if (n_rows == 0) return PKB_OK;
  PKB_REQUIRE(host_dst, "pkb_batch_get_rows: host_dst is NULL");
  PKB_CUDA(cudaSetDevice(b->c->device));
  // stored with padded rows: compacted per utterance on the way out
  if (which == PKB_BUF_LOGLIK)
    return pkb::copy_rows_compact(b->c, host_dst, b->loglik.p, b->meta, b->pad_off, b->am->num_pdfs, row0,
                                  n_rows);
  if (which == PKB_BUF_LOGLIK16)
    return pkb::copy_rows_compact(b->c, host_dst, b->loglik16.p, b->meta, b->pad_off, b->am->num_pdfs,
                                  row0, n_rows, sizeof(uint16_t));
  if (which == PKB_BUF_LOGLIK_OFF)
    return pkb::copy_rows_compact(b->c, host_dst, b->loglik_off.p, b->meta, b->pad_off, 1, row0, n_rows);
  PKB_CUDA(cudaMemcpyAsync(host_dst, ptr + row0 * row_bytes, n_rows * row_bytes,
                           cudaMemcpyDeviceToHost, b->c->stream));
  return PKB_OK;
}

int pkb_batch_get(pkb_batch_t *b, int which, void *host_dst) {
  PKB_REQUIRE(b, "pkb_batch_get: batch is NULL");
  char *ptr = nullptr;
  size_t row_bytes = 0;
  int64_t rows = 0;
  PKB_TRY(batch_buf(b, which, &ptr, &row_bytes, &rows));
  return pkb_batch_get_rows(b, which, 0, rows, host_dst);
}

int pkb_batch_checksum(pkb_batch_t *b, int which, double *sum_out) {
  PKB_REQUIRE(b && sum_out, "pkb_batch_checksum: NULL argument");
  PKB_REQUIRE(which != PKB_BUF_PCM && which != PKB_BUF_LOGLIK16 && which != PKB_BUF_LOGLIK_OFF,
              "pkb_batch_checksum: FP32 per-frame buffers only");
  PKB_CUDA(cudaSetDevice(b->c->device));
  char *ptr = nullptr;
  size_t row_bytes = 0;
  int64_t rows = 0;
  PKB_TRY(batch_buf(b, which, &ptr, &row_bytes, &rows));
  const int64_t n = rows * static_cast<int64_t>(row_bytes / sizeof(float));
  if (which == PKB_BUF_LOGLIK)
    PKB_TRY(pkb::launch_checksum_rows(b->c, b->loglik.as<float>(), b->am->num_pdfs, b->gemm_rows,
                                      b->ws.row_map.as<int32_t>(), b->sum.as<double>()));
  else
    PKB_TRY(pkb::launch_checksum(b->c, reinterpret_cast<const float *>(ptr), n, b->sum.as<double>()));
  PKB_CUDA(cudaMemcpyAsync(sum_out, b->sum.p, sizeof(double), cudaMemcpyDeviceToHost, b->c->stream));
  PKB_CUDA(cudaStreamSynchronize(b->c->stream));
  return pkb::check_device_error(b->c, "pkb_batch_checksum");
}

// ---------------------------------------------------------------- GPU Viterbi
int pkb_fst_create(pkb_ctx_t *c, int num_states, int start_state, const float *final_weights,
                   const int32_t *first_arc, int num_arcs, const int32_t *arcs, pkb_fst_t **fst) {
  PKB_REQUIRE(c && fst, "pkb_fst_create: NULL argument");
  *fst = nullptr;
  PKB_CUDA(cudaSetDevice(c->device));
  return pkb::fst_build(c, num_states, start_state, final_weights, first_arc, num_arcs, arcs, fst);
}

int pkb_fst_load(pkb_ctx_t *c, const char *path, pkb_fst_t **fst) {
  PKB_REQUIRE(c && path && fst, "pkb_fst_load: NULL argument");
  *fst = nullptr;
  File fd;
  PKB_TRY(fd.open(path));
  // Fst::Read, src/fst.cc:29-92
  char name[32];
  PKB_TRY(fd.read(name, 32));
  name[31] = 0;
  if (strcmp(name, "pk::fst_0") != 0) {
    pkb::set_error("Corruption: section_name == 'pk::fst_0' expected, but '%s' found", name);
    return PKB_ERR_CORRUPT;
  }
  int32_t size = 0, ns = 0, na = 0, start = 0;
  PKB_TRY(fd.read_i32(&size));
  PKB_TRY(fd.read_i32(&ns));
  PKB_TRY(fd.read_i32(&na));
  PKB_TRY(fd.read_i32(&start));
  const int64_t expect = 12 + static_cast<int64_t>(ns) * 8 + static_cast<int64_t>(na) * 16;
  if (ns < 0 || na < 0 || expect != size) {
    pkb::set_error("Corruption: section_size == %lld expected, but %d found", static_cast<long long>(expect), size);
    return PKB_ERR_CORRUPT;
  }
  std::vector<float> fin(ns);
  std::vector<int32_t> first(ns), arcs(static_cast<size_t>(na) * 4);
  if (ns) PKB_TRY(fd.read(fin.data(), sizeof(float) * ns));
  if (ns) PKB_TRY(fd.read(first.data(), sizeof(int32_t) * ns));
  if (na) PKB_TRY(fd.read(arcs.data(), sizeof(int32_t) * 4 * static_cast<size_t>(na)));
  return pkb_fst_create(c, ns, start, fin.data(), first.data(), na, arcs.data(), fst);
}

void pkb_fst_destroy(pkb_fst_t *fst) {
  if (!fst) return;
  if (fst->c) cudaSetDevice(fst->c->device);
  delete fst;
}

int pkb_batch_decode(pkb_batch_t *b, const pkb_fst_t *fst, float beam, int max_tokens, int max_words,
                     int32_t *words_out, int32_t *n_words_out, float *weight_out) {
  PKB_REQUIRE(b && fst, "pkb_batch_decode: NULL argument");
  PKB_REQUIRE(b->am, "pkb_batch_decode: the batch has no model");
  PKB_REQUIRE(!b->compact, "pkb_batch_decode: reads the FP32 log-likelihoods (switch the compact output off)");
  PKB_TRY(pkb::check_decode_graph(b->c, b->am, fst, "pkb_batch_decode"));
  PKB_TRY(pkb::check_decode_outputs(max_words, words_out, n_words_out, weight_out, "pkb_batch_decode"));
  Ctx *c = b->c;
  PKB_CUDA(cudaSetDevice(c->device));
  const int n = b->meta.n_utts;
  if (n == 0) return PKB_OK;
  pkb::ViterbiConfig cfg;
  if (beam > 0.0f) cfg.beam = beam;
  if (max_tokens > 0) cfg.max_tokens = max_tokens;
  cfg.max_words = max_words;
  pkb_am *am = b->am;
  const size_t tid_bytes = am->tid2pdf.size() * sizeof(int32_t);
  if (b->vit_tid2pdf.cap < tid_bytes) {
    PKB_TRY(b->vit_tid2pdf.ensure(tid_bytes));
    PKB_CUDA(cudaMemcpyAsync(b->vit_tid2pdf.p, am->tid2pdf.data(), tid_bytes, cudaMemcpyHostToDevice, c->stream));
  }
  const size_t words_bytes = static_cast<size_t>(n) * max_words * sizeof(int32_t);
  const size_t out_bytes = words_bytes + static_cast<size_t>(n) * (sizeof(int32_t) + sizeof(float));
  PKB_TRY(b->vit_out.ensure(out_bytes));
  int32_t *d_words = b->vit_out.as<int32_t>();
  int32_t *d_nw = reinterpret_cast<int32_t *>(b->vit_out.as<char>() + words_bytes);
  float *d_wt = reinterpret_cast<float *>(d_nw + n);
  PKB_CUDA(cudaMemsetAsync(b->vit_out.p, 0, out_bytes, c->stream));
  PKB_TRY(pkb::launch_viterbi(c, fst, cfg, b->loglik.as<float>(), am->num_pdfs, b->ws.pad_off.as<int64_t>(),
                              b->meta.d_num_frames, n, b->vit_tid2pdf.as<int32_t>(),
                              static_cast<int>(am->tid2pdf.size()), &b->vit_work, d_words, d_nw, d_wt));
  PKB_CUDA(cudaMemcpyAsync(words_out, d_words, words_bytes, cudaMemcpyDeviceToHost, c->stream));
  PKB_CUDA(cudaMemcpyAsync(n_words_out, d_nw, sizeof(int32_t) * n, cudaMemcpyDeviceToHost, c->stream));
  PKB_CUDA(cudaMemcpyAsync(weight_out, d_wt, sizeof(float) * n, cudaMemcpyDeviceToHost, c->stream));
  PKB_CUDA(cudaStreamSynchronize(c->stream));
  return pkb::check_device_error(c, "pkb_batch_decode");
}

static_assert(sizeof(pkb_lattice_arc_t) == 28 && offsetof(pkb_lattice_arc_t, acoustic_cost) == 24,
              "pkb_lattice_arc_t is 28 bytes without padding");

int pkb_batch_lattice(pkb_batch_t *b, const pkb_fst_t *fst, float beam, float lattice_beam, int max_tokens,
                      int max_arcs, int64_t *n_arcs_out, double *best_cost_out) {
  PKB_REQUIRE(b && fst && n_arcs_out && best_cost_out, "pkb_batch_lattice: NULL argument");
  PKB_REQUIRE(b->am, "pkb_batch_lattice: the batch has no model");
  PKB_REQUIRE(!b->compact, "pkb_batch_lattice: reads the FP32 log-likelihoods (switch the compact output off)");
  PKB_REQUIRE(lattice_beam > 0.0f, "pkb_batch_lattice: lattice_beam must be > 0 (got %g)", lattice_beam);
  PKB_TRY(pkb::check_decode_graph(b->c, b->am, fst, "pkb_batch_lattice"));
  Ctx *c = b->c;
  PKB_CUDA(cudaSetDevice(c->device));
  b->lat_total = 0;
  b->lat_fst = nullptr;
  const int n = b->meta.n_utts;
  if (n == 0) {
    b->lat_fst = fst;
    b->lat_rec = pkb::LatticeRecords{};
    return PKB_OK;
  }
  pkb::ViterbiConfig cfg;
  if (beam > 0.0f) cfg.beam = beam;
  if (max_tokens > 0) cfg.max_tokens = max_tokens;
  pkb_am *am = b->am;
  const size_t tid_bytes = am->tid2pdf.size() * sizeof(int32_t);
  if (b->vit_tid2pdf.cap < tid_bytes) {
    PKB_TRY(b->vit_tid2pdf.ensure(tid_bytes));
    PKB_CUDA(cudaMemcpyAsync(b->vit_tid2pdf.p, am->tid2pdf.data(), tid_bytes, cudaMemcpyHostToDevice, c->stream));
  }
  int t_max = 0;
  for (int u = 0; u < n; ++u) t_max = std::max(t_max, b->meta.num_frames[u]);
  pkb::Lattice lat{};
  // default: the most the search can log, every arc of the graph at every time of the longest
  // utterance (1.84 M entries, 14.7 MB, for 10 s on the 40-word loop; 33 M, 267 MB, on the 180-word loop)
  const int64_t bound = static_cast<int64_t>(t_max + 1) * std::max(fst->num_arcs, 1);
  lat.max_arcs = max_arcs > 0 ? max_arcs : static_cast<int>(std::min<int64_t>(bound, INT32_MAX));
  lat.grp_stride = 2 * (t_max + 1);
  lat.beam = lattice_beam;
  // per utterance: the log; group offsets; kept count, best cost and first output record
  PKB_TRY(b->lat_log.ensure(static_cast<size_t>(n) * lat.max_arcs * sizeof(unsigned long long)));
  const size_t grp_bytes = (static_cast<size_t>(n) * lat.grp_stride * sizeof(int) + 7) & ~static_cast<size_t>(7);
  PKB_TRY(b->lat_aux.ensure(grp_bytes + 3 * sizeof(int64_t) * static_cast<size_t>(n)));
  lat.log = b->lat_log.as<unsigned long long>();
  lat.grp = b->lat_aux.as<int>();
  lat.n_out = reinterpret_cast<long long *>(b->lat_aux.as<char>() + grp_bytes);
  lat.best_out = reinterpret_cast<double *>(lat.n_out + n);
  long long *d_first = lat.n_out + 2 * n;
  PKB_TRY(pkb::launch_lattice(c, fst, cfg, b->loglik.as<float>(), am->num_pdfs, b->ws.pad_off.as<int64_t>(),
                              b->meta.d_num_frames, n, b->vit_tid2pdf.as<int32_t>(), &b->vit_work, lat));
  static_assert(sizeof(long long) == sizeof(int64_t), "int64_t is long long");
  PKB_CUDA(cudaMemcpyAsync(n_arcs_out, lat.n_out, sizeof(int64_t) * n, cudaMemcpyDeviceToHost, c->stream));
  PKB_CUDA(cudaMemcpyAsync(best_cost_out, lat.best_out, sizeof(double) * n, cudaMemcpyDeviceToHost, c->stream));
  PKB_CUDA(cudaStreamSynchronize(c->stream));
  PKB_TRY(pkb::check_device_error(c, "pkb_batch_lattice"));
  // the kept arcs as records, every utterance's back to back
  std::vector<long long> first(n);
  int64_t total = 0;
  for (int u = 0; u < n; ++u) {
    first[u] = total;
    total += std::max<int64_t>(n_arcs_out[u], 0);
  }
  PKB_TRY(b->lat_arcs.ensure(std::max<int64_t>(total, 1) * sizeof(pkb_lattice_arc_t)));
  PKB_CUDA(cudaMemcpyAsync(d_first, first.data(), sizeof(long long) * n, cudaMemcpyHostToDevice, c->stream));
  PKB_TRY(pkb::lattice_expand(c, fst, lat, b->loglik.as<float>(), am->num_pdfs, b->ws.pad_off.as<int64_t>(), n,
                              b->vit_tid2pdf.as<int32_t>(), d_first, b->lat_arcs.as<pkb_lattice_arc_t>()));
  PKB_CUDA(cudaStreamSynchronize(c->stream));
  PKB_TRY(pkb::check_device_error(c, "pkb_batch_lattice"));
  b->lat_total = total;
  b->lat_fst = fst;
  b->lat_rec.arcs = b->lat_arcs.as<pkb_lattice_arc_t>();
  b->lat_rec.first = d_first;
  b->lat_rec.n_arcs = lat.n_out;
  b->lat_rec.best = lat.best_out;
  b->lat_rec.n_utts = n;
  return PKB_OK;
}

int pkb_batch_lattice_get(pkb_batch_t *b, pkb_lattice_arc_t *arcs_out) {
  PKB_REQUIRE(b, "pkb_batch_lattice_get: the batch is NULL");
  PKB_REQUIRE(b->lat_total >= 0, "pkb_batch_lattice_get: no pkb_batch_lattice on this batch yet");
  if (b->lat_total == 0) return PKB_OK;
  PKB_REQUIRE(arcs_out, "pkb_batch_lattice_get: NULL argument");
  PKB_CUDA(cudaSetDevice(b->c->device));
  PKB_CUDA(cudaMemcpyAsync(arcs_out, b->lat_arcs.p, sizeof(pkb_lattice_arc_t) * b->lat_total,
                           cudaMemcpyDeviceToHost, b->c->stream));
  PKB_CUDA(cudaStreamSynchronize(b->c->stream));
  return pkb::check_device_error(b->c, "pkb_batch_lattice_get");
}

int pkb_batch_nbest(pkb_batch_t *b, const pkb_fst_t *fst, int n, int max_words, int32_t *words_out,
                    int32_t *n_words_out, double *graph_cost_out, double *acoustic_cost_out, int32_t *n_hyps_out) {
  PKB_REQUIRE(b && fst, "pkb_batch_nbest: NULL argument");
  PKB_REQUIRE(b->lat_fst, "pkb_batch_nbest: no valid pkb_batch_lattice on this batch");
  PKB_REQUIRE(b->lat_fst == fst, "pkb_batch_nbest: the FST is not the one of the latest pkb_batch_lattice");
  PKB_TRY(pkb::check_nbest_args(n, max_words, words_out, n_words_out, graph_cost_out, acoustic_cost_out,
                                n_hyps_out, "pkb_batch_nbest"));
  PKB_CUDA(cudaSetDevice(b->c->device));
  PKB_TRY(pkb::launch_nbest(b->c, fst, b->lat_rec, n, max_words, &b->nbest_work, words_out, n_words_out,
                            graph_cost_out, acoustic_cost_out, n_hyps_out));
  return pkb::check_device_error(b->c, "pkb_batch_nbest");
}

// ---------------------------------------------------------------- fused host path
int pkb_pcm_to_loglik_i16(pkb_ctx_t *c, pkb_am_t *am, const int16_t *pcm,
                          const int32_t *num_samples, int n_utts, const float *global_stats,
                          float prob_scale, float *loglik_out, float *feats_out,
                          int32_t *num_frames_out) {
  PKB_REQUIRE(c && am, "pkb_pcm_to_loglik_i16: NULL argument");
  pkb_batch_t *created = nullptr;
  PKB_TRY(pkb_batch_create(c, am, n_utts, num_samples, global_stats, prob_scale, &created));
  std::unique_ptr<pkb_batch, decltype(&pkb_batch_destroy)> b(created, pkb_batch_destroy);
  if (num_frames_out)
    for (int u = 0; u < n_utts; ++u) num_frames_out[u] = b->meta.num_frames[u];
  if (b->meta.total_frames == 0) return PKB_OK;
  PKB_TRY(pkb_batch_set_pcm_i16(b.get(), pcm));
  PKB_TRY(pkb_batch_run(b.get(), PKB_STAGE_ALL));
  if (loglik_out) PKB_TRY(pkb_batch_get(b.get(), PKB_BUF_LOGLIK, loglik_out));
  if (feats_out) PKB_TRY(pkb_batch_get(b.get(), PKB_BUF_FEATS, feats_out));
  PKB_CUDA(cudaStreamSynchronize(c->stream));
  return pkb::check_device_error(c, "pkb_pcm_to_loglik_i16");
}

}  // extern "C"
