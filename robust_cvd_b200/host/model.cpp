// model.cpp -- data model, file formats and small image utilities behind lib_python.
// Reference behaviour cited per function; see model.h.
#include "model.h"

#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstring>
#include <fstream>
#include <iostream>
#include <sstream>
#include <stdexcept>
#include <sys/stat.h>
#include <zlib.h>

namespace rcvdh {

static bool g_logStdout = false;
void setLogToStdout(bool v) { g_logStdout = v; }
void logInfo(const std::string& s) { (g_logStdout ? std::cout : std::cerr) << s << std::endl; }
static bool fileExists(const std::string& f) { struct stat st; return stat(f.c_str(), &st) == 0; }
static void makeDirs(const std::string& dir) {   // mkdir -p
  for (size_t pos = 1; pos <= dir.size(); ++pos)
    if (pos == dir.size() || dir[pos] == '/') { const std::string sub = dir.substr(0, pos); if (!fileExists(sub)) ::mkdir(sub.c_str(), 0777); }
}
static std::string fmtInt6(int v) { char b[32]; snprintf(b, sizeof(b), "%06d", v); return b; }

// Eigen::Quaternion::_transformVector: v + 2w (q x v) + 2 q x (q x v), float arithmetic
Vec3f Quatf::rotate(const Vec3f& v) const {
  float ux = y * v.z - z * v.y, uy = z * v.x - x * v.z, uz = x * v.y - y * v.x;
  ux += ux; uy += uy; uz += uz;
  return {v.x + w * ux + (y * uz - z * uy), v.y + w * uy + (z * ux - x * uz), v.z + w * uz + (x * uy - y * ux)};
}

// --- .raw images: i32 rows, i32 cols, i32 cvType, u64 elemSize, rows*cols*elemSize bytes (lib/core/CvUtil.cpp:25-42) ---
void freadim(const std::string& fileName, Image& dst) {
  FILE* f = fopen(fileName.c_str(), "rb");
  if (!f) throw std::runtime_error("Could not open image file '" + fileName + "'.");
  int32_t hdr[3]; uint64_t es = 0;
  if (fread(hdr, 4, 3, f) != 3 || fread(&es, 8, 1, f) != 1) { fclose(f); throw std::runtime_error("Truncated raw image header."); }
  dst.create(hdr[0], hdr[1], hdr[2]);
  if (es != dst.elemSize()) { fclose(f); throw std::runtime_error("Raw image element size mismatch."); }
  const size_t n = dst.data.size();
  if (n && fread(dst.data.data(), 1, n, f) != n) { fclose(f); throw std::runtime_error("Truncated raw image data."); }
  fclose(f);
}
void fwriteim(const std::string& fileName, const Image& src) {
  FILE* f = fopen(fileName.c_str(), "wb");
  if (!f) throw std::runtime_error("Could not write image file '" + fileName + "'.");
  int32_t hdr[3] = {src.rows, src.cols, src.type}; uint64_t es = src.elemSize();
  fwrite(hdr, 4, 3, f); fwrite(&es, 8, 1, f); fwrite(src.data.data(), 1, src.data.size(), f);
  fclose(f);
}

// --- 8-bit non-interlaced PNG decoder (cv::imread(IMREAD_GRAYSCALE / IMREAD_COLOR) for the mask streams) ---
Image imreadPng(const std::string& fileName, bool grayscale) {
  std::ifstream is(fileName, std::ios::binary);
  Image out;
  if (!is) return out;
  std::vector<uint8_t> buf((std::istreambuf_iterator<char>(is)), std::istreambuf_iterator<char>());
  static const uint8_t sig[8] = {0x89, 'P', 'N', 'G', 0x0d, 0x0a, 0x1a, 0x0a};
  if (buf.size() < 8 || memcmp(buf.data(), sig, 8)) return out;
  auto be32 = [&](size_t o) { return (uint32_t(buf[o]) << 24) | (uint32_t(buf[o + 1]) << 16) | (uint32_t(buf[o + 2]) << 8) | buf[o + 3]; };
  uint32_t w = 0, h = 0; int bitDepth = 0, colorType = 0, interlace = 0;
  std::vector<uint8_t> idat, plte;
  for (size_t o = 8; o + 12 <= buf.size();) {
    const uint32_t len = be32(o); const std::string typ(reinterpret_cast<char*>(&buf[o + 4]), 4);
    if (o + 12 + len > buf.size()) break;
    const uint8_t* d = &buf[o + 8];
    if (typ == "IHDR") { w = be32(o + 8); h = be32(o + 12); bitDepth = d[8]; colorType = d[9]; interlace = d[12]; }
    else if (typ == "PLTE") plte.assign(d, d + len);
    else if (typ == "IDAT") idat.insert(idat.end(), d, d + len);
    else if (typ == "IEND") break;
    o += 12 + len;
  }
  if (!w || !h || bitDepth != 8 || interlace) throw std::runtime_error("Unsupported PNG (need 8-bit, non-interlaced): " + fileName);
  const int ch = colorType == 0 ? 1 : colorType == 2 ? 3 : colorType == 3 ? 1 : colorType == 4 ? 2 : 4;
  const size_t stride = size_t(w) * ch;
  std::vector<uint8_t> raw((stride + 1) * h);
  uLongf rawLen = raw.size();
  if (uncompress(raw.data(), &rawLen, idat.data(), idat.size()) != Z_OK || rawLen != raw.size()) throw std::runtime_error("PNG inflate failed: " + fileName);
  std::vector<uint8_t> pix(stride * h);
  for (uint32_t y = 0; y < h; ++y) {
    const uint8_t ft = raw[y * (stride + 1)]; const uint8_t* s = &raw[y * (stride + 1) + 1];
    uint8_t* d = &pix[y * stride]; const uint8_t* up = y ? &pix[(y - 1) * stride] : nullptr;
    for (size_t i = 0; i < stride; ++i) {
      const int a = i >= size_t(ch) ? d[i - ch] : 0, b = up ? up[i] : 0, c = (up && i >= size_t(ch)) ? up[i - ch] : 0;
      int v = s[i];
      switch (ft) {
        case 1: v += a; break; case 2: v += b; break; case 3: v += (a + b) / 2; break;
        case 4: { const int p = a + b - c, pa = std::abs(p - a), pb = std::abs(p - b), pc = std::abs(p - c); v += (pa <= pb && pa <= pc) ? a : (pb <= pc ? b : c); break; }
        default: break;
      }
      d[i] = uint8_t(v);
    }
  }
  out.create(int(h), int(w), cvMakeType(CV_8U, grayscale ? 1 : 3));
  for (size_t i = 0; i < size_t(w) * h; ++i) {
    int r, g, b;
    const uint8_t* p = &pix[i * ch];
    if (colorType == 0 || colorType == 4) r = g = b = p[0];
    else if (colorType == 3) { r = plte[p[0] * 3]; g = plte[p[0] * 3 + 1]; b = plte[p[0] * 3 + 2]; }
    else { r = p[0]; g = p[1]; b = p[2]; }
    if (grayscale) out.data[i] = (colorType == 0 || colorType == 4) ? uint8_t(r) : uint8_t((r * 4899 + g * 9617 + b * 1868 + 8192) >> 14);
    else { out.data[i * 3] = uint8_t(b); out.data[i * 3 + 1] = uint8_t(g); out.data[i * 3 + 2] = uint8_t(r); }
  }
  return out;
}

// --- FrameRange ---
static std::vector<std::string> explode(const std::string& s, char sep) {
  std::vector<std::string> out; std::string cur; std::istringstream is(s);
  while (std::getline(is, cur, sep)) out.push_back(cur);
  return out;
}
static void trim(std::string& s) {
  const size_t a = s.find_first_not_of(" \t"), b = s.find_last_not_of(" \t");
  s = (a == std::string::npos) ? "" : s.substr(a, b - a + 1);
}
void FrameRange::fromString(const std::string& str) {
  frames.clear();
  for (const std::string& piece : explode(str, ',')) {
    std::vector<std::string> sub = explode(piece, '-');
    if (sub.size() < 1 || sub.size() > 2) throw std::runtime_error("Malformed range piece.");
    const int start = std::stoi(sub[0]); const int end = sub.size() > 1 ? std::stoi(sub[1]) : start;
    for (int f = start; f <= end; ++f) frames.insert(f);
  }
}
std::string FrameRange::toString() const {
  if (isEmpty()) return "";
  std::string res; auto it = frames.begin(); int start = *it, last = start; ++it;
  auto add = [&]() { if (!res.empty()) res += ","; res += (last == start) ? std::to_string(start) : std::to_string(start) + "-" + std::to_string(last); };
  for (; it != frames.end(); ++it) { if (*it - last > 1) { add(); start = *it; } last = *it; }
  add();
  return res;
}
void FrameRange::resolve(int numFrames, bool clip) {
  if (clip) { std::set<int> c; for (int f : frames) if (f >= 0 && f < numFrames) c.insert(f); frames = c; }
  if (frames.empty()) for (int f = 0; f < numFrames; ++f) frames.insert(f);
  if (firstFrame() < 0 || lastFrame() >= numFrames) throw std::runtime_error("Frame range contains out-of-range frame indices.");
}
void FrameRange::checkEmpty() const { if (frames.empty()) throw std::runtime_error("Frame range is empty."); }
int FrameRange::firstFrame() const { checkEmpty(); return *frames.begin(); }
int FrameRange::lastFrame() const { checkEmpty(); return *frames.rbegin(); }
bool FrameRange::isConsecutive() const { return (lastFrame() - firstFrame() + 1) == int(frames.size()); }

// --- XformDescriptor (lib/DepthMapTransform.cpp:106-265) ---
static const char* kValueStr[] = {"None", "Scale", "ScaleShift"};
static const char* kDepthStr[] = {"None", "Identity", "Global", "Grid"};
static const char* kSpatialStr[] = {"None", "Identity", "VerticalLinear", "CornersBilinear", "BilinearGrid", "BicubicGrid"};
template <class E, size_t N> static void parseEnum(E& out, const std::string& s, const char* (&tab)[N]) {
  for (size_t i = 0; i < N; ++i) if (s == tab[i]) { out = E(int(i)); return; }
  throw std::runtime_error("Invalid enum value '" + s + "'.");
}
void XformDescriptor::reset(XformType t) {
  *this = XformDescriptor();
  if (t == XformType::Spatial) { type = XformType::Spatial; depthType = DepthXformType::None; spatialType = SpatialXformType::Identity; }
}
std::string XformDescriptor::str() const {
  std::string res; char b[160];
  if (type == XformType::Depth) {
    res = std::string(kDepthStr[int(depthType)]) + "(";
    switch (depthType) {
      case DepthXformType::Identity: break;
      case DepthXformType::Global: res += kValueStr[int(valueXform)]; break;
      case DepthXformType::Grid:
        if (gridSize[2] > 1) snprintf(b, sizeof(b), "%s, %s, %d, %d, %d, %f, %f", kValueStr[int(valueXform)], cubicInterpolation ? "Cubic" : "Linear", gridSize[0], gridSize[1], gridSize[2], depthMinMax[0], depthMinMax[1]);
        else snprintf(b, sizeof(b), "%s, %s, %d, %d, %d", kValueStr[int(valueXform)], cubicInterpolation ? "Cubic" : "Linear", gridSize[0], gridSize[1], gridSize[2]);
        res += b; break;
      default: throw std::runtime_error("Invalid depth transform type.");
    }
    res += ")";
  } else {
    res = kSpatialStr[int(spatialType)];
    if (spatialType == SpatialXformType::BilinearGrid || spatialType == SpatialXformType::BicubicGrid) { snprintf(b, sizeof(b), "(%d, %d)", gridSize[0], gridSize[1]); res += b; }
  }
  return res;
}
void XformDescriptor::parse(const std::string& s) {
  depthType = DepthXformType::None; spatialType = SpatialXformType::None;
  const size_t pos = s.find('(');
  const std::string typeStr = s.substr(0, pos);
  std::vector<std::string> args;
  auto getArgs = [&]() {
    if (pos == std::string::npos || s.empty() || s.back() != ')') throw std::runtime_error("Malformed descriptor string.");
    args = explode(s.substr(pos + 1, s.size() - 1 - (pos + 1)), ',');
    for (auto& a : args) trim(a);
  };
  auto checkNum = [&](size_t n) { if (args.size() != n) throw std::runtime_error("Incorrect number of parameters."); };
  if (type == XformType::Depth) {
    getArgs();
    if (typeStr == "BicubicGrid" || typeStr == "BilinearGrid") {   // backwards-compatibility form (:198-206)
      if (args.size() < 3) throw std::runtime_error("Incorrect number of parameters.");
      args = {args[0], typeStr == "BicubicGrid" ? "Cubic" : "Linear", args[1], args[2], "1"};
      depthType = DepthXformType::Grid;
    } else parseEnum(depthType, typeStr, kDepthStr);
    switch (depthType) {
      case DepthXformType::Identity: checkNum(0); break;
      case DepthXformType::Global: checkNum(1); parseEnum(valueXform, args[0], kValueStr); break;
      case DepthXformType::Grid:
        if (args.size() < 5) throw std::runtime_error("Incorrect number of parameters.");
        parseEnum(valueXform, args[0], kValueStr);
        if (args[1] == "Cubic") cubicInterpolation = true; else if (args[1] == "Linear") cubicInterpolation = false; else throw std::runtime_error("Invalid interpolation mode.");
        gridSize[0] = std::stoi(args[2]); gridSize[1] = std::stoi(args[3]); gridSize[2] = std::stoi(args[4]);
        if (gridSize[2] <= 1) checkNum(5); else { checkNum(7); depthMinMax[0] = std::stof(args[5]); depthMinMax[1] = std::stof(args[6]); }
        break;
      default: throw std::runtime_error("Invalid depth transform type.");
    }
  } else {
    parseEnum(spatialType, typeStr, kSpatialStr);
    if (spatialType == SpatialXformType::BilinearGrid || spatialType == SpatialXformType::BicubicGrid) { getArgs(); checkNum(2); gridSize[0] = std::stoi(args[0]); gridSize[1] = std::stoi(args[1]); }
  }
}

// --- Xform ---
void fillDepthConfig(const XformDescriptor& d, rcvd_config& cfg) {
  cfg.depth_type = int(d.depthType); cfg.value_xform = int(d.valueXform); cfg.depth_cubic = d.cubicInterpolation ? 1 : 0;
  cfg.depth_grid_x = d.gridSize[0]; cfg.depth_grid_y = d.gridSize[1];
}
void fillSpatialConfig(const XformDescriptor& d, rcvd_config& cfg) {
  cfg.spatial_type = int(d.spatialType); cfg.spatial_grid_x = d.gridSize[0]; cfg.spatial_grid_y = d.gridSize[1];
}
Xform::Xform(const XformDescriptor& desc) : desc_(desc) {
  if (desc.type == XformType::Depth) {
    const int k = valueParams();
    switch (desc.depthType) {
      case DepthXformType::Identity: break;
      case DepthXformType::Global: params_.assign(k, 1.0); break;   // lib/DepthMapTransform.cpp:531
      case DepthXformType::Grid: {
        const auto& g = desc.gridSize;
        if ((g[0] > 1 || g[1] > 1) && (g[0] < 2 || g[1] < 2)) throw std::runtime_error("Spatial grid transforms must have at least two rows and columns, respectively.");
        const int n = k * g[0] * g[1] * g[2];
        if (n <= 1) throw std::runtime_error("Grid transform cannot have an empty grid.");
        if (g[2] > 1) throw std::runtime_error("Bilateral (depth-wise) grids are not supported in this build.");
        params_.assign(n, 1.0); break; }   // :707
      default: throw std::runtime_error("Invalid depth transform type.");
    }
  } else {
    switch (desc.spatialType) {
      case SpatialXformType::Identity: break;
      case SpatialXformType::VerticalLinear: params_.assign(4, 0.0); break;
      case SpatialXformType::CornersBilinear: params_.assign(8, 0.0); break;
      case SpatialXformType::BilinearGrid: case SpatialXformType::BicubicGrid:
        if (desc.gridSize[0] < 2 || desc.gridSize[1] < 2) throw std::logic_error("Need at least two rows and columns in depth transform grid.");
        params_.assign(size_t(desc.gridSize[0]) * desc.gridSize[1] * 2, 0.0); break;
      default: throw std::runtime_error("Invalid spatial transform type.");
    }
  }
}
std::unique_ptr<Xform> Xform::clone() const { auto r = std::make_unique<Xform>(desc_); r->params_ = params_; return r; }
void Xform::copyFrom(const Xform& o) { if (o.desc_ != desc_) throw std::runtime_error("Can only copy parameters from same type of transform."); params_ = o.params_; }
std::string Xform::str() const {
  std::string res = desc_.str() + " ["; char b[64];
  for (size_t i = 0; i < params_.size(); ++i) { snprintf(b, sizeof(b), "%s%.2f", i ? ", " : "", params_[i]); res += b; }
  return res + "]";
}
void denseConfig(const XformDescriptor& d, rcvd_config& cfg) {
  memset(&cfg, 0, sizeof(cfg)); cfg.num_frames = 1; cfg.depth_type = RCVD_DEPTH_IDENTITY; cfg.value_xform = RCVD_VALUE_SCALE; cfg.spatial_type = RCVD_SPATIAL_IDENTITY;
  if (d.type == XformType::Depth) fillDepthConfig(d, cfg); else fillSpatialConfig(d, cfg);
  if (cfg.value_xform == RCVD_VALUE_NONE) cfg.value_xform = RCVD_VALUE_SCALE;
}
Image Xform::paramMap(const DepthFrame& df) const {
  if (desc_.type != XformType::Depth || desc_.depthType != DepthXformType::Grid) throw std::runtime_error("Parameter map not implemented for this transform type.");
  rcvd_config cfg; denseConfig(desc_, cfg);
  const int w = df.width(), h = df.height();
  Image out; out.create(h, w, cvMakeType(CV_64F, valueParams()));
  if (rcvd_depth_param_map(&cfg, currentDevice(), params_.data(), out.ptr<double>(), h, w) != RCVD_OK) throw std::runtime_error(rcvd_last_error());
  return out;
}
Image Xform::warp(int h, int w) const {
  if (desc_.type != XformType::Spatial) throw std::runtime_error("Transform has the wrong type.");
  rcvd_config cfg; denseConfig(desc_, cfg);
  Image out; out.create(h, w, cvMakeType(CV_32F, 2));
  if (rcvd_spatial_warp(&cfg, currentDevice(), params_.data(), out.ptr<float>(), h, w) != RCVD_OK) throw std::runtime_error(rcvd_last_error());
  return out;
}
Image Xform::apply(const Image& src) const {
  rcvd_config cfg; denseConfig(desc_, cfg);
  Image out; out.create(src.rows, src.cols, cvMakeType(CV_32F, 1));
  if (rcvd_depth_apply(&cfg, currentDevice(), params_.data(), src.ptr<float>(), out.ptr<float>(), src.rows, src.cols) != RCVD_OK) throw std::runtime_error(rcvd_last_error());
  return out;
}

// --- Intrinsics::resolveMissingFov (lib/DepthPhoto.cpp:114-158) ---
void Intrinsics::resolveMissingFov(float aspect) {
  bool vSet = vFov > 0, hSet = hFov > 0;
  if (vSet && hSet) return;
  if (aspect == 0) throw std::runtime_error("Aspect ratio must be non-zero.");
  const float kDefaultHFov = 0.508015513f, kDefaultVFov = 0.666488587f;
  const float defaultAspect = tanf(kDefaultHFov / 2.f) / tanf(kDefaultVFov / 2.f);
  if (!vSet && !hSet) { if (aspect > defaultAspect) { vFov = kDefaultVFov; vSet = true; } else { hFov = kDefaultHFov; hSet = true; } }
  if (vSet) { const float hh = std::tan(vFov / 2.0f); hFov = std::atan(hh * aspect) * 2.0f; }
  else if (hSet) { const float hw = std::tan(hFov / 2.0f); vFov = std::atan(hw / aspect) * 2.0f; }
}

// --- streams / frames ---
const Image* ColorFrame::image() {
  if (!loaded_) {
    loaded_ = true;
    const std::string fn = stream_.path() + "/frame_" + fmtInt6(index_) + stream_.extension();
    if (fileExists(fn)) {
      img_ = std::make_unique<Image>();
      if (stream_.extension() == ".raw") freadim(fn, *img_);
      else {
        Image u8 = imreadPng(fn, cvChannels(stream_.type()) == 1);
        if (u8.empty()) throw std::runtime_error("Could not read image '" + fn + "'.");
        if (cvDepth(stream_.type()) == CV_32F) {   // byte -> float: convertTo(.., 1/256) (lib/ColorStream.cpp:121-129)
          img_->create(u8.rows, u8.cols, stream_.type());
          float* d = img_->ptr<float>(); for (size_t i = 0; i < u8.data.size(); ++i) d[i] = u8.data[i] * (1.f / 256.f);
        } else *img_ = std::move(u8);
      }
      if (img_->type != stream_.type()) throw std::runtime_error("Image has incorrect type.");
      if (stream_.width_ < 0) { stream_.width_ = img_->cols; stream_.height_ = img_->rows; }
    }
  }
  return img_.get();
}
ColorFrame& ColorStream::frame(int i) { if (i < 0 || i >= int(frames_.size())) throw std::runtime_error("Frame index out of range."); return *frames_[i]; }
void ColorStream::setDir(const std::string& dir) { dir_ = dir; path_ = video_.path() + "/" + dir_; }
int ColorStream::width() { if (width_ < 0) { for (auto& f : frames_) if (f->image()) break; if (width_ < 0) width_ = height_ = 0; } return width_; }
int ColorStream::height() { width(); return height_; }

DepthFrame::DepthFrame(DepthVideo& v, DepthStream& s, int index) : video_(v), stream_(s), index_(index) { resetDepthXform(); resetSpatialXform(); }
void DepthFrame::resetDepthXform() { depthXform_ = std::make_unique<Xform>(stream_.depthXformDesc()); xformed_.reset(); }
void DepthFrame::resetSpatialXform() { spatialXform_ = std::make_unique<Xform>(stream_.spatialXformDesc()); }
int DepthFrame::width() const { return stream_.width(); }
int DepthFrame::height() const { return stream_.height(); }
float DepthFrame::invAspect() const { return video_.invAspect(); }
const Image* DepthFrame::sourceDepth() {
  if (!sourceLoaded_) {
    sourceLoaded_ = true;
    const std::string fn = stream_.path() + "/depth/frame_" + fmtInt6(index_) + ".raw";
    if (fileExists(fn)) {
      source_ = std::make_unique<Image>();
      freadim(fn, *source_);
      if (source_->type != cvMakeType(CV_32F, 1)) throw std::runtime_error("Depth image has incorrect type.");
      float* d = source_->ptr<float>();
      for (size_t i = 0; i < size_t(source_->rows) * source_->cols; ++i) d[i] = (std::isfinite(d[i]) && d[i] > 0.f) ? 1.f / d[i] : 0.f;   // lib/DepthStream.cpp:200-211
      if (stream_.width_ < 0) { stream_.width_ = source_->cols; stream_.height_ = source_->rows; }
      else if (stream_.width_ != source_->cols || stream_.height_ != source_->rows) throw std::runtime_error("Depth frame has inconsistent dimensions.");
    }
  }
  return (source_ && !source_->empty()) ? source_.get() : nullptr;
}
const Image* DepthFrame::depth() {
  // lib/DepthStream.cpp:275-291: the transformed depth is re-applied whenever the transform's descriptor or parameters differ from the
  // ones it was computed with (Python mutates transforms in place, e.g. depthXform().copyFrom(...), after depth() has been called)
  const Image* s = sourceDepth();
  if (!s) return nullptr;
  if (!xformed_ || depthXform_->desc() != appliedDesc_ || depthXform_->params() != appliedParams_) {
    appliedDesc_ = depthXform_->desc(); appliedParams_ = depthXform_->params();
    xformed_ = std::make_unique<Image>(depthXform_->apply(*s));
  }
  return xformed_.get();
}
void DepthFrame::setDepth(const Image& depth) {
  if (depth.type != cvMakeType(CV_32F, 1)) throw std::runtime_error("Depth image has incorrect type.");
  if (stream_.width_ < 0) { stream_.width_ = depth.cols; stream_.height_ = depth.rows; }
  else if (stream_.width_ != depth.cols || stream_.height_ != depth.rows) throw std::runtime_error("Depth frame has inconsistent dimensions.");
  source_ = std::make_unique<Image>(depth); sourceLoaded_ = true; xformed_.reset(); medianValid_ = false;
}
float DepthFrame::sourceDepthMedian() {
  if (!medianValid_) {
    const Image* d = sourceDepth();
    if (!d) throw std::runtime_error("Missing depth image.");
    std::vector<float> s(d->ptr<float>(), d->ptr<float>() + size_t(d->rows) * d->cols);
    std::nth_element(s.begin(), s.begin() + s.size() / 2, s.end());
    median_ = s[s.size() / 2]; medianValid_ = true;
  }
  return median_;
}
void DepthFrame::clear() { clearCache(); intrinsics = Intrinsics(); extrinsics = Extrinsics(); }
DepthFrame& DepthStream::frame(int i) { if (i < 0 || i >= int(frames_.size())) throw std::runtime_error("Frame index out of range."); return *frames_[i]; }
void DepthStream::setDir(const std::string& dir) { dir_ = dir; path_ = video_.path() + "/" + dir_; }
int DepthStream::width() { if (width_ < 0) { for (auto& f : frames_) if (f->sourceDepth()) break; if (width_ < 0) width_ = height_ = 0; } return width_; }
int DepthStream::height() { width(); return height_; }
void DepthStream::preloadSourceDepth(const std::vector<int>& frames, bool medians) {
  if (frames.empty()) return;
  auto one = [&](size_t i) { DepthFrame& f = frame(frames[i]); if (f.sourceDepth() && medians) f.sourceDepthMedian(); };
  one(0);
  parallelFor(frames.size() - 1, [&](size_t i) { one(i + 1); });
}
void DepthStream::resetDepthXforms(const XformDescriptor& desc) { depthXformDesc_ = desc; for (auto& f : frames_) f->resetDepthXform(); }
void DepthStream::resetSpatialXforms(const XformDescriptor& desc) { spatialXformDesc_ = desc; for (auto& f : frames_) f->resetSpatialXform(); }

// --- DepthVideo ---
void DepthVideo::init(const std::string& path, int width, int height, const std::vector<float>& pts) {
  colorStreams_.clear(); depthStreams_.clear();
  path_ = path; pts_ = pts; width_ = width; height_ = height;
  aspect_ = width / float(height); invAspect_ = 1.f / aspect_;
  duration_ = pts_.empty() ? 0.f : pts_.back() * pts_.size() / float(pts_.size() - 1);
}
bool DepthVideo::hasColorStream(const std::string& n) const { for (auto& s : colorStreams_) if (s->name_ == n) return true; return false; }
int DepthVideo::colorStreamIndex(const std::string& n) const { for (size_t i = 0; i < colorStreams_.size(); ++i) if (colorStreams_[i]->name_ == n) return int(i); throw std::runtime_error("Color stream '" + n + "' not found."); }
ColorStream& DepthVideo::colorStream(int i) { if (i < 0 || i >= numColorStreams()) throw std::runtime_error("Color stream index out of range."); return *colorStreams_[i]; }
void DepthVideo::createColorStream(const std::string& name, const std::string& dir, const std::string& ext, int type, std::pair<int, int> size) {
  if (type != cvMakeType(CV_8U, 1) && type != cvMakeType(CV_8U, 3) && type != cvMakeType(CV_32F, 1) && type != cvMakeType(CV_32F, 3))
    throw std::runtime_error("Color streams only support 1 or 3 channels and byte or float depth.");
  colorStreams_.push_back(std::make_unique<ColorStream>(*this));
  ColorStream& cs = *colorStreams_.back();
  cs.name_ = name; cs.setDir(dir); cs.extension_ = ext; cs.type_ = type; cs.width_ = size.first; cs.height_ = size.second;
  for (int f = 0; f < numFrames(); ++f) cs.frames_.push_back(std::make_unique<ColorFrame>(cs, f));
}
bool DepthVideo::hasDepthStream(const std::string& n) const { for (auto& s : depthStreams_) if (s->name_ == n) return true; return false; }
int DepthVideo::depthStreamIndex(const std::string& n) const { for (size_t i = 0; i < depthStreams_.size(); ++i) if (depthStreams_[i]->name_ == n) return int(i); throw std::runtime_error("Depth stream '" + n + "' not found."); }
DepthStream& DepthVideo::depthStream(int i) { if (i < 0 || i >= numDepthStreams()) throw std::runtime_error("Depth stream index out of range."); return *depthStreams_[i]; }
void DepthVideo::createDepthStream(const std::string& name, const std::string& dir, std::pair<int, int> size) {
  depthStreams_.push_back(std::make_unique<DepthStream>(*this));
  DepthStream& ds = *depthStreams_.back();
  ds.name_ = name; ds.setDir(dir); ds.depthXformDesc_.reset(); ds.spatialXformDesc_.reset(XformType::Spatial); ds.width_ = size.first; ds.height_ = size.second;
  for (int f = 0; f < numFrames(); ++f) { ds.frames_.push_back(std::make_unique<DepthFrame>(*this, ds, f)); ds.frames_.back()->intrinsics.resolveMissingFov(aspect_); }
}
void DepthVideo::printInfo() const {
  logInfo("Path: " + path_);
  char b[256]; snprintf(b, sizeof(b), "Dimensions: %d x %d (%f aspect ratio)", width_, height_, aspect_); logInfo(b);
  snprintf(b, sizeof(b), "Frame count: %d (%.2fs duration)", numFrames(), duration_); logInfo(b);
  logInfo("Color streams: " + std::to_string(numColorStreams()));
  for (auto& s : colorStreams_) logInfo("  '" + s->name_ + "' (dir '" + s->dir_ + "', extension '" + s->extension_ + "')");
  logInfo("Depth streams: " + std::to_string(numDepthStreams()));
  for (auto& s : depthStreams_) logInfo("  '" + s->name_ + "' (dir '" + s->dir_ + "', depth xform " + s->depthXformDesc_.str() + ", spatial xform " + s->spatialXformDesc_.str() + ")");
}
// video.dat, byte-compatible with the reference writer (lib/DepthVideo.cpp:300-385).
template <class T> static void wr(std::ostream& os, const T& v) { os.write(reinterpret_cast<const char*>(&v), sizeof(T)); }
static void wrstr(std::ostream& os, const std::string& s) { wr<uint64_t>(os, s.size()); os.write(s.data(), s.size()); }
static void wrXformDesc(std::ostream& os, const XformDescriptor& d) { wr<int32_t>(os, int32_t(d.type)); wrstr(os, d.str()); }
void DepthVideo::save() {
  std::ofstream os(path_ + "/video.dat", std::ios::binary);
  if (!os) throw std::runtime_error("Could not write video.dat.");
  wr<uint32_t>(os, 0xDEADBEEF); wr<uint32_t>(os, 13); wr<uint32_t>(os, 3);
  wr<int32_t>(os, numFrames()); for (float p : pts_) wr<float>(os, p);
  wr<int32_t>(os, numColorStreams());
  for (auto& cs : colorStreams_) { wrstr(os, cs->name_); wrstr(os, cs->dir_); wrstr(os, cs->extension_); wr<int32_t>(os, cs->type_); wr<int32_t>(os, cs->width_); wr<int32_t>(os, cs->height_); wr<bool>(os, false); }
  wr<int32_t>(os, numDepthStreams());
  for (auto& ds : depthStreams_) {
    wrstr(os, ds->name_); wrstr(os, ds->dir_); wrXformDesc(os, ds->depthXformDesc_); wrXformDesc(os, ds->spatialXformDesc_);
    wr<int32_t>(os, ds->width_); wr<int32_t>(os, ds->height_); wr<bool>(os, false);
    for (auto& f : ds->frames_) {
      wr<int32_t>(os, 0 /* Projection::Perspective */); wr<float>(os, f->intrinsics.vFov); wr<float>(os, f->intrinsics.hFov); wr<float>(os, f->intrinsics.centerLat); wr<float>(os, f->intrinsics.centerLon);
      wr<float>(os, f->extrinsics.position.x); wr<float>(os, f->extrinsics.position.y); wr<float>(os, f->extrinsics.position.z);
      wr<float>(os, f->extrinsics.orientation.x); wr<float>(os, f->extrinsics.orientation.y); wr<float>(os, f->extrinsics.orientation.z); wr<float>(os, f->extrinsics.orientation.w);
      wr<bool>(os, f->enabled);
      for (const Xform* x : {&f->depthXform(), &f->spatialXform()}) { wrXformDesc(os, x->desc()); os.write(reinterpret_cast<const char*>(x->params().data()), sizeof(double) * x->params().size()); }
    }
  }
  wr<float>(os, duration_); wr<int32_t>(os, width_); wr<int32_t>(os, height_); wr<float>(os, aspect_); wr<float>(os, invAspect_);
  wr<uint32_t>(os, 0xDEADBEEF);
}
// Reader for the file save() writes.  Note: the reference's own load() (lib/DepthVideo.cpp:120-298) does not consume the
// per-stream "has GOP table" byte that its save() emits (:329-332, :355-359 vs the commented-out reads at :191-197, :236-245),
// so it cannot re-read format-13 files; this reader follows the WRITER's layout.
template <class T> static T rd(std::istream& is) { T v{}; is.read(reinterpret_cast<char*>(&v), sizeof(T)); if (!is) throw std::runtime_error("Unexpected end of 'video.dat'."); return v; }
static std::string rdstr(std::istream& is) { const uint64_t n = rd<uint64_t>(is); if (n > (1u << 20)) throw std::runtime_error("Corrupt string in 'video.dat'."); std::string s(n, '\0'); is.read(s.data(), n); if (!is) throw std::runtime_error("Unexpected end of 'video.dat'."); return s; }
static XformDescriptor rdXformDesc(std::istream& is) { XformDescriptor d; d.type = XformType(rd<int32_t>(is)); const std::string str = rdstr(is); const XformType t = d.type; d.parse(str); d.type = t; return d; }
void DepthVideo::load(const std::string& path) {
  std::ifstream is(path + "/video.dat", std::ios::binary);
  if (!is) throw std::runtime_error("Could not find 'video.dat'.");
  if (rd<uint32_t>(is) != 0xDEADBEEF) throw std::runtime_error("Did not see magic marker at beginning of file.");
  const uint32_t fileFormat = rd<uint32_t>(is), dpFormat = rd<uint32_t>(is);
  if (fileFormat > 13) throw std::runtime_error("File format too new.");
  if (fileFormat < 13 || dpFormat != 3) throw std::runtime_error("File format too old.");   // only the current writer's format is supported here
  colorStreams_.clear(); depthStreams_.clear(); path_ = path;
  const int n = rd<int32_t>(is); if (n < 0 || n > (1 << 24)) throw std::runtime_error("Corrupt frame count in 'video.dat'.");
  pts_.resize(n); for (float& p : pts_) p = rd<float>(is);
  const int ncs = rd<int32_t>(is);
  for (int i = 0; i < ncs; ++i) {
    colorStreams_.push_back(std::make_unique<ColorStream>(*this));
    ColorStream& cs = *colorStreams_.back();
    cs.name_ = rdstr(is); cs.setDir(rdstr(is)); cs.extension_ = rdstr(is); cs.type_ = rd<int32_t>(is); cs.width_ = rd<int32_t>(is); cs.height_ = rd<int32_t>(is);
    if (rd<bool>(is)) throw std::runtime_error("GOP tables are not supported.");
    for (int f = 0; f < n; ++f) cs.frames_.push_back(std::make_unique<ColorFrame>(cs, f));
  }
  const int nds = rd<int32_t>(is);
  for (int i = 0; i < nds; ++i) {
    depthStreams_.push_back(std::make_unique<DepthStream>(*this));
    DepthStream& ds = *depthStreams_.back();
    ds.name_ = rdstr(is); ds.setDir(rdstr(is)); ds.depthXformDesc_ = rdXformDesc(is); ds.spatialXformDesc_ = rdXformDesc(is);
    ds.width_ = rd<int32_t>(is); ds.height_ = rd<int32_t>(is);
    if (rd<bool>(is)) throw std::runtime_error("GOP tables are not supported.");
    for (int f = 0; f < n; ++f) {
      ds.frames_.push_back(std::make_unique<DepthFrame>(*this, ds, f));
      DepthFrame& df = *ds.frames_.back();
      if (rd<int32_t>(is) != 0) throw std::runtime_error("Only perspective intrinsics are supported.");
      df.intrinsics.vFov = rd<float>(is); df.intrinsics.hFov = rd<float>(is); df.intrinsics.centerLat = rd<float>(is); df.intrinsics.centerLon = rd<float>(is);
      df.extrinsics.position.x = rd<float>(is); df.extrinsics.position.y = rd<float>(is); df.extrinsics.position.z = rd<float>(is);
      df.extrinsics.orientation.x = rd<float>(is); df.extrinsics.orientation.y = rd<float>(is); df.extrinsics.orientation.z = rd<float>(is); df.extrinsics.orientation.w = rd<float>(is);
      df.enabled = rd<bool>(is);
      for (int k = 0; k < 2; ++k) {
        const XformDescriptor d = rdXformDesc(is);
        if (k == 0 && d != ds.depthXformDesc_) throw std::runtime_error("Inconsistent depth transform.");
        Xform& x = k == 0 ? df.depthXform() : df.spatialXform();
        if (d != x.desc()) throw std::runtime_error("Inconsistent spatial transform.");
        is.read(reinterpret_cast<char*>(x.params().data()), sizeof(double) * x.params().size());
        if (!is) throw std::runtime_error("Unexpected end of 'video.dat'.");
      }
    }
  }
  duration_ = rd<float>(is); width_ = rd<int32_t>(is); height_ = rd<int32_t>(is); aspect_ = rd<float>(is); invAspect_ = rd<float>(is);
  if (rd<uint32_t>(is) != 0xDEADBEEF) throw std::runtime_error("Did not see magic marker at end of file.");
}
void DepthVideo::saveDepth(int stream) {
  DepthStream& ds = depthStream(stream);
  for (int f = 0; f < numFrames(); ++f) {
    const std::string fn = ds.path() + "/depth/frame_" + fmtInt6(f) + ".raw";
    const Image* d = ds.frame(f).depth();
    if (d) {
      Image disp; disp.create(d->rows, d->cols, cvMakeType(CV_32F, 1));
      const float* s = d->ptr<float>(); float* o = disp.ptr<float>();
      for (size_t i = 0; i < size_t(d->rows) * d->cols; ++i) o[i] = (std::isfinite(s[i]) && s[i] > 0.f) ? 1.f / s[i] : 0.f;   // invalid depth -> 0 (:611-618)
      makeDirs(ds.path() + "/depth");
      fwriteim(fn, disp);
    } else if (fileExists(fn)) {
      std::remove(fn.c_str());
    }
  }
}
void importVideo(DepthVideo& video, const std::string& path, bool discoverStreams) {
  logInfo("Importing 3D video '" + path + "'...");
  std::ifstream is(path + "/frames.txt", std::ios::binary);
  if (is.fail()) throw std::runtime_error("Could not open frame file.");
  int n = -1, w = -1, h = -1; is >> n >> w >> h;
  if (n <= 0) throw std::runtime_error("Invalid frame file.");
  std::vector<float> pts(n); float minPts = 0.f;
  for (int i = 0; i < n; ++i) {
    float p; is >> p; if (i == 0) minPts = p; p -= minPts;
    if (i > 0 && p <= pts[i - 1]) throw std::runtime_error("Non-monotonic PTS detected.");
    pts[i] = p;
  }
  video.init(path, w, h, pts);
  if (discoverStreams) throw std::runtime_error("Stream discovery is not supported in this build (pose_optimization.py passes discoverStreams=False).");
}

// --- pose conversions (lib/PoseOptimizer.cpp:769-781, :968-974) ---
void quatToAngleAxis(const Quatf& qf, double aa[3]) {
  const double qx = qf.x, qy = qf.y, qz = qf.z, qw = qf.w;
  auto rot = [&](double vx, double vy, double vz, double o[3]) {   // Eigen quaternion * vector in double
    double ux = qy * vz - qz * vy, uy = qz * vx - qx * vz, uz = qx * vy - qy * vx; ux += ux; uy += uy; uz += uz;
    o[0] = vx + qw * ux + (qy * uz - qz * uy); o[1] = vy + qw * uy + (qz * ux - qx * uz); o[2] = vz + qw * uz + (qx * uy - qy * ux);
  };
  double right[3], up[3], front[3]; rot(1, 0, 0, right); rot(0, 1, 0, up); rot(-0.0, -0.0, -1, front);
  // rotation.col(0) = right, col(1) = up, col(2) = -front ; R(i,j) = col j, row i
  double R[3][3]; for (int i = 0; i < 3; ++i) { R[i][0] = right[i]; R[i][1] = up[i]; R[i][2] = -front[i]; }
  // ceres::RotationMatrixToQuaternion
  double q[4]; const double trace = R[0][0] + R[1][1] + R[2][2];
  if (trace >= 0.0) { double t = std::sqrt(trace + 1.0); q[0] = 0.5 * t; t = 0.5 / t; q[1] = (R[2][1] - R[1][2]) * t; q[2] = (R[0][2] - R[2][0]) * t; q[3] = (R[1][0] - R[0][1]) * t; }
  else {
    int i = 0; if (R[1][1] > R[0][0]) i = 1; if (R[2][2] > R[i][i]) i = 2; const int j = (i + 1) % 3, k = (j + 1) % 3;
    double t = std::sqrt(R[i][i] - R[j][j] - R[k][k] + 1.0); q[i + 1] = 0.5 * t; t = 0.5 / t;
    q[0] = (R[k][j] - R[j][k]) * t; q[j + 1] = (R[j][i] + R[i][j]) * t; q[k + 1] = (R[k][i] + R[i][k]) * t;
  }
  // ceres::QuaternionToAngleAxis
  const double s2 = q[1] * q[1] + q[2] * q[2] + q[3] * q[3];
  if (s2 > 0.0) {
    const double s = std::sqrt(s2), c = q[0];
    const double two_theta = 2.0 * ((c < 0.0) ? std::atan2(-s, -c) : std::atan2(s, c));
    const double k = two_theta / s; aa[0] = q[1] * k; aa[1] = q[2] * k; aa[2] = q[3] * k;
  } else { aa[0] = q[1] * 2.0; aa[1] = q[2] * 2.0; aa[2] = q[3] * 2.0; }
}
Quatf angleAxisToQuat(const double aa[3]) {
  double R[3][3];   // R[i][j]: row i, column j  (ceres::AngleAxisToRotationMatrix, column-major adapter)
  const double th2 = aa[0] * aa[0] + aa[1] * aa[1] + aa[2] * aa[2];
  if (th2 > std::numeric_limits<double>::epsilon()) {
    const double th = std::sqrt(th2), wx = aa[0] / th, wy = aa[1] / th, wz = aa[2] / th, c = std::cos(th), s = std::sin(th);
    R[0][0] = c + wx * wx * (1.0 - c); R[1][0] = wz * s + wx * wy * (1.0 - c); R[2][0] = -wy * s + wx * wz * (1.0 - c);
    R[0][1] = wx * wy * (1.0 - c) - wz * s; R[1][1] = c + wy * wy * (1.0 - c); R[2][1] = wx * s + wy * wz * (1.0 - c);
    R[0][2] = wy * s + wx * wz * (1.0 - c); R[1][2] = -wx * s + wy * wz * (1.0 - c); R[2][2] = c + wz * wz * (1.0 - c);
  } else {
    R[0][0] = 1; R[1][0] = aa[2]; R[2][0] = -aa[1]; R[0][1] = -aa[2]; R[1][1] = 1; R[2][1] = aa[0]; R[0][2] = aa[1]; R[1][2] = -aa[0]; R[2][2] = 1;
  }
  // Eigen::Quaterniond(Matrix3d)
  double q[4] /* x y z w */; double t = R[0][0] + R[1][1] + R[2][2];
  if (t > 0.0) { t = std::sqrt(t + 1.0); q[3] = 0.5 * t; t = 0.5 / t; q[0] = (R[2][1] - R[1][2]) * t; q[1] = (R[0][2] - R[2][0]) * t; q[2] = (R[1][0] - R[0][1]) * t; }
  else {
    int i = 0; if (R[1][1] > R[0][0]) i = 1; if (R[2][2] > R[i][i]) i = 2; const int j = (i + 1) % 3, k = (j + 1) % 3;
    t = std::sqrt(R[i][i] - R[j][j] - R[k][k] + 1.0); q[i] = 0.5 * t; t = 0.5 / t; q[3] = (R[k][j] - R[j][k]) * t; q[j] = (R[j][i] + R[i][j]) * t; q[k] = (R[k][i] + R[i][k]) * t;
  }
  Quatf o; o.x = float(q[0]); o.y = float(q[1]); o.z = float(q[2]); o.w = float(q[3]); return o;
}

}  // namespace rcvdh
