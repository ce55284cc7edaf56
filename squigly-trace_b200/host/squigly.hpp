// squigly.hpp -- host side of the B200 backend, mirroring the reference's module interfaces.
//
// north_star keeps the host in Haskell (Obj.hs, BIH.hs, Main.hs unchanged, `foreign import ccall` into
// include/sqt.h).  This image has no GHC, so the host is written here in C++ with the reference's own
// names, argument meaning and error behaviour, on top of the same C ABI the Haskell binding would use
// (INTEGRATION.md shows that binding).  Everything in this directory is host logic: parsing, BIH build,
// flattening, PNG output, CLI.  All per-ray / per-sample work is behind sqt_render / sqt_intersect_batch.
#pragma once
#include <cstdint>
#include <memory>
#include <optional>
#include <stdexcept>
#include <string>
#include <utility>
#include <vector>

#include "../../include/sqt.h"

namespace squigly {

// V3.hs:5
struct V3 { float x = 0, y = 0, z = 0; };
// Color.hs:78-83
struct Material { float reflective = 0; V3 surfColor; float emissive = 0; V3 emitColor; };
// Geometry.hs:49-54 (the material is referenced by its index in the .sq file)
struct Triangle { V3 tFirst, tSecond, tThird; uint32_t material = 0; };
// Geometry.hs:44-47
struct Ray { V3 vertex, direction; };
// Geometry.hs:71-75 ; `surface` is the index of the triangle in the parsed list
struct Intersection { V3 intersectPoint; float dist = 0; int32_t surface = -1; };
// Geometry.hs:153
struct Bounds { V3 lo, hi; };
// Geometry.hs:41
struct Camera { V3 position; float rotation[9] = {1, 0, 0, 0, 1, 0, 0, 0, 1}; };
enum class Axis : uint32_t { X = 0, Y = 1, Z = 2 };

// ---- Obj.hs -----------------------------------------------------------------------------------
struct ParsedScene { std::vector<Triangle> triangles; std::vector<Material> materials; };
// trisFromObj :: Bool -> String -> IO [Triangle]   (Obj.hs:49-58).  dataDir stands for the literal "./data/".
ParsedScene trisFromObj(bool debug, const std::string &objContents, const std::string &dataDir = "./data/");
// loadCamera :: FilePath -> IO Camera   (Obj.hs:60-65); throws "Failed to parse /data/camera" like the reference
Camera loadCamera(const std::string &path);
// rotMatrixRads (Geometry.hs:90-102), row-major
void rotMatrixRads(float alp, float bet, float gam, float out[9]);
std::string readFile(const std::string &path);

// ---- BIH.hs -----------------------------------------------------------------------------------
// Tree BIHNode (Vector Triangle) (BIH.hs:26,37-39) in arrays; node 0 is the root, pre-order.
struct BIHTreeNode {
    bool leaf = false;
    Axis axis = Axis::X; float lmax = 0, rmin = 0; uint32_t left = 0, right = 0;   // Branch (BIHN axis lmax rmin) l r
    uint32_t first = 0, count = 0;                                                 // Leaf: range of `order`
};
struct BIH {
    Bounds bounds;                       // BIH.hs:41
    std::vector<BIHTreeNode> tree;       // BIH.hs:42
    std::vector<uint32_t> order;         // `flatten` (BIH.hs:50-52): triangle indices, leaf by leaf
    std::vector<Triangle> triangles;     // the parsed list the indices refer to
    std::vector<Material> materials;
};
BIH makeBIH(ParsedScene scene);                      // BIH.hs:62-65
int height(const BIH &b);                            // BIH.hs:46-48
int numLeaves(const BIH &b);                         // BIH.hs:54-56
int longestLeaf(const BIH &b);                       // BIH.hs:58-60
std::string showBIH(const BIH &b);                   // `show bih` stand-in for --debug (Main.hs:68-70)

// The structure-of-arrays the C ABI takes (include/sqt.h): 16-byte nodes, 48-byte triangles in leaf order.
struct FlatBIH {
    float root_bounds[6];
    std::vector<sqt_node> nodes;
    std::vector<sqt_tri> tris;
    std::vector<sqt_material> mats;
    sqt_scene_desc desc() const;
};
FlatBIH flattenForDevice(const BIH &b);

// ---- Geometry.hs:62-65 ------------------------------------------------------------------------
// data Scene a = Scene { geometry :: a, intersect :: a -> Ray -> Maybe Intersection }
// The device-backed plug-in keeps the record shape; `intersect` is batched because one FFI call per ray
// would be absurd, and the single-ray form is the batch of one.
class DeviceBIH;   // geometry uploaded to one or more B200s
struct SceneBIH {
    std::shared_ptr<DeviceBIH> geometry;
    std::vector<std::optional<Intersection>> (*intersectBatch)(const DeviceBIH &, const std::vector<Ray> &);
    std::optional<Intersection> intersect(const Ray &r) const;
};
SceneBIH sceneFromBIH(const BIH &bih, int nGpus = 1);     // Main.hs:55-56

// ---- Lib.hs -----------------------------------------------------------------------------------
// Settings (Lib.hs:54-63) plus the two knobs north_star adds
struct Settings {
    int samples = 10;
    std::pair<int, int> dimensions{540, 540};
    std::string savePath = "./render/result.png";
    std::string objPath = "./data/scene.obj";
    std::string cameraPath = "./data/camera";
    bool debug = false;
    std::string debugPath;
    bool cast = false;
    // extensions (not in the reference)
    int bounces = 3;            // Lib.hs:129 hard-codes 3
    int gpus = 1;
    bool corrected = false;     // false = Lib.hs:69-85 index convention verbatim (SURVEY A.5)
    uint64_t seed = 0;
    int progress = 0;           // > 0: render in chunks of this many samples, writing a preview after each
    bool adaptive = false;      // with progress: retire converged pixels after every chunk (sqt_render_retire)
    float adaptiveRel = 0.0f, adaptiveAbs = 0.0f;
    int adaptiveMin = 16;
    int denoise = -1;           // with progress: >= 0 also writes <stem>-denoised.png after every chunk (sqt_denoise levels)
    bool aa = false;            // box-filtered pixels (sqt_set_lens jitter)
    float aperture = 0.0f, focus = 0.0f;    // --lens=APERTURE,FOCUS (focus > 0: a thin lens is set)
};
struct RenderReport { sqt_stats stats{}; int rows = 0, cols = 0; };
// render :: Scene a -> Camera -> Settings -> IO ()   (Lib.hs:68-75): computes the image on the device(s) and writes it
RenderReport render(const SceneBIH &scene, const Camera &cam, const Settings &settings);
// the same without writeImage, for callers that want the pixels
RenderReport renderToBuffer(const SceneBIH &scene, const Camera &cam, const Settings &settings,
                            std::vector<uint8_t> &rgb8, std::vector<float> *accum);
sqt_render_params paramsFromSettings(const Settings &s);

// ---- massiv-io writeImage stand-in (Lib.hs:75): PNG by extension --------------------------------
void writeImage(const std::string &path, const uint8_t *rgb8, int rows, int cols);

}  // namespace squigly
