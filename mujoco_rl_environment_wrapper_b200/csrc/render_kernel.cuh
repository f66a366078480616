// render_kernel.cuh — agent cameras (SURVEY 8 f4; reference: MuJoCo_Gym/mujoco_parent.py:496-575,
// `get_camera_data` -> mjv_updateScene + mjr_render + mjr_readPixels on an off-screen GLFW window).
//
// The reference rasterises with MuJoCo's OpenGL renderer; here every pixel is a primary ray against the
// env's primitive geoms (the same ray / geom routines the rangefinder uses), shaded with a two-sided
// head-light:  rgb = clamp(geom_rgba.rgb, 0, 1) * (RENDER_AMBIENT + RENDER_DIFFUSE * |n . d|), black where
// nothing is hit, 8 bits per channel, rows bottom-up like glReadPixels.  Lights, materials, textures,
// shadows and fog of the OpenGL pipeline are not modelled (pixel parity with the reference is not claimed;
// the CPU oracle restates exactly this image formation in fp64).
//
// One CTA per env: warp 0 redoes the kinematics pass from the env's qpos, the CTA flattens the geoms into a
// broadcast-friendly list in shared memory and culls them per 16 x 8 pixel tile (bounding sphere against the
// tile's view cone, conservative, so the image is unchanged), then one warp shades one tile: every lane takes
// 4 neighbouring pixels, walks the tile's short geom list (warp-uniform) and writes three 32-bit words.
#pragma once
#include "step_kernel.cuh"

namespace mjb {

#define RENDER_AMBIENT 0.4f
#define RENDER_DIFFUSE 0.6f
#define RENDER_MAX_CAMS 8

struct RenderCams { int n; int id[RENDER_MAX_CAMS]; };

// ---- ray tests in the geom's local frame (lp = R^T (o - pos) is shared by all rays of a camera, lv = R^T d) ------
// Same first non-negative crossing as ray_geom (step_kernel.cuh) / the oracle; boxes by slabs instead of face by
// face (a third of the instructions; arena walls and target boxes are what most camera rays test).
MJB_DEV float ray_local(int type, const float* size, f3 lp, f3 lv) {
  if (type == MJB_GEOM_PLANE) {
    if (lv.z > -MJB_MINVAL) return -1.f;
    float x = -lp.z / lv.z;
    if (x < 0) return -1.f;
    float p0 = lp.x + x * lv.x, p1 = lp.y + x * lv.y;
    return ((size[0] <= 0 || fabsf(p0) <= size[0]) && (size[1] <= 0 || fabsf(p1) <= size[1])) ? x : -1.f;
  }
  if (type == MJB_GEOM_SPHERE) {   // lv is a unit vector
    float b = dot(lv, lp), det = b * b - (dot(lp, lp) - size[0] * size[0]);
    if (det < 0) return -1.f;
    float sq = sqrtf(det), x0 = -b - sq, x1 = -b + sq;
    return x0 >= 0 ? x0 : (x1 >= 0 ? x1 : -1.f);
  }
  if (type == MJB_GEOM_BOX) {
    float tn = -MJB_BIG, tf = MJB_BIG;
#pragma unroll
    for (int a = 0; a < 3; a++) {
      const float p = comp(lp, a), v = comp(lv, a), s = size[a];
      if (fabsf(v) < MJB_MINVAL) {
        if (fabsf(p) > s) return -1.f;
      } else {
        const float inv = 1.f / v, t1 = (-s - p) * inv, t2 = (s - p) * inv;
        tn = fmaxf(tn, fminf(t1, t2));
        tf = fminf(tf, fmaxf(t1, t2));
      }
    }
    if (tn > tf || tf < 0.f) return -1.f;
    return tn >= 0.f ? tn : tf;
  }
  // capsule: cylinder side, then the two end spheres
  float best = -1.f;
  const float r = size[0], h = size[1];
  float x[2];
  if (quad_roots(lv.x * lv.x + lv.y * lv.y, lp.x * lv.x + lp.y * lv.y, lp.x * lp.x + lp.y * lp.y - r * r, x))
    for (int i = 0; i < 2; i++)
      if (fabsf(lp.z + x[i] * lv.z) <= h && x[i] >= 0 && (best < 0 || x[i] < best)) best = x[i];
  for (int sg = -1; sg <= 1; sg += 2) {
    f3 d = lp - mk3(0, 0, sg * h);
    if (quad_roots(dot(lv, lv), dot(lv, d), dot(d, d) - r * r, x))
      for (int i = 0; i < 2; i++)
        if (sg * (lp.z + x[i] * lv.z) >= h && x[i] >= 0 && (best < 0 || x[i] < best)) best = x[i];
  }
  return best;
}

// |normal . direction| at the hit, in the geom's local frame
MJB_DEV float hit_cosine(int type, const float* size, f3 lp, f3 lv, float t) {
  if (type == MJB_GEOM_PLANE) return fabsf(lv.z);
  f3 p = lp + lv * t;
  if (type == MJB_GEOM_SPHERE) return fabsf(dot(p, lv)) * MJB_RSQRT(fmaxf(dot(p, p), 1e-20f));
  if (type == MJB_GEOM_CAPSULE) {
    f3 n = mk3(p.x, p.y, p.z - fminf(fmaxf(p.z, -size[1]), size[1]));
    return fabsf(dot(n, lv)) * MJB_RSQRT(fmaxf(dot(n, n), 1e-20f));
  }
  float ax = fabsf(p.x) / size[0], ay = fabsf(p.y) / size[1], az = fabsf(p.z) / size[2];   // box: the face reached
  return (ax >= ay && ax >= az) ? fabsf(lv.x) : (ay >= az ? fabsf(lv.y) : fabsf(lv.z));
}

// colours of the first geom along 4 rays that share the origin `o` (unit directions d[4]); geom-outer loop: one
// geom record load and one local origin serve all four rays.  Packed 0x00BBGGRR each.
MJB_DEV_NOINLINE void shade_rays4(const float* GL, const uint16_t* list, int nlist, f3 o, const f3* d, uint32_t* col) {
  float best[4] = {MJB_BIG, MJB_BIG, MJB_BIG, MJB_BIG};
  int bi[4] = {-1, -1, -1, -1};
  MJB_NOUNROLL
  for (int i = 0; i < nlist; i++) {   // ascending geom ids: ties resolve as in the oracle's loop
    const int g = list[i];
    const float* G = GL + g * GL_STRIDE;
    const int type = __float_as_int(G[GL_TYPE]);
    const f3 oc = ld3(G + GL_POS) - o;
    const float l2 = dot(oc, oc), rb = G[GL_RBOUND], rb2 = rb * rb;
    const bool inside = l2 <= rb2 || type == MJB_GEOM_PLANE;   // no bounding-sphere rejection possible
    float R[9];
#pragma unroll
    for (int k = 0; k < 9; k++) R[k] = G[GL_MAT + k];
    const f3 lp = type == MJB_GEOM_SPHERE ? oc * -1.f : mulTv(R, oc * -1.f);   // spheres stay in world axes
#pragma unroll
    for (int j = 0; j < 4; j++) {
      if (!inside) {
        float tca = dot(oc, d[j]);
        if (tca < 0.f || l2 - tca * tca > rb2 || tca - rb > best[j]) continue;
      }
      float t = ray_local(type, G + GL_SIZE, lp, type == MJB_GEOM_SPHERE ? d[j] : mulTv(R, d[j]));
      if (t >= 0.f && t < best[j]) { best[j] = t; bi[j] = g; }
    }
  }
#pragma unroll
  for (int j = 0; j < 4; j++) {
    if (bi[j] < 0) { col[j] = 0u; continue; }
    const float* G = GL + bi[j] * GL_STRIDE;
    const int type = __float_as_int(G[GL_TYPE]);
    const f3 lp = mulTv(G + GL_MAT, o - ld3(G + GL_POS)), lv = mulTv(G + GL_MAT, d[j]);
    const float I = RENDER_AMBIENT + RENDER_DIFFUSE * fminf(hit_cosine(type, G + GL_SIZE, lp, lv, best[j]), 1.f);
    uint32_t r = (uint32_t)(G[GL_RGB] * I * 255.f + 0.5f), gg = (uint32_t)(G[GL_RGB + 1] * I * 255.f + 0.5f),
             bb = (uint32_t)(G[GL_RGB + 2] * I * 255.f + 0.5f);
    col[j] = r | (gg << 8) | (bb << 16);
  }
}

#if !defined(MJB_HOST_EMU)
#define RENDER_TILE_W 16
#define RENDER_TILE_H 8
#define RENDER_TILE_BATCH 128   // tiles whose geom lists are resident at once

// direction of the ray through image-plane point (fx, fy) in pixels (pixel centres are at +0.5)
MJB_DEV f3 pixel_dir(const float* cw, float th, float fx, float fy, int width, int height) {
  float u = (fx / width * 2.f - 1.f) * th * ((float)width / (float)height), v = (fy / height * 2.f - 1.f) * th;
  f3 dl = mk3(u, v, -1.f);   // camera frame: looks along -z, +y up
  return mulv(cw + 3, dl * MJB_RSQRT(dot(dl, dl)));
}

// out: u8 [num_envs, cams.n, height, width, 3]
__global__ void __launch_bounds__(256) k_render(const __grid_constant__ DevModel dm, const uint32_t* __restrict__ image,
                                                const RenderHdr rh, const uint32_t* __restrict__ rtab,
                                                const float* __restrict__ qpos_g, int num_envs, const RenderCams cams, int width,
                                                int height, uint8_t* __restrict__ out) {
  extern __shared__ __align__(128) uint32_t smem[];
  uint32_t* img = smem;
  float* scratch = reinterpret_cast<float*>(img + dm.image_words);
  uint32_t* tab = reinterpret_cast<uint32_t*>(scratch + dm.env_words);
  float* GL = reinterpret_cast<float*>(tab + rh.words);
  float* CW = GL + dm.ngeom * GL_STRIDE;   // per requested camera: world pos[3], rotation[9]
  const int lstride = (dm.ngeom + 2) & ~1;  // u16 per tile: count, then geom ids
  uint16_t* TL = reinterpret_cast<uint16_t*>(CW + 12 * RENDER_MAX_CAMS);
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nwarps = blockDim.x >> 5;
  for (int i = tid; i < dm.image_words; i += blockDim.x) img[i] = image[i];
  for (int i = tid; i < rh.words; i += blockDim.x) tab[i] = rtab[i];
  __syncthreads();
  Ctx c{&dm, img, scratch, lane, nullptr, 0};
  const float* rgba = reinterpret_cast<const float*>(tab + rh.off_rgba);
  const int tiles_x = (width + RENDER_TILE_W - 1) / RENDER_TILE_W, tiles_y = (height + RENDER_TILE_H - 1) / RENDER_TILE_H;
  const int tiles_cam = tiles_x * tiles_y, ntiles = tiles_cam * cams.n;
  const bool words = (width & 3) == 0;   // 4-pixel groups never straddle the right edge: 12-byte stores
  for (int env = blockIdx.x; env < num_envs; env += gridDim.x) {
    if (tid < 32) {
      float* qpos = SF(qpos);
      for (int i = lane; i < dm.nq; i += 32) qpos[i] = qpos_g[(size_t)env * dm.qpos_stride + i];
      __syncwarp();
      fk(c);
    }
    __syncthreads();
    for (int g = tid; g < dm.ngeom; g += blockDim.x) {
      GeomW w = geom_world(c, g);
      float* G = GL + g * GL_STRIDE;
      st3(G + GL_POS, w.pos);
      for (int i = 0; i < 9; i++) G[GL_MAT + i] = w.mat[i];
      for (int i = 0; i < 3; i++) { G[GL_SIZE + i] = w.size[i]; G[GL_RGB + i] = rgba[4 * g + i]; }
      G[GL_TYPE] = __int_as_float(rgba[4 * g + 3] > 0.f ? w.type : -1);   // alpha == 0: invisible
      G[GL_RBOUND] = CF(geom_rbound)[g];
    }
    for (int k = tid; k < cams.n; k += blockDim.x) {
      const uint32_t* cr = tab + rh.off_cam + cams.id[k] * CAM_STRIDE;
      const float* cf = reinterpret_cast<const float*>(cr);
      int mb = (int)cr[CAM_MB];
      f3 p = ld3(cf + CAM_POS);
      q4 q = ldq(cf + CAM_QUAT);
      if (mb >= 0) { p = ld3(SF(xpos) + 3 * mb) + mulv(SF(xmat) + 9 * mb, p); q = qmul(ldq(SF(xquat) + 4 * mb), q); }
      st3(CW + 12 * k, p);
      q2m(q, CW + 12 * k + 3);
    }
    __syncthreads();
    for (int t0 = 0; t0 < ntiles; t0 += RENDER_TILE_BATCH) {
      const int nb = min(RENDER_TILE_BATCH, ntiles - t0);
      // (1) per tile: the geoms whose bounding sphere reaches into the tile's view cone.  f(p) = |p_perp| cos(a)
      //     - p_axis sin(a) is 1-Lipschitz and <= 0 inside the cone, so f(centre) > radius proves "not visible".
      for (int t = warp; t < nb; t += nwarps) {   // a warp per tile, a lane per geom, ballot-compacted in id order
        const int tile = t0 + t, k = tile / tiles_cam, r = tile - k * tiles_cam, ty = r / tiles_x, tx = r - ty * tiles_x;
        const float* cw = CW + 12 * k;
        const float th = reinterpret_cast<const float*>(tab + rh.off_cam + cams.id[k] * CAM_STRIDE)[CAM_TANHALF];
        const float x0 = tx * RENDER_TILE_W, y0 = ty * RENDER_TILE_H;
        const float x1 = fminf(x0 + RENDER_TILE_W, (float)width), y1 = fminf(y0 + RENDER_TILE_H, (float)height);
        const f3 o = ld3(cw), axis = pixel_dir(cw, th, 0.5f * (x0 + x1), 0.5f * (y0 + y1), width, height);
        // lanes 0..3 take one corner each
        float ca = dot(axis, pixel_dir(cw, th, (lane & 1) ? x1 : x0, (lane & 2) ? y1 : y0, width, height));
        ca = fminf(ca, __shfl_xor_sync(0xffffffffu, ca, 1));
        ca = fminf(ca, __shfl_xor_sync(0xffffffffu, ca, 2));
        ca = fmaxf(__shfl_sync(0xffffffffu, ca, 0) - 1e-4f, 0.f);   // widen by rounding slack
        const float sa = sqrtf(fmaxf(1.f - ca * ca, 0.f));
        uint16_t* L = TL + t * lstride;
        int n = 0;
        MJB_NOUNROLL
        for (int g0 = 0; g0 < dm.ngeom; g0 += 32) {
          const int g = g0 + lane;
          bool keep = false;
          if (g < dm.ngeom) {
            const float* G = GL + g * GL_STRIDE;
            const int type = __float_as_int(G[GL_TYPE]);
            keep = type >= 0;
            if (keep && type != MJB_GEOM_PLANE) {
              f3 v = ld3(G + GL_POS) - o;
              float pa = dot(v, axis), pp = sqrtf(fmaxf(dot(v, v) - pa * pa, 0.f));
              keep = pp * ca - pa * sa <= G[GL_RBOUND] * 1.0001f + 1e-5f;
            }
          }
          const uint32_t m = __ballot_sync(0xffffffffu, keep);
          if (keep) L[1 + n + __popc(m & ((1u << lane) - 1u))] = (uint16_t)g;
          n += __popc(m);
        }
        if (lane == 0) L[0] = (uint16_t)n;
      }
      __syncthreads();
      // (2) one warp per tile, one lane per 4-pixel group (4 groups per tile row)
      for (int t = warp; t < nb; t += nwarps) {
        const int tile = t0 + t, k = tile / tiles_cam, r = tile - k * tiles_cam, ty = r / tiles_x, tx = r - ty * tiles_x;
        const int iy = ty * RENDER_TILE_H + (lane >> 2), ix0 = tx * RENDER_TILE_W + (lane & 3) * 4;
        if (iy >= height || ix0 >= width) continue;
        const float* cw = CW + 12 * k;
        const float th = reinterpret_cast<const float*>(tab + rh.off_cam + cams.id[k] * CAM_STRIDE)[CAM_TANHALF];
        const f3 o = ld3(cw);
        const uint16_t* L = TL + t * lstride;
        const int nl = L[0];
        uint32_t col[4];
        f3 d[4];
#pragma unroll
        for (int j = 0; j < 4; j++) d[j] = pixel_dir(cw, th, ix0 + j + 0.5f, iy + 0.5f, width, height);   // columns past the edge are not stored
        shade_rays4(GL, L + 1, nl, o, d, col);
        uint8_t* dst = out + ((((size_t)env * cams.n + k) * height + iy) * width + ix0) * 3;
        if (words) {  // 12 bytes = three aligned words
          uint32_t* d32 = reinterpret_cast<uint32_t*>(dst);
          d32[0] = col[0] | (col[1] << 24);
          d32[1] = (col[1] >> 8) | (col[2] << 16);
          d32[2] = (col[2] >> 16) | (col[3] << 8);
        } else {
          for (int j = 0; j < 4 && ix0 + j < width; j++) {
            dst[3 * j] = col[j] & 0xff; dst[3 * j + 1] = (col[j] >> 8) & 0xff; dst[3 * j + 2] = (col[j] >> 16) & 0xff;
          }
        }
      }
      __syncthreads();   // the tile lists (and, after the last batch, the scratch) are reused
    }
  }
}
#endif

}  // namespace mjb
