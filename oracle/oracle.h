/* oracle.h - C interface shared by the two CPU checkers of the render hot path.
 *
 * TEST INFRASTRUCTURE ONLY.  Nothing under oracle/ is on the product path: only
 * tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference
 * legs may load these libraries, and only as the checker / reported baseline.
 *
 *   oracle/liboracle.so        - oracle.c, a plain-C restatement of the reference's
 *                                per-pixel path (kernel.cu:1614-1690 and callees).
 *   oracle/_ref/libref_oracle.so - the reference's OWN code (kernel.cu read in place
 *                                from /root/reference, mechanically patched into
 *                                oracle/_ref/, compiled as host C++) behind the
 *                                same entry point.  Used to pin the restatement.
 *
 * Both export `oracle_render` with the descriptor below.
 */
#ifndef ORE_ORACLE_H
#define ORE_ORACLE_H
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct oracle_frame {
    int32_t width, height;   /* full frame size (dx,dy use the full size, kernel.cu:1624-1625) */
    int32_t y0, y1;          /* rows rendered: [y0,y1), row 0 = first row of `pixels`          */
    int32_t y_step;          /* render rows y0, y0+y_step, ... (<y1); 1 = every row            */
    float cam_org[3];        /* camera::Org   (kernel.cu:1695)                                 */
    float cam_yaw, cam_pitch;/* camera::Camyaw/Campitch in degrees (kernel.cu:261)             */
    float aspect;            /* global `aspect` = (float)tan(90*0.5*3.1415/180) (kernel.cu:1701)*/
    int32_t n_spheres;
    const float* spheres;    /* n x 4: cx,cy,cz, radius MEMBER (= ctor r*r, kernel.cu:287)     */
    int32_t n_lights;
    const float* lights;     /* n x 7: pos.xyz,size,r,g,b (kernel.cu:1246-1261)                */
    int32_t tex_w, tex_h;    /* object texture, sprite planes (sprite.h:29-45)                 */
    const float *tex_r, *tex_g, *tex_b;   /* tex_w*tex_h floats each, row-major                */
    int32_t sky_w, sky_h;    /* skybox texture                                                 */
    const float *sky_r, *sky_g, *sky_b;
    float sky_size;          /* skybox ctor arg (10000, kernel.cu:1700)                        */
    /* "next" primitives of castRay / castLightRay (kernel.cu:360-509, loops :1344-1372,1512-1536) */
    int32_t n_cubes;
    const float* cubes;      /* n x 6: cube ctor args c1.xyz, c2.xyz (kernel.cu:391-396)       */
    int32_t n_planes;        /* the reference copies ONE plane to the device (kernel.cu:1213-1217):
                                the _ref build accepts 0 or 1, the C restatement any count       */
    const float* planes;     /* n x 6: plane ctor args pos.xyz, normal.xyz (kernel.cu:364-367) */
    /* triangle mesh with its flat BVH, exactly as the reference's `mesh` holds it after its OBJ loader and
     * createBvhMesh() ran (kernel.cu:559-1017); use oracle_ref_build_mesh (the _ref library) to obtain these from
     * an OBJ file with the reference's OWN loader/builder */
    int32_t n_tris;
    const float* tris;       /* n x 27: `triangle` = points[3], normal, vecNormal[3], vt[3] (kernel.cu:206-212) */
    int32_t mesh_has_normals;/* mesh::has_normals (kernel.cu:567)                                           */
    int32_t n_boxes;         /* mesh::bvhbox_count leaf boxes                                                */
    const float* box_bounds; /* n_boxes x 6: cube bounds[0].xyz, bounds[1].xyz of Bvhbox::bvhbox            */
    const int32_t* box_offsets; /* n_boxes + 1: leaf j holds box_indices[box_offsets[j] .. box_offsets[j+1]) */
    const int32_t* box_indices; /* triangle indices per leaf, in the leaf's order (Bvhbox::indexes)          */
} oracle_frame;

/* Renders the selected rows.  Outputs are packed by rendered row (row k of the
 * output = image row y0 + k*y_step), `width` entries per row; any may be NULL.
 *   pixels : 0x00RRGGBB                         (rgbToInt, kernel.cu:546-556)
 *   hit_id : nearest primitive, -1 = miss: sphere i -> i, cube i -> n_spheres + i, plane i ->
 *            n_spheres + n_cubes + i, triangle i -> n_spheres + n_cubes + n_planes + i
 *            (castRay loops, kernel.cu:1293-1372; hit_type 1, 3, 2, 0)
 *   hit_t  : nearest t (bit pattern matters), +inf on miss
 *   counts : [0] primary sphere::intersect calls, [1] shadow-phase calls in the
 *            reference's loop order incl. early break (kernel.cu:1501-1510),
 *            [2] sky-sphere calls, [3] hit pixels.  liboracle only; the _ref
 *            build leaves counts zero (it is the unmodified arithmetic, uninstrumented).
 * Returns 0 on success.  n_threads <= 0 means all host threads (OpenMP). */
int oracle_render(const oracle_frame* f, uint32_t* pixels, int32_t* hit_id, float* hit_t,
                  uint64_t* counts, int n_threads);

/* Single ray-sphere test exactly as sphere::intersect (kernel.cu:293-354).
 * radius_member is the stored member (ctor r*r).  Returns the bool; *t as written. */
int oracle_sphere_intersect(const float org[3], const float dir[3], const float centre[3],
                            float radius_member, float* t);

/* Single ray-box test exactly as cube::intersect (kernel.cu:460-483), the reference's max/min macros and their NaN
 * behaviour included; also the leaf-box test of the mesh loops.  c1, c2: the ctor's corners in either order.  Returns
 * the bool; *t as written (tmin on a hit, tmax otherwise; negative t can be a hit). */
int oracle_cube_intersect(const float org[3], const float dir[3], const float c1[3], const float c2[3], float* t);

/* Single ray-plane test exactly as plane::intersect (kernel.cu:369-380): one-sided, t >= 0. */
int oracle_plane_intersect(const float org[3], const float dir[3], const float pos[3], const float normal[3], float* t);

/* Single ray-triangle test exactly as mesh::rayIntersect (kernel.cu:1024-1059).  tri: the 9 vertex floats (points[3]).
 * Returns the bool; *t, *u, *v as written, 0 where the test returns before writing them. */
int oracle_tri_intersect(const float org[3], const float dir[3], const float tri[9], float* t, float* u, float* v);

/* rgbToInt (kernel.cu:546-556) */
uint32_t oracle_rgb_to_int(int r, int g, int b);

/* _ref library only: runs the reference's OWN OBJ loader and BVH builder (mesh::mesh, createBvhMesh,
 * kernel.cu:577-936) on `obj_path` and copies out the flat arrays in the oracle_frame layout.
 * Returns 0 on success, 1 if a capacity is too small or the file cannot be read. */
int oracle_ref_build_mesh(const char* obj_path, float* tris, int32_t cap_tris, int32_t* n_tris, int32_t* has_normals,
                          float* box_bounds, int32_t* box_offsets, int32_t cap_boxes, int32_t* n_boxes,
                          int32_t* box_indices, int32_t cap_indices);

/* "reference" or "port" */
const char* oracle_kind(void);

#ifdef __cplusplus
}
#endif
#endif
