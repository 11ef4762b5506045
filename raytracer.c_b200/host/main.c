/*
 * main.c -- command-line driver, the counterpart of the reference's main.c:176-445.
 *
 * Same required options (`-w -h -s -o`, main.c:149-174,189-193), same default scene
 * (main.c:244-397 via scene_default), same camera (main.c:424-425), same summary lines
 * (main.c:435-439) and the PNG goes out with the stbi_write_png argument convention
 * (main.c:41).  Extra options select the other benchmark scenes:
 *   -d <max depth>           run-time MAX_DEPTH (default 5)
 *   -S <seed>                Philox key (default 1666943821, main.c:182)
 *   -g <device>              CUDA device ordinal
 *   -c default|spheres:N|mesh:GRID|obj:FILE
 *   -i path|whitted|nee      integrator: trace_path (upstream default), cast_ray (raytracer.c:207-211), or trace_path
 *                            with next-event estimation (same image in expectation, less noise)
 *   -G <gpus>                render on GPUs 0..n-1 of the box (samples sharded, one ncclReduce; default $RTB_NUM_GPUS or 1)
 *   -D stochastic|split      dielectric estimator: one child per vertex (default) or the reference's two-way split
 *   -m <sx,sy,sz,ry,tx,ty,tz> with obj:FILE -- place the mesh like the reference's driver would: scale, rotation about
 *                            y (degrees), translation, composed into a mat4 and applied with apply_matrix (main.c:140-147)
 *   -a <prefix>              also write the first-hit feature buffers of the frame (render_ex_aov): <prefix>_albedo.pfm,
 *                            <prefix>_normal.pfm (RGB) and <prefix>_depth.pfm (grey), the guides of the built-in
 *                            denoiser (-n) and what an external one such as oidnDenoise --alb --nrm reads; single GPU only
 *   -n <passes>              write the DENOISED frame to the PNG (render_ex_denoised: the built-in a-trous denoiser
 *                            guided by the feature buffers, <passes> a-trous passes, 0 = the default); single GPU only
 * Deliberately NOT reproduced: the option parser's mis-parse of values whose second
 * character is h/w/s/o (SURVEY.md section 5) and the SIGINT handler's double free.
 */
#include <string.h>
#include <time.h>

#include "raytracer.h"
#include "scenes.h"

int rt_write_png(const char *filename, int w, int h, int comp, const void *data, int stride_in_bytes);
int rt_write_pfm(const char *filename, int w, int h, int comp, const float *data);

typedef struct
{
  Options options;
  int max_depth, device, integrator, gpus, dielectric;
  uint64_t seed;
  const char *scene, *placement, *aov_prefix;
  int denoise; /* -n given */
  DenoiseParams dn;
} Cli;

static void usage(const char *prog)
{
  fprintf(stderr, "Usage: %s -w <width> -h <height> -s <samples per pixel> -o <filename>\n", prog);
  fprintf(stderr, "       [-d <max depth>] [-S <seed>] [-g <cuda device>] [-c default|spheres:N|mesh:GRID|obj:FILE]\n");
  fprintf(stderr, "       [-i path|whitted] [-G <gpus>] [-D stochastic|split] [-m sx,sy,sz,ry_deg,tx,ty,tz]\n");
  fprintf(stderr, "       [-a <prefix>: also write <prefix>_albedo.pfm, <prefix>_normal.pfm, <prefix>_depth.pfm]\n");
  fprintf(stderr, "       [-n <passes>: denoise the frame with the built-in a-trous filter, 0 = default passes]\n");
}

static bool parse_cli(int argc, char **argv, Cli *cli)
{
  for (int i = 1; i < argc; i++)
  {
    const char *a = argv[i];
    if (a[0] != '-' || a[1] == '\0' || a[2] != '\0')
    {
      fprintf(stderr, "unexpected argument '%s'\n", a);
      return false;
    }
    if (i + 1 >= argc)
    {
      fprintf(stderr, "option '%s' needs a value\n", a);
      return false;
    }
    const char *val = argv[++i];
    switch (a[1])
    {
    case 'w': cli->options.width = atoi(val); break;
    case 'h': cli->options.height = atoi(val); break;
    case 's': cli->options.samples = atoi(val); break;
    case 'o': cli->options.result = (char *)val; break;
    case 'd': cli->max_depth = atoi(val); break;
    case 'S': cli->seed = strtoull(val, NULL, 10); break;
    case 'g': cli->device = atoi(val); break;
    case 'c': cli->scene = val; break;
    case 'i':
      cli->integrator = (strcmp(val, "whitted") == 0) ? RT_INTEGRATOR_WHITTED
                        : (strcmp(val, "nee") == 0)   ? RT_INTEGRATOR_PATH_NEE
                                                      : RT_INTEGRATOR_PATH;
      break;
    case 'G': cli->gpus = atoi(val); break;
    case 'D': cli->dielectric = (strcmp(val, "split") == 0) ? RT_DIELECTRIC_SPLIT : RT_DIELECTRIC_STOCHASTIC; break;
    case 'm': cli->placement = val; break;
    case 'a': cli->aov_prefix = val; break;
    case 'n':
      cli->denoise = 1;
      denoise_params_default(&cli->dn);
      if (atoi(val) != 0)
        cli->dn.iterations = atoi(val);
      break;
    default:
      fprintf(stderr, "unknown option '%s'\n", a);
      return false;
    }
  }
  if (cli->aov_prefix && cli->gpus > 1)
  {
    fprintf(stderr, "-a (feature buffers) renders on one GPU: it cannot be combined with -G %d\n", cli->gpus);
    return false;
  }
  if (cli->denoise && cli->gpus > 1)
  {
    fprintf(stderr, "-n (denoiser) renders on one GPU: it cannot be combined with -G %d\n", cli->gpus);
    return false;
  }
  return cli->options.width >= 2 && cli->options.height >= 2 && cli->options.samples >= 1;
}

/* <prefix><suffix>.pfm */
static bool write_pfm(const char *prefix, const char *suffix, int w, int h, int comp, const float *data)
{
  char *name = (char *)malloc(strlen(prefix) + strlen(suffix) + 5);
  if (!name)
    return false;
  sprintf(name, "%s%s.pfm", prefix, suffix);
  printf("writing %s...\n", name);
  bool ok = rt_write_pfm(name, w, h, comp, data) != 0;
  if (!ok)
    fprintf(stderr, "could not write '%s'\n", name);
  free(name);
  return ok;
}

int main(int argc, char **argv)
{
  Cli cli;
  memset(&cli, 0, sizeof(cli));
  cli.options.width = 320; /* main.c:24-30 */
  cli.options.height = 180;
  cli.options.samples = 50;
  cli.options.result = "result.png";
  cli.options.obj = "assets/cube.obj";
  cli.max_depth = MAX_DEPTH;
  cli.seed = SCENE_SEED;
  cli.scene = "default";

  printf("seed = %llu\n", (unsigned long long)SCENE_SEED);
  if (argc <= 1 || !parse_cli(argc, argv, &cli))
  {
    usage(argv[0]);
    return EXIT_FAILURE;
  }
  Options *opt = &cli.options;

  size_t fb_len = (size_t)opt->width * opt->height * 3;
  uint8_t *framebuffer = (uint8_t *)calloc(fb_len, 1);
  if (!framebuffer)
  {
    fprintf(stderr, "could not allocate framebuffer\n");
    return EXIT_FAILURE;
  }

  Camera camera;
  init_camera(&camera, VECTOR(0.0, 0, 50), VECTOR(0, 0, 0), opt);

  RenderParams rp;
  render_params_default(&rp);
  rp.max_depth = cli.max_depth;
  rp.seed = cli.seed;
  rp.device = cli.device;
  rp.integrator = cli.integrator;
  rp.dielectric_mode = cli.dielectric;
  if (cli.gpus > 0)
    rp.num_gpus = cli.gpus;

  RenderAov aov_bufs = { NULL, NULL, NULL, NULL };
  const RenderAov *aov = NULL;
  if (cli.aov_prefix)
  {
    const size_t n_px = (size_t)opt->width * opt->height;
    aov_bufs.albedo = (float *)calloc(3 * n_px, sizeof(float));
    aov_bufs.normal = (float *)calloc(3 * n_px, sizeof(float));
    aov_bufs.depth = (float *)calloc(n_px, sizeof(float));
    if (!aov_bufs.albedo || !aov_bufs.normal || !aov_bufs.depth)
    {
      fprintf(stderr, "could not allocate the feature buffers\n");
      return EXIT_FAILURE;
    }
    aov = &aov_bufs;
  }

  const DenoiseParams *dn = cli.denoise ? &cli.dn : NULL;
  struct timespec t0, t1;
  clock_gettime(CLOCK_MONOTONIC, &t0);
  /* the CUDA context comes up on a second thread while the scene is generated or read from disk */
  render_warm_up(&rp);
  /* development aid ($RTB_TIMING): where a run of the driver spends its time */
  const bool timing = getenv("RTB_TIMING") != NULL;
  struct timespec tm = t0;
#define CLI_MARK(what) do { if (timing) { struct timespec now_; clock_gettime(CLOCK_MONOTONIC, &now_); \
    fprintf(stderr, "main: %s %.1f ms\n", what, 1e3 * (double)(now_.tv_sec - tm.tv_sec) + 1e-6 * (double)(now_.tv_nsec - tm.tv_nsec)); tm = now_; } } while (0)

/* with -n the denoised frame, else exactly the frame of render_ex_aov / render_scene_aov */
#define RENDER_EX(...) (dn ? render_ex_denoised(__VA_ARGS__, dn) : render_ex_aov(__VA_ARGS__))
#define RENDER_SCENE(...) (dn ? render_scene_denoised(__VA_ARGS__, dn) : render_scene_aov(__VA_ARGS__))
  if (strcmp(cli.scene, "default") == 0)
  {
    Object scene[SCENE_DEFAULT_COUNT];
    size_t n = scene_default(scene, opt->width, opt->height);
    RENDER_EX(framebuffer, scene, n, &camera, opt, &rp, aov);
  }
  else if (strncmp(cli.scene, "spheres:", 8) == 0)
  {
    Object *scene = NULL;
    SceneMix mix = { 0.5, 0.2, 0.2 }; /* main.c:104-119 */
    size_t n = scene_sphere_field(&scene, (size_t)atol(cli.scene + 8), opt->width, opt->height, mix, cli.seed);
    RENDER_EX(framebuffer, scene, n, &camera, opt, &rp, aov);
    free(scene);
  }
  else if (strncmp(cli.scene, "mesh:", 5) == 0 || strncmp(cli.scene, "obj:", 4) == 0)
  {
    TriangleMesh mesh = { 0, NULL };
    if (cli.scene[0] == 'm')
    {
      double aspect = (double)opt->width / (double)opt->height;
      scene_heightfield_mesh(&mesh, atoi(cli.scene + 5), 20 * aspect * 0.98, 29.0, -12.0, 5.0);
    }
    else if (!load_obj(cli.scene + 4, &mesh))
      return EXIT_FAILURE;
    CLI_MARK("mesh (generate / load_obj)");
    if (cli.placement)
    {
      /* scale, then rotate about y, then translate: M = T * Ry * S, row-major like vector.h */
      double v[7] = { 1, 1, 1, 0, 0, 0, 0 };
      sscanf(cli.placement, "%lf,%lf,%lf,%lf,%lf,%lf,%lf", &v[0], &v[1], &v[2], &v[3], &v[4], &v[5], &v[6]);
      const double a = v[3] * (PI / 180), c = cos(a), s = sin(a);
      mat4 m = { c * v[0], 0, s * v[2], v[4],
                 0, v[1], 0, v[5],
                 -s * v[0], 0, c * v[2], v[6],
                 0, 0, 0, 1 };
      apply_matrix(&mesh, m);
      CLI_MARK("apply_matrix");
    }
    SceneObject *scene = NULL;
    Sphere *spheres = NULL;
    size_t n = scene_mesh_room(&scene, &spheres, &mesh, opt->width, opt->height);
    RENDER_SCENE(framebuffer, scene, n, &camera, opt, &rp, aov);
    CLI_MARK("render_scene (first call: CUDA context + upload + BVH + render + read-back)");
    free(scene);
    free(spheres);
    free_mesh(&mesh);
  }
  else
  {
    usage(argv[0]);
    return EXIT_FAILURE;
  }

  clock_gettime(CLOCK_MONOTONIC, &t1);
  double seconds = (double)(t1.tv_sec - t0.tv_sec) + 1e-9 * (double)(t1.tv_nsec - t0.tv_nsec);

  printf("%d x %d (%d) pixels\n", opt->width, opt->height, opt->width * opt->height);
  printf("cast %lld rays\n", ray_count);
  printf("checked %lld possible intersections\n", intersection_test_count);
  printf("rendering took %f seconds\n", seconds);
  printf("writing result to '%s'...\n", opt->result);

  if (rt_write_png(opt->result, opt->width, opt->height, 3, framebuffer, opt->width * 3) == 0)
  {
    free(framebuffer);
    return EXIT_FAILURE;
  }
  CLI_MARK("write PNG");
  if (aov && !(write_pfm(cli.aov_prefix, "_albedo", opt->width, opt->height, 3, aov->albedo) &&
               write_pfm(cli.aov_prefix, "_normal", opt->width, opt->height, 3, aov->normal) &&
               write_pfm(cli.aov_prefix, "_depth", opt->width, opt->height, 1, aov->depth)))
    return EXIT_FAILURE;
  printf("done.\n");
  free(framebuffer);
  free(aov_bufs.albedo);
  free(aov_bufs.normal);
  free(aov_bufs.depth);
  return EXIT_SUCCESS;
}
