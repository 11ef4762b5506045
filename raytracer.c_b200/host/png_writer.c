/*
 * png_writer.c -- minimal PNG encoder for the RGB8 framebuffer render() fills.
 *
 * The reference hands its framebuffer to the vendored stb_image_write
 * (`stbi_write_png(name, W, H, 3, fb, W*3)`, main.c:41); that third-party file is not
 * copied.  rt_write_png() has the same argument meaning and return convention (0 on
 * failure) and writes a valid, uncompressed PNG: zlib "stored" blocks, filter type 0.
 * Any consumer of the reference's output (an image viewer, PIL) reads it the same way.
 *
 * rt_write_pfm() writes float images (the feature buffers of render_ex_aov / render_scene_aov) as Portable FloatMap,
 * the format denoisers read (oidnDenoise --alb --nrm).
 */
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

/* CRC-32 (PNG, polynomial 0xEDB88320), eight bytes per step ("slicing by 8"): table k holds the CRC of a byte
 * followed by k zero bytes.  The frame of a 1080p render is 6 MB; with a byte-at-a-time CRC and an Adler-32 that
 * took a modulo per byte, writing it cost 65 ms on the build container (38 ms on the B200 box's host), with this
 * form 27 ms, most of it the two copies and the fwrite. */
static uint32_t crc_table[8][256];
static int crc_ready = 0;

static void crc_init(void)
{
  for (uint32_t n = 0; n < 256; n++)
  {
    uint32_t c = n;
    for (int k = 0; k < 8; k++)
      c = (c & 1) ? (0xEDB88320u ^ (c >> 1)) : (c >> 1);
    crc_table[0][n] = c;
  }
  for (uint32_t n = 0; n < 256; n++)
    for (int k = 1; k < 8; k++)
      crc_table[k][n] = crc_table[0][crc_table[k - 1][n] & 0xFF] ^ (crc_table[k - 1][n] >> 8);
  crc_ready = 1;
}

static uint32_t crc_update(uint32_t crc, const uint8_t *buf, size_t len)
{
  size_t i = 0;
  for (; i + 8 <= len; i += 8)
  {
    /* bytes are combined explicitly: no alignment or endianness assumption */
    const uint32_t lo = crc ^ ((uint32_t)buf[i] | (uint32_t)buf[i + 1] << 8 | (uint32_t)buf[i + 2] << 16 | (uint32_t)buf[i + 3] << 24);
    crc = crc_table[7][lo & 0xFF] ^ crc_table[6][(lo >> 8) & 0xFF] ^ crc_table[5][(lo >> 16) & 0xFF] ^ crc_table[4][lo >> 24] ^
          crc_table[3][buf[i + 4]] ^ crc_table[2][buf[i + 5]] ^ crc_table[1][buf[i + 6]] ^ crc_table[0][buf[i + 7]];
  }
  for (; i < len; i++)
    crc = crc_table[0][(crc ^ buf[i]) & 0xFF] ^ (crc >> 8);
  return crc;
}

/* Adler-32 with the modulo deferred: 5552 is the largest n with 255 n (n + 1) / 2 + (n + 1)(65521 - 1) < 2^32 (zlib's NMAX) */
static void adler_update(uint32_t *pa, uint32_t *pb, const uint8_t *buf, size_t len)
{
  uint32_t a = *pa, b = *pb;
  while (len > 0)
  {
    const size_t n = len < 5552 ? len : 5552;
    for (size_t i = 0; i < n; i++)
    {
      a += buf[i];
      b += a;
    }
    a %= 65521u;
    b %= 65521u;
    buf += n;
    len -= n;
  }
  *pa = a;
  *pb = b;
}

static void put_u32(uint8_t *p, uint32_t v)
{
  p[0] = (uint8_t)(v >> 24);
  p[1] = (uint8_t)(v >> 16);
  p[2] = (uint8_t)(v >> 8);
  p[3] = (uint8_t)v;
}

static int write_chunk(FILE *f, const char *type, const uint8_t *data, size_t len)
{
  uint8_t head[8];
  put_u32(head, (uint32_t)len);
  memcpy(head + 4, type, 4);
  uint32_t crc = crc_update(0xFFFFFFFFu, head + 4, 4);
  if (len)
    crc = crc_update(crc, data, len);
  uint8_t tail[4];
  put_u32(tail, crc ^ 0xFFFFFFFFu);
  if (fwrite(head, 1, 8, f) != 8)
    return 0;
  if (len && fwrite(data, 1, len, f) != len)
    return 0;
  return fwrite(tail, 1, 4, f) == 4;
}

int rt_write_png(const char *filename, int w, int h, int comp, const void *data, int stride_in_bytes)
{
  if (!filename || !data || w <= 0 || h <= 0 || (comp != 1 && comp != 3 && comp != 4))
    return 0;
  if (!crc_ready)
    crc_init();

  /* raw scanlines: filter byte 0 + pixels */
  size_t row = (size_t)w * comp + 1;
  size_t raw_len = row * (size_t)h;
  uint8_t *raw = (uint8_t *)malloc(raw_len);
  if (!raw)
    return 0;
  for (int y = 0; y < h; y++)
  {
    raw[y * row] = 0;
    memcpy(raw + y * row + 1, (const uint8_t *)data + (size_t)y * stride_in_bytes, (size_t)w * comp);
  }

  /* zlib container with stored deflate blocks of at most 65535 bytes */
  size_t n_blocks = (raw_len + 65534) / 65535;
  if (n_blocks == 0)
    n_blocks = 1;
  size_t z_len = 2 + raw_len + 5 * n_blocks + 4;
  uint8_t *z = (uint8_t *)malloc(z_len);
  if (!z)
  {
    free(raw);
    return 0;
  }
  size_t o = 0;
  z[o++] = 0x78;
  z[o++] = 0x01;
  uint32_t a = 1, b = 0;
  size_t pos = 0;
  for (size_t k = 0; k < n_blocks; k++)
  {
    size_t len = raw_len - pos < 65535 ? raw_len - pos : 65535;
    z[o++] = (k + 1 == n_blocks) ? 1 : 0;
    z[o++] = (uint8_t)(len & 0xFF);
    z[o++] = (uint8_t)(len >> 8);
    z[o++] = (uint8_t)(~len & 0xFF);
    z[o++] = (uint8_t)((~len >> 8) & 0xFF);
    memcpy(z + o, raw + pos, len);
    adler_update(&a, &b, raw + pos, len);
    o += len;
    pos += len;
  }
  put_u32(z + o, (b << 16) | a);
  o += 4;

  FILE *f = fopen(filename, "wb");
  int ok = f != NULL;
  if (ok)
  {
    static const uint8_t sig[8] = { 0x89, 'P', 'N', 'G', 0x0D, 0x0A, 0x1A, 0x0A };
    uint8_t ihdr[13];
    put_u32(ihdr, (uint32_t)w);
    put_u32(ihdr + 4, (uint32_t)h);
    ihdr[8] = 8;
    ihdr[9] = (comp == 1) ? 0 : (comp == 3 ? 2 : 6);
    ihdr[10] = ihdr[11] = ihdr[12] = 0;
    ok = fwrite(sig, 1, 8, f) == 8 && write_chunk(f, "IHDR", ihdr, 13) && write_chunk(f, "IDAT", z, o) &&
         write_chunk(f, "IEND", NULL, 0);
    ok = (fclose(f) == 0) && ok;
  }
  free(raw);
  free(z);
  return ok;
}

/* Portable FloatMap: "PF" (RGB, comp 3) or "Pf" (grey, comp 1), "<w> <h>", scale -1.0 (= little-endian samples),
 * then the rows BOTTOM to top.  `data` is row-major with row 0 at the top, like the framebuffer.  1 on success. */
int rt_write_pfm(const char *filename, int w, int h, int comp, const float *data)
{
  if (!filename || !data || w <= 0 || h <= 0 || (comp != 1 && comp != 3))
    return 0;
  const size_t row = (size_t)w * comp;
  uint8_t *buf = (uint8_t *)malloc(4 * row);
  if (!buf)
    return 0;
  FILE *f = fopen(filename, "wb");
  int ok = f != NULL && fprintf(f, "%s\n%d %d\n-1.0\n", comp == 3 ? "PF" : "Pf", w, h) > 0;
  for (int y = h - 1; ok && y >= 0; y--)
  {
    for (size_t i = 0; i < row; i++)
    {
      uint32_t v;
      memcpy(&v, data + (size_t)y * row + i, 4);
      buf[4 * i + 0] = (uint8_t)v;
      buf[4 * i + 1] = (uint8_t)(v >> 8);
      buf[4 * i + 2] = (uint8_t)(v >> 16);
      buf[4 * i + 3] = (uint8_t)(v >> 24);
    }
    ok = fwrite(buf, 1, 4 * row, f) == 4 * row;
  }
  if (f)
    ok = (fclose(f) == 0) && ok;
  free(buf);
  return ok;
}
