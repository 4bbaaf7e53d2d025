/* lnb_host_util.h -- small helpers shared by the encoder and decoder host code (plain C). */
#ifndef LNB_HOST_UTIL_H
#define LNB_HOST_UTIL_H

#include <stdint.h>
#include <stddef.h>
#include "linne.h"
#include "lnb_shim.h"
#include "lnb_framing.h"

#define LNB_ALIGNMENT 16
#define LNB_MAX_DEVICES 16                 /* block ranges (devices) one handle shards a whole-stream call over */
#define LNB_ROUNDUP(v, n) ((((v) + ((n) - 1)) / (n)) * (n))

/* grow-only device / host buffers owned by a handle */
typedef struct LnbBuf { void *ptr; size_t cap; } LnbBuf;

int  lnb_buf_reserve_device(LnbDevice *dev, LnbBuf *buf, size_t bytes);
void lnb_buf_release_device(LnbDevice *dev, LnbBuf *buf);
int  lnb_buf_reserve_host(LnbBuf *buf, size_t bytes);       /* pinned */
void lnb_buf_release_host(LnbBuf *buf);

/* 30-byte stream header (big-endian fields) */
LINNEApiResult lnb_header_check_for_encode(const struct LINNEHeader *h);
int  lnb_header_fields_valid(const struct LINNEHeader *h);  /* decoder-side validation */
void lnb_header_write(const struct LINNEHeader *h, uint8_t *dst);
void lnb_header_read(const uint8_t *src, struct LINNEHeader *h);

void lnb_fill_stream_cfg(LnbStreamCfg *cfg, const struct LINNEHeader *h);

/* Block ranges a whole-stream call of `blocks` blocks is cut into on `devices` devices (>= 1).  More than one range per
 * device turns the call into a pipeline: the ranges run on their own streams from their own host threads, so one
 * range's upload, another's kernels and a third's download overlap (the copy engines work beside the SMs) -- worth it
 * from a few thousand blocks per device on.  LINNE_B200_PIPELINE=N forces N ranges per device (0 or 1: none).
 * Returns 1 when the call should simply run on the handle's own device. */
uint32_t lnb_plan_ranges(uint32_t blocks, uint32_t devices);

/* Devices of the G ranges of a sharded call: ordinal[k] = k mod D on a handle asked for `requested` > 1 devices, D = no
 * more than the `visible` ones (>= 1); the handle's own device `own` otherwise.  Returns D, the devices in use. */
uint32_t lnb_place_ranges(uint32_t requested, int visible, int own, uint32_t G, int *ordinal);

/* rendezvous of the shard workers of one call with the thread that made it: every worker reports ("sized"), the caller
 * looks at all reports and releases them ("placed") */
#include <pthread.h>
typedef struct LnbRendezvous { pthread_mutex_t lock; pthread_cond_t cv; uint32_t reported; int released; } LnbRendezvous;
void lnb_rendezvous_init(LnbRendezvous *r);
void lnb_rendezvous_destroy(LnbRendezvous *r);
void lnb_rendezvous_report_and_wait(LnbRendezvous *r);      /* worker */
void lnb_rendezvous_collect(LnbRendezvous *r, uint32_t workers);   /* caller: returns when all have reported (lock held off) */
void lnb_rendezvous_release(LnbRendezvous *r);              /* caller */

/* Turnstile of the ranges of one call that share a device: their bulk transfers take turns in range order (phase 0:
 * host -> device, phase 1: device -> host).  Ranges started side by side otherwise move in lockstep -- all uploads
 * share the link, then all kernels share the SMs, then all downloads share the link -- and nothing overlaps; with the
 * turnstile range k + 1 uploads while range k computes and range k - 1 downloads.  `stride` = ranges between two
 * that share a device (the number of devices in use). */
typedef struct LnbTurnstile { pthread_mutex_t lock; pthread_cond_t cv; uint32_t stride; uint8_t passed[2][LNB_MAX_DEVICES]; } LnbTurnstile;
void lnb_turnstile_init(LnbTurnstile *t, uint32_t stride);
void lnb_turnstile_destroy(LnbTurnstile *t);
void lnb_turnstile_wait(LnbTurnstile *t, int phase, uint32_t k);    /* until range k - stride has passed `phase` */
void lnb_turnstile_pass(LnbTurnstile *t, int phase, uint32_t k);    /* idempotent */

#endif
